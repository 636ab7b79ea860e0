"""GPU: the safety layer against the full affine voltage map (fp_safety_project_affine) against the oracle's fp64
restatement of the same active-set method (oracle/safety_affine_ref.py project_affine, itself checked against the QP handed to
a generic solver by tests/test_oracle_safety_affine.py), on three maps: the reference's own fit with its scalers folded
in, a dense LinDistFlow sensitivity map of IEEE-33, and the reference's row-sum (2-banded) map, which must reproduce
fp_safety_project.  Outputs are fp32, so 1e-6 relative; slacks are fp64 from the same formulas, so 1e-9."""
import os

import numpy as np
import pytest
import torch

from _feeders import lindistflow_map
from oracle import env_ref, ieee33, safety_affine_ref, safety_ref

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_predictor.npz")


def _stub(args, state_row):
    """A RefFlexEnv-shaped object carrying one GPU env's current values (what parse_actions reads)."""
    st = state_row                                                  # [P(33), Q(33), Ppv(5), V(33), price, E(5)]
    ref = env_ref.RefFlexEnv.__new__(env_ref.RefFlexEnv)
    ref.args = env_ref._Args(dict(env_ref.DEFAULT_ARGS)); ref.args.update(args)
    ref.base_powergrid = ieee33.create_network()
    G = ref.base_powergrid
    ref.current_active_demand = {b: float(st[i]) for i, b in enumerate(G['bus_numbers'])}
    ref.current_reactive_demand = {b: float(st[33 + i]) for i, b in enumerate(G['bus_numbers'])}
    ref.current_pv_power = {b: float(st[66 + i]) for i, b in enumerate(G['PVs_at_buildings'])}
    ref.current_ess_energy = {b: float(st[66 + 5 + 33 + 1 + i]) for i, b in enumerate(G['ESSs_at_buildings'])}
    return ref


def _proposal(ref, a):
    pct, ch, dis, qpv = safety_ref.parse_actions(ref, a)
    return np.array([[pct[b], ch[b], dis[b], qpv[b]] for b in ref.base_powergrid['buildings']])


def _lindistflow():
    """dV_n / dP_m = -sum R_l, dV_n / dQ_m = -sum X_l over the lines shared by the root paths of buses n and m."""
    return lindistflow_map(ieee33.tree_arrays(ieee33.create_network()))


def _map(env, name):
    g = np.load(GOLD)
    if name == "reference_fit":
        from flexgpu.predictor import VoltagePredictor
        pred = VoltagePredictor.from_linear_model(env, g["coef"], g["intercept"], g["x_scale"], g["x_min"], g["y_scale"], g["y_min"])
        return pred.A, pred.c
    if name == "lindistflow":
        return _lindistflow()
    coef = g["coef"].astype(np.float64)                             # row-sum: what fp_safety_project evaluates
    n = coef.shape[0]
    A = np.zeros((n, 2 * n)); A[np.arange(n), 2 * np.arange(n)] = coef[:, :n].sum(1); A[np.arange(n), 2 * np.arange(n) + 1] = coef[:, n:].sum(1)
    return A, g["intercept"].astype(np.float64)


def _env(cuda, profiles, n, seed=21):
    from flexgpu import BatchedFlexProvisionEnv
    env = BatchedFlexProvisionEnv(None, n_envs=n, device=cuda, profiles=profiles, seed=seed)
    env.reset(return_obs=False)
    g = torch.Generator(device=cuda).manual_seed(3)
    for _ in range(3):
        env.step(torch.rand(n, 5, 4, device=cuda, generator=g), want_info=False)
    actions = torch.randn(n, 5, 4, device=cuda, generator=g) * 0.6 + 0.4      # raw policy outputs, some outside [0, 1]
    return env, actions


def _limits(env, A, c, lo_q=0.3, hi_q=0.85):
    """Limits placed on the spread of the map's predictions at the current demands, so that a good share of the envs
    is pushed outside on one side or the other."""
    st = env.get_state(torch.float64).cpu().numpy()
    x = np.empty((st.shape[0], 66)); x[:, 0::2] = st[:, :33]; x[:, 1::2] = st[:, 33:66]
    V = x @ A.T + c
    return float(np.quantile(V.min(1), lo_q)), float(np.quantile(V.max(1), hi_q))


def _agent_bus(env):
    G = ieee33.create_network()
    return np.array([G['bus_numbers'].index(b) for b in env.agent_ids])


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("name", ["reference_fit", "lindistflow", "banded"])
def test_affine_projection_matches_restatement(cuda, profiles, args, name, dtype):
    n = 3001                                                        # ragged: not a multiple of the 8 envs of a CTA
    env, actions = _env(cuda, profiles, n)
    A, c = _map(env, name)
    v_min, v_max = _limits(env, A, c)
    env.load_safety_map(A, c, v_min=v_min, v_max=v_max)
    a = actions.to(dtype)
    adj, slack, moved, status = env.safety_project_affine(a, want_info=True)
    adj_agent = env.safety_project_affine(a, layout="agent")
    assert adj.shape == (n, 20) and adj_agent.shape == (n, 5, 4) and slack.shape == (n, 33) and status.shape == (n,)
    assert torch.equal(adj.view(n, 4, 5).permute(0, 2, 1), adj_agent)
    assert bool((status >= 0).all()), "every env converges within the cap"
    frac = float((status > 0).double().mean())
    assert 0.05 < frac < 0.95, frac                                 # the case mix exercises both branches
    # envs already inside: the proposal cast to fp32, bit for bit (the row-sum layer with a flat map moves nothing)
    env.load_safety_model(np.zeros((33, 66)), np.full(33, 1.0))
    noop = env.safety_project(a)
    inside = status == 0
    assert torch.equal(adj[inside], noop[inside])
    assert not bool(moved[inside].any()) and not bool(slack[inside].any())
    st = env.get_state(torch.float64).cpu().numpy()
    a_np, adj_np, slack_np, moved_np, status_np = a.double().cpu().numpy(), adj.cpu().numpy(), slack.cpu().numpy(), moved.cpu().numpy(), status.cpu().numpy()
    bus = _agent_bus(env)
    n_iter = []
    for e in list(range(0, n, 23)) + [n - 1]:
        ref = _stub(args, st[e])
        y0 = _proposal(ref, a_np[e])
        want, wslack, wstatus = safety_affine_ref.project_affine(y0, st[e, :33], st[e, 33:66], bus, A, c, v_min, v_max)
        want_tm = want.T.reshape(-1)
        assert np.max(np.abs(adj_np[e] - want_tm) / np.maximum(1.0, np.abs(want_tm))) < 1e-6, (e, adj_np[e], want_tm)
        assert np.allclose(slack_np[e], wslack, rtol=1e-9, atol=1e-9), (e, slack_np[e], wslack)
        assert (status_np[e] == 0) == (wstatus == 0), (e, status_np[e], wstatus)
        assert np.array_equal(moved_np[e], (want != y0).any(axis=1)), (e, moved_np[e])
        n_iter.append(wstatus)
    assert max(n_iter) > 0
    if name == "banded":
        # the row-sum map is the reference's reading: fp_safety_project computes the same optimum in closed form
        g = np.load(GOLD)
        env.load_safety_model(g["coef"].astype(np.float64), g["intercept"].astype(np.float64))
        env.load_safety_map(A, c, v_min=float(env.args_dict["v_min"]), v_max=float(env.args_dict["v_max"]))
        want, wslack, wmoved = env.safety_project(a, want_info=True)
        got, gslack, gmoved, gstatus = env.safety_project_affine(a, want_info=True)
        assert bool((gstatus >= 0).all())
        assert float(((got - want).abs() / want.abs().clamp(min=1.0)).max()) < 1e-6
        assert torch.equal(gmoved, wmoved)
        assert torch.allclose(gslack[:, torch.as_tensor(bus, device=cuda)], wslack, rtol=1e-9, atol=1e-9)
    env.close()


def test_affine_projection_single_env_and_hopeless(cuda, profiles, args):
    env, actions = _env(cuda, profiles, 1, seed=5)
    A, c = _lindistflow()
    env.load_safety_map(A, c + 0.3)                                 # every bus far above v_max
    adj, slack, moved, status = env.safety_project_affine(actions, want_info=True)
    st = env.get_state(torch.float64).cpu().numpy()[0]
    y0 = _proposal(_stub(args, st), actions.double().cpu().numpy()[0])
    want, wslack, _ = safety_affine_ref.project_affine(y0, st[:33], st[33:66], _agent_bus(env), A, c + 0.3,
                                                float(env.args_dict["v_min"]), float(env.args_dict["v_max"]))
    assert int(status[0]) > 0 and bool(moved.all())
    assert np.max(np.abs(adj.cpu().numpy()[0] - want.T.reshape(-1)) / np.maximum(1.0, np.abs(want.T.reshape(-1)))) < 1e-6
    assert np.allclose(slack.cpu().numpy()[0], wslack, rtol=1e-9, atol=1e-9)
    env.close()
    # hopeless envs: limits no action can reach leave slack, and every env still converges
    n = 2048
    env, actions = _env(cuda, profiles, n, seed=6)
    env.load_safety_map(A, c, v_min=1.5, v_max=2.0)
    adj, slack, moved, status = env.safety_project_affine(actions, want_info=True)
    assert bool((status > 0).all())
    assert bool((slack.sum(1) > 0).any())
    assert bool((adj.view(n, 4, 5)[:, :3] >= 0).all())
    env.close()


def test_affine_projection_misuse(cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv
    from flexgpu._lib import FlexGpuError
    env = BatchedFlexProvisionEnv(None, n_envs=16, device=cuda, profiles=profiles, seed=1)
    env.reset(return_obs=False)
    a = torch.rand(16, 5, 4, device=cuda)
    with pytest.raises(FlexGpuError):
        env.safety_project_affine(a)                                # before load_safety_map
    env.load_safety_model(np.zeros((33, 66)), np.ones(33))          # the row-sum model does not count as the map
    with pytest.raises(FlexGpuError):
        env.safety_project_affine(a)
    A, c = _lindistflow()
    with pytest.raises(FlexGpuError):
        env.load_safety_map(A[:, :65], c)                           # n_in != 2 n_bus
    with pytest.raises(FlexGpuError):
        env.load_safety_map(A[:32], c[:32])                         # n_out != n_bus
    bad = A.copy(); bad[3, 7] = np.nan
    with pytest.raises(FlexGpuError):
        env.load_safety_map(bad, c)
    with pytest.raises(FlexGpuError):
        env.load_safety_map(A, c, v_min=1.1, v_max=0.9)
    with pytest.raises(FlexGpuError):
        env.load_safety_map(A, c, slack_weight=0.0)
    env.load_safety_map(A, c)
    with pytest.raises(ValueError):
        env.safety_project_affine(a[:, :4])                         # wrong number of actions
    out = env.safety_project_affine(a)
    assert out.shape == (16, 20) and bool(torch.isfinite(out).all())
    env.close()
