"""GPU parity on feeders that are NOT the built-in IEEE 33-bus case with five buildings: the run-time-table (RtShape)
instantiations of the thread kernels and the warp kernels at any depth, on every entry of the feeder catalogue
(tests/_feeders.py) in both kernel variants the library accepts for it.  Mirror comparisons are bit for bit; Newton and
the fp64 env restatement are held to the power-flow bars (1e-8 p.u. on V, P, Q, 1e-7 on line currents) and rewards to
1e-6 relative."""
import numpy as np
import pytest
import torch

import _feeders as F
from _env_check import (actions, bits, check_state, draws, feeder_profiles, make_env, mirror_actions, reset_both,
                        scaled_profiles)
from _preview_ref import mirror_copy, mirror_restore
from flexgpu._lib import INFO_KEYS
from oracle import c_mirror, env_ref, ieee33, pf_ref, safety_affine_ref, safety_ref

pytestmark = pytest.mark.gpu

CASES = F.cases()
IDS = [f"{f}-{v}" for f, v in CASES]


def _variant(v):
    return c_mirror.VARIANT_WARP if v == "warp" else c_mirror.VARIANT_THREAD


def _heavy(net):
    """Every other day's demand x 2.4: an episode (121 rows) runs through both a normal and a heavily loaded day, with
    voltage violations on the latter."""
    return scaled_profiles(feeder_profiles(net), every_other_day=True)


@pytest.fixture(scope="module", params=CASES, ids=IDS)
def setup(request, cuda):
    from flexgpu.network import Network
    name, variant = request.param
    net = F.feeder(name)
    prof = feeder_profiles(net)
    tree = ieee33.tree_arrays(net)
    fonet = c_mirror.make_net(tree, F.env_args(net, variant), net['buildings'], variant=_variant(variant))
    n = 200
    env = make_env(cuda, prof, n, variant, net=net)
    yield env, fonet, prof, tree, Network(net), n
    env.close()


def test_power_flow_bit_exact_vs_mirror_and_close_to_newton(setup):
    env, fonet, prof, tree, network, n = setup
    rng = np.random.default_rng(1)
    p = network.base_p[None, 1:] * rng.uniform(0.5, 1.6, (300, network.n_bus - 1))
    q = network.base_q[None, 1:] * rng.uniform(0.5, 1.6, (300, network.n_bus - 1))
    out = {k: (v.cpu().numpy() if v is not None else None) for k, v in env.power_flow(p, q).items()}
    ref = c_mirror.mirror_power_flow(fonet, p, q)
    for k in ("V", "P", "Q", "Isq"):
        assert np.array_equal(out[k], ref[k]), k
    assert np.array_equal(out["iters"], ref["iters"]) and not out["failed"].any()
    for i in (0, 17, 299):                                         # independent dense Newton on pf.py:65-98
        sol = pf_ref.solve_newton(tree, np.concatenate([[0.0], p[i]]), np.concatenate([[0.0], q[i]]))
        assert np.max(np.abs(out["V"][i] - np.sqrt(sol['v']))) < 1e-8
        assert np.max(np.abs(out["P"][i] - sol['P'][1:])) < 1e-8


def test_env_steps_bit_exact_vs_mirror(setup):
    env, fonet, prof, tree, network, n = setup
    mb = c_mirror.MirrorBatch(fonet, prof.as_dict(), n)
    na, nb = env.n_agents, env.n_bus
    reset_both(env, mb, np.random.default_rng(2))
    rng = np.random.default_rng(2)
    for t in range(6):
        a = rng.normal(0.4, 0.5, (n, 4 * na))
        r, d, info = env.step(torch.from_numpy(a), want_info=True)
        rr, dd, ii = mb.step(a)
        assert np.array_equal(r.cpu().numpy(), rr) and np.array_equal(d.cpu().numpy(), dd)
        assert np.array_equal(info["voltage_penalty"].cpu().numpy(), ii[:, 5])
    check_state(env, mb, "6 steps")
    obs = env.get_obs(); state = env.get_state()
    assert obs.shape == (n, na, 6 * env.history) and state.shape == (n, 3 * nb + 2 * na + 1)
    # step(return_obs=True) on a run-time-table feeder (fewer agents: packed observation row, two-launch
    # fallback of fp_step_obs) == step + get_obs, and the window ring agrees with the fp64 history ring
    a = rng.normal(0.4, 0.5, (n, 4 * na))
    r, d, info, o2 = env.step(torch.from_numpy(a), return_obs=True)
    rr, dd, ii = mb.step(a)
    assert np.array_equal(r.cpu().numpy(), rr)
    cur = mb.current_obs()                                         # [n, na, 6] after the step
    assert np.array_equal(o2[:, :, -6:].cpu().numpy(), cur.astype(np.float32))
    assert torch.equal(o2[:, :, :-6], obs[:, :, 6:])               # shifted by one entry
    assert torch.equal(env.get_obs(push=False, dtype=torch.float64)[:, :, :-6].float(), o2[:, :, 6:])


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_power_flow_across_loading_to_collapse(cuda, case):
    """~2000 rows from 0.3x the base loading to well past voltage collapse, every bus jittered: V, P, Q, Isq, pass counts
    and failure flags equal the mirror's; 64 converged rows up to 1.6x against dense Newton (near collapse the sweep's
    fixed point contracts slowly and Newton from a flat start may not converge at all)."""
    from flexgpu.network import Network
    name, variant = case
    net = F.feeder(name)
    tree = ieee33.tree_arrays(net)
    network = Network(net)
    env = make_env(cuda, feeder_profiles(net), 64, variant, net=net)
    fonet = c_mirror.make_net(tree, F.env_args(net, variant), net['buildings'], variant=_variant(variant))
    rng = np.random.default_rng(21)
    m = 2000
    s = np.geomspace(0.3, 60.0, m)[:, None]
    p = network.base_p[None, 1:] * s * rng.uniform(0.85, 1.15, (m, network.n_bus - 1))
    q = network.base_q[None, 1:] * s * rng.uniform(0.85, 1.15, (m, network.n_bus - 1))
    out = {k: v.cpu().numpy() for k, v in env.power_flow(p, q).items()}
    ref = c_mirror.mirror_power_flow(fonet, p, q)
    for k in ("V", "P", "Q", "Isq"):
        assert np.array_equal(out[k], ref[k], equal_nan=True), k
    assert np.array_equal(out["iters"], ref["iters"]) and np.array_equal(out["failed"], ref["failed"])
    ok = np.nonzero(~out["failed"])[0]
    assert out["failed"].any() and len(ok) > m // 4
    light = ok[s[ok, 0] <= 1.6]
    for i in rng.choice(light, 64, replace=False):
        sol = pf_ref.solve_newton(tree, np.r_[0.0, p[i]], np.r_[0.0, q[i]])
        assert np.max(np.abs(out["V"][i] - np.sqrt(sol['v']))) <= 1e-8, (i, s[i])
        assert np.max(np.abs(out["P"][i] - sol['P'][1:])) <= 1e-8, (i, s[i])
        assert np.max(np.abs(out["Q"][i] - sol['Q'][1:])) <= 1e-8, (i, s[i])
        assert np.max(np.abs(np.sqrt(out["Isq"][i]) - np.sqrt(sol['ell'][1:]))) <= 1e-7, (i, s[i])
    env.close()


def _ref_envs(net, prof, idx, start, e0, a0, raw, injected):
    args = F.env_args(net)
    args.pop("kernel_variant")
    if raw:
        args["alg"] = "safemaddpg"
    refs = []
    for e in idx:
        r = env_ref.RefFlexEnv(args, net=net, profiles=prof.as_dict(), rng=np.random.RandomState(0),
                               force_fail=lambda _env, e=e: bool(injected[0] is not None and injected[0][e]))
        r.reset_with(start[e], e0[e], a0[e])
        refs.append(r)
    return refs


@pytest.mark.parametrize("kind", ["f32", "f64", "policy", "raw"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_episode_bit_exact_vs_mirror(cuda, monkeypatch, case, kind):
    """Reset and 95 steps to the episode limit on a ragged batch whose persistent CTAs make several trips each, with a
    NaN-action step, an injected-failure step, a masked step and heavily loaded days: every output and every piece of
    state equals the mirror's at every step; four envs also follow the fp64 restatement of the env."""
    name, variant = case
    monkeypatch.setenv("FLEXGPU_GRID_STEP", "2")                    # 2 persistent CTAs: 4 trips over 8 tiles
    net = F.feeder(name)
    raw = kind == "raw"
    prof = _heavy(net)
    n = 32 * 7 + 7
    env = make_env(cuda, prof, n, variant, net=net, **({"alg": "safemaddpg"} if raw else {}))
    na = env.n_agents
    fonet = c_mirror.make_net(ieee33.tree_arrays(net), F.env_args(net, variant), net['buildings'], raw_actions=raw,
                              variant=_variant(variant))
    mb = c_mirror.MirrorBatch(fonet, prof.as_dict(), n)
    start, e0, a0 = reset_both(env, mb, np.random.default_rng(11))
    check_state(env, mb, "reset")
    idx = [0, 3, n // 2, n - 1]                                     # NaN actions, injected failure, plain, masked out
    injected = [None]
    refs = _ref_envs(net, prof, idx, start, e0, a0, raw, injected) if kind == "f64" else []
    for e, r in zip(idx, refs):
        assert np.max(np.abs(env.voltages[e].cpu().numpy() - r._get_bus_v())) < 1e-8
    rng = np.random.default_rng(12)
    violations = failures = 0
    for t in range(env.episode_limit - 1):
        a = actions(kind, rng, (n, na, 4), 0.4)
        inj = mask = None
        if t == 30:
            a[::13, 0, 1] = np.nan
        if t == 50:
            inj = np.zeros(n, dtype=np.uint8); inj[3::17] = 1
            env.inject_failure(inj); injected[0] = inj
        if t == 70:
            mask = (rng.uniform(size=n) < 0.6).astype(np.uint8); mask[0] = 1; mask[n - 1] = 0
        r, d, info = env.step(torch.from_numpy(a), mask=mask, translate=kind == "policy")
        rr, dd, ii = mb.step(mirror_actions(kind, a), inject=inj, mask=mask)
        sel = slice(None) if mask is None else mask.astype(bool)
        assert np.array_equal(r.cpu().numpy()[sel], rr[sel]), t
        assert np.array_equal(d.cpu().numpy()[sel], dd[sel]), t
        got = np.stack([info[k].cpu().numpy() for k in INFO_KEYS], 1)
        assert np.array_equal(got[sel], ii[sel]), t
        check_state(env, mb, f"step {t}")
        violations += int(mb.vcount.sum()); failures += int(ii[:, 7].sum())
        for e, ref in zip(idx, refs):
            if mask is not None and not mask[e]:
                continue
            rw, dn, inf = ref.step(mirror_actions(kind, a[e]).reshape(-1))
            assert abs(rr[e] - rw) <= 1e-6 * abs(rw) + 1e-12, (t, e, rr[e], rw)
            assert bool(dd[e]) == dn, (t, e)
            assert (ii[e, 7] == 1.0) == bool(inf.get("solver_failed", False)), (t, e)
            assert np.max(np.abs(mb.V[e] - ref._get_bus_v())) < 1e-8, (t, e)
            assert np.max(np.abs(mb.E_cur[e] - ref._get_ess_energy())) < 1e-15, (t, e)
        if inj is not None:
            env.inject_failure(None); injected[0] = None
    assert bool(env.steps.cpu().numpy().max() == env.episode_limit)
    assert failures >= n // 13, failures
    assert violations > 0 or name == "custom14", violations        # custom14's light loads stay inside the band at 2.4x
    env.close()


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_preview_equals_step_and_mirror(cuda, case):
    """preview_step with K = 1 and K = 3 (fp32, fp64 and translated candidates) returns the following step's reward,
    done, info, voltages and mask, and the mirror's; the handle's bytes are unchanged by the previews."""
    name, variant = case
    net = F.feeder(name)
    prof = _heavy(net)
    n = 32 * 3 + 5
    env = make_env(cuda, prof, n, variant, net=net)
    na = env.n_agents
    fonet = c_mirror.make_net(ieee33.tree_arrays(net), F.env_args(net, variant), net['buildings'], variant=_variant(variant))
    mb = c_mirror.MirrorBatch(fonet, prof.as_dict(), n)
    reset_both(env, mb, np.random.default_rng(31))
    env.keep_line_flows(True)
    rng = np.random.default_rng(32)
    for t, kind in enumerate(["f32", "f64", "policy", "f32", "f64"]):
        k = 1 if t % 2 == 0 else 3
        cand = actions(kind, rng, (k, n, na, 4), 0.4)
        cand[k - 1, ::11, 0, 2] = np.nan
        before = F.snapshot(env)
        c = torch.from_numpy(cand if k > 1 else cand[0])
        r, d, info, V, vm = env.preview_step(c, translate=kind == "policy", want_voltage=True, want_mask=True)
        F.assert_same_bytes(before, F.snapshot(env))
        r, d, V, vm = (x.reshape(k, n, *x.shape[(2 if k > 1 else 1):]) for x in (r, d, V, vm))
        info = {key: v.reshape(k, n) for key, v in info.items()}
        saved = mirror_copy(mb)
        for j in range(k):                                          # the mirror's step for each candidate, then undone
            rr, dd, ii = mb.step(mirror_actions(kind, cand[j]))
            assert np.array_equal(r[j].cpu().numpy(), rr) and np.array_equal(d[j].cpu().numpy(), dd), (t, j)
            assert np.array_equal(np.stack([info[key][j].cpu().numpy() for key in INFO_KEYS], 1), ii)
            assert np.array_equal(V[j].cpu().numpy(), mb.V) and np.array_equal(vm[j].cpu().numpy().view(np.uint64), mb.vmask)
            mirror_restore(mb, saved)
        j = k - 1                                                   # commit the last candidate
        rs, ds, infos = env.step(torch.from_numpy(cand[j]), translate=kind == "policy")
        mb.step(mirror_actions(kind, cand[j]))
        assert torch.equal(bits(r[j]), bits(rs)) and torch.equal(d[j], ds), t
        for key in infos:
            assert torch.equal(bits(info[key][j]), bits(infos[key])), (t, key)
        assert torch.equal(bits(V[j]), bits(env.voltages)) and torch.equal(vm[j], env.violation_mask), t
        check_state(env, mb, f"step {t}")
    env.close()


@pytest.mark.parametrize("variant", ["thread", "warp"])
@pytest.mark.parametrize("name", ["chain33", "ieee33_4agents", "two_bus", "limits_16x8"])
def test_observations_and_host_step(cuda, name, variant):
    """step(return_obs=True) and step(return_obs="ring") equal step + get_obs / obs_ring().dense(); step_host through
    the zero-copy route (pinned fp32) and the staged route (pageable, fp64) equals step bit for bit."""
    net = F.feeder(name)
    prof = _heavy(net)
    n = 32 * 4 + 9
    envs = [make_env(cuda, prof, n, variant, net=net) for _ in range(3)]
    na = envs[0].n_agents
    start, e0, a0 = draws(41, envs[0])
    for env in envs:
        env.reset(start, e0, a0, return_obs=False)
    rng = np.random.default_rng(42)
    for t in range(30):
        a = actions("f32" if t % 3 else "f64", rng, (n, na, 4), 0.4)
        if t == 10:
            a[::7, na - 1, 0] = np.nan
        r0, d0, i0 = envs[0].step(torch.from_numpy(a))
        o0 = envs[0].get_obs()
        if t % 2 == 0:
            r1, d1, i1, o1 = envs[1].step(torch.from_numpy(a), return_obs=True)
        else:
            r1, d1, i1, ring = envs[1].step(torch.from_numpy(a), return_obs="ring")
            o1 = ring.dense()
        assert torch.equal(bits(r0), bits(r1)) and torch.equal(d0, d1), t
        assert torch.equal(o0, o1), t
        assert torch.equal(envs[0].rec, envs[1].rec) and torch.equal(bits(envs[0].voltages), bits(envs[1].voltages)), t
        if a.dtype == np.float32:
            h = torch.from_numpy(a.reshape(n, -1)).pin_memory().numpy()    # zero-copy
        else:
            h = a.reshape(n, -1).copy()                                      # staged
        r2, d2, i2 = envs[2].step_host(h, want_info=True)
        assert torch.equal(envs[2].get_obs(), o0), t                 # the same push as the other two envs
        assert np.array_equal(r2, r0.cpu().numpy()) and np.array_equal(d2, d0.cpu().numpy()), t
        for k in i0:
            assert np.array_equal(i2[k], i0[k].cpu().numpy()), (t, k)
        assert torch.equal(envs[0].rec, envs[2].rec) and torch.equal(bits(envs[0].voltages), bits(envs[2].voltages)), t
    for env in envs:
        env.close()


def _safety_env(cuda, net, n, seed):
    env = make_env(cuda, feeder_profiles(net), n, "thread", net=net)
    na = env.n_agents
    env.reset(*draws(seed, env), return_obs=False)
    g = torch.Generator(device=cuda).manual_seed(seed)
    for _ in range(3):
        env.step(torch.rand(n, na, 4, device=cuda, generator=g), want_info=False)
    actions = torch.randn(n, na, 4, device=cuda, generator=g) * 0.6 + 0.4           # raw policy outputs, some outside [0, 1]
    return env, actions


SAFETY_FEEDERS = ["two_bus", "custom14", "chain33", "slack_star", "ieee33_4agents"]      # 1, 3, 5, 2 and 4 agents


@pytest.mark.parametrize("name", SAFETY_FEEDERS)
def test_safety_project_on_other_feeders(cuda, args, name):
    """fp_safety_project (row sums of the fitted map) against the closed form, with the feeder's LinDistFlow map."""
    net = F.feeder(name)
    n = 32 * 5 + 3
    env, actions = _safety_env(cuda, net, n, 51)
    nb, na = env.n_bus, env.n_agents
    A, _ = F.lindistflow_map(ieee33.tree_arrays(net))
    coef = np.hstack([A[:, 0::2], A[:, 1::2]]) * 20.0                  # the reference's [W_P | W_Q] layout
    icpt = 1.0 + np.random.default_rng(52).uniform(-0.12, 0.12, nb)
    env.load_safety_model(coef, icpt)
    adj, slack, moved = env.safety_project(actions, want_info=True)
    adj_agent = env.safety_project(actions, layout="agent")
    assert adj.shape == (n, 4 * na) and adj_agent.shape == (n, na, 4)
    assert torch.equal(adj.view(n, 4, na).permute(0, 2, 1), adj_agent)
    st = env.get_state(torch.float64).cpu().numpy()
    a_np, adj_np, slack_np, moved_np = actions.double().cpu().numpy(), adj.cpu().numpy(), slack.cpu().numpy(), moved.cpu().numpy()
    n_moved = 0
    for e in range(n):
        ref = F.ref_stub(net, args, st[e])
        want, wslack, wlam = safety_ref.safety_layer(ref, a_np[e], coef, icpt)
        assert np.max(np.abs(adj_np[e] - want) / np.maximum(1.0, np.abs(want))) < 1e-6, (e, adj_np[e], want)
        assert np.allclose(slack_np[e], wslack, rtol=1e-9, atol=1e-12), e
        assert np.array_equal(moved_np[e], wlam > 0), e
        n_moved += int((wlam > 0).sum())
    assert n_moved > 0
    env.close()


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("map_kind", ["lindistflow", "dense"])
@pytest.mark.parametrize("name", SAFETY_FEEDERS)
def test_safety_project_affine_on_other_feeders(cuda, args, name, map_kind, dtype):
    """fp_safety_project_affine against the active-set restatement on the feeder's LinDistFlow map and on a random dense
    map, limits placed so that a good share of the envs is pushed outside; on 3 envs also against the posed QP."""
    net = F.feeder(name)
    n = 32 * 5 + 3
    env, actions = _safety_env(cuda, net, n, 61)
    nb, na = env.n_bus, env.n_agents
    tree = ieee33.tree_arrays(net)
    if map_kind == "lindistflow":
        A, c = F.lindistflow_map(tree)
    else:
        rng = np.random.default_rng(62)
        A = -rng.uniform(0.0, 0.02, (nb, 2 * nb)); c = np.ones(nb)
    st = env.get_state(torch.float64).cpu().numpy()
    x = np.empty((n, 2 * nb)); x[:, 0::2] = st[:, :nb]; x[:, 1::2] = st[:, nb:2 * nb]
    Vp = x @ A.T + c
    v_min, v_max = float(np.quantile(Vp.min(1), 0.3)), float(np.quantile(Vp.max(1), 0.85))
    if v_max <= v_min:
        v_max = v_min + 1e-3
    env.load_safety_map(A, c, v_min=v_min, v_max=v_max)
    a = actions.to(dtype)
    adj, slack, moved, status = env.safety_project_affine(a, want_info=True)
    adj_agent = env.safety_project_affine(a, layout="agent")
    assert adj.shape == (n, 4 * na) and slack.shape == (n, nb) and status.shape == (n,)
    assert torch.equal(adj.view(n, 4, na).permute(0, 2, 1), adj_agent)
    assert bool((status >= 0).all())
    bus = np.array([net['bus_numbers'].index(b) for b in net['buildings']])
    is_b = -np.ones(nb, dtype=int); is_b[bus] = np.arange(na)
    a_np, adj_np, slack_np, moved_np, status_np = (t.cpu().numpy() for t in (a.double(), adj, slack, moved, status))
    moved_envs = []
    for e in range(n):
        ref = F.ref_stub(net, args, st[e])
        pct, ch, dis, qpv = safety_ref.parse_actions(ref, a_np[e])
        y0 = np.array([[pct[b], ch[b], dis[b], qpv[b]] for b in net['buildings']])
        want, wslack, wstatus = safety_affine_ref.project_affine(y0, st[e, :nb], st[e, nb:2 * nb], bus, A, c, v_min, v_max)
        want_tm = want.T.reshape(-1)
        assert np.max(np.abs(adj_np[e] - want_tm) / np.maximum(1.0, np.abs(want_tm))) < 1e-6, (e, adj_np[e], want_tm)
        assert np.allclose(slack_np[e], wslack, rtol=1e-9, atol=1e-9), (e, slack_np[e], wslack)
        assert (status_np[e] == 0) == (wstatus == 0), (e, status_np[e], wstatus)
        assert np.array_equal(moved_np[e], (want != y0).any(axis=1)), e
        if wstatus > 0:
            moved_envs.append((e, y0, want))
    assert 0 < len(moved_envs) < n
    if map_kind == "lindistflow" and dtype == torch.float64:
        for e, y0, got in moved_envs[:3]:                           # the QP handed to a generic solver
            qp, _ = safety_affine_ref.solve_affine_qp(y0, st[e, :nb], st[e, nb:2 * nb], is_b, A, c, v_min, v_max)
            cost = lambda y: safety_affine_ref.affine_cost(y, y0, st[e, :nb], st[e, nb:2 * nb], bus, A, c, v_min, v_max)
            assert cost(got) <= cost(qp) * (1 + 1e-7) + 1e-9, e
            # the cost is ||y - y0||^2 plus convex penalties: at the minimiser y*, cost(y) >= cost(y*) + ||y - y*||^2,
            # so the generic solver's point can sit no further from ours than its excess cost allows
            assert np.sum((got - qp) ** 2) <= max(cost(qp) - cost(got), 0.0) + 1e-12, e
    env.close()


@pytest.mark.parametrize("name", ["over_17_chains", "over_9_slots"])
def test_thread_variant_rejects_feeders_beyond_its_limits(cuda, name):
    from flexgpu import FlexGpuError
    net = F.feeder(name)
    with pytest.raises(FlexGpuError, match="use FP_VARIANT_WARP"):
        make_env(cuda, feeder_profiles(net), 64, "thread", net=net)
    env = make_env(cuda, feeder_profiles(net), 64, "warp", net=net)    # the warp variant runs it (tests above: parity)
    env.close()


def _bad_feeders():
    base = F.custom14()
    out = {}
    lines = [(i, i + 1, .1, .05) for i in range(1, 34)]                # 34 buses
    out["34_buses"] = F.make_network(lines, {}, [5])
    out["agent_on_slack"] = dict(base, buildings=[1, 9, 14], PVs_at_buildings=[1, 9, 14], ESSs_at_buildings=[1, 9, 14])
    out["two_agents_one_bus"] = dict(base, buildings=[9, 9, 14], PVs_at_buildings=[9, 9, 14], ESSs_at_buildings=[9, 9, 14])
    return out


@pytest.mark.parametrize("variant", ["thread", "warp"])
def test_create_rejects_invalid_feeders(cuda, variant):
    """34 buses, an agent on the slack bus, two agents on one bus (through the env), and a parent array that is
    disconnected or cyclic (through fp_create itself, since the network dict cannot express either)."""
    import ctypes as C
    from flexgpu import FlexGpuError, _lib
    from flexgpu.config import make_fp_config, normalize_args
    from flexgpu.network import Network
    for key, net in _bad_feeders().items():
        with pytest.raises((FlexGpuError, ValueError)):
            make_env(cuda, None if key == "34_buses" else feeder_profiles(net), 8, variant, net=net)
    net = F.custom14()
    network = Network(net)
    lib = _lib.lib()
    for bad in ("cycle", "disconnected", "self"):
        cfg = make_fp_config(normalize_args(F.env_args(net, variant)), network)
        if bad == "cycle":                                          # 8 -> 9 -> 8: neither reaches the slack bus
            cfg.parent[network.position[8]] = network.position[9]
        elif bad == "disconnected":                                 # bus 11 and its subtree hang from nothing
            cfg.parent[network.position[11]] = -1
        else:
            cfg.parent[network.position[5]] = network.position[5]
        h = C.c_void_p()
        assert lib.fp_create(C.byref(cfg), 8, 0, C.byref(h)) != 0, bad
        assert not h.value
    cfg = make_fp_config(normalize_args(F.env_args(net, variant)), network)     # the unmodified config is accepted
    h = C.c_void_p()
    assert lib.fp_create(C.byref(cfg), 8, 0, C.byref(h)) == 0
    lib.fp_destroy(h)
