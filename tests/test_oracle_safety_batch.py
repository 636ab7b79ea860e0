"""CPU: the batch restatement of the safety layer (tests/_safety_batch_ref.py, what test_gpu_safety_scale.py checks every
row against) equals the scalar oracle (oracle/safety_ref.py, oracle/safety_affine_ref.py) bit for bit, NaN positions
included (zeros of either sign compare equal), on 20 000 (env, agent) cases built around the edges: NaN in each action component, +-inf, +-1e30, exact 0 and
1, PV = 0, ESS energy at e_min and e_max, charge above and below discharge with both positive, and row sums of either
sign and zero."""
import numpy as np
import pytest

import _safety_batch_ref as B
from oracle import env_ref, ieee33, safety_affine_ref, safety_ref

NA = 5
N_ENVS = 4000                                                   # x 5 agents = 20 000 cases


def _stub(args, pv, e_now):
    ref = env_ref.RefFlexEnv.__new__(env_ref.RefFlexEnv)
    ref.args = env_ref._Args(dict(args))
    ref.base_powergrid = ieee33.create_network()
    G = ref.base_powergrid
    ref.current_pv_power = {b: float(pv[i]) for i, b in enumerate(G['PVs_at_buildings'])}
    ref.current_ess_energy = {b: float(e_now[i]) for i, b in enumerate(G['ESSs_at_buildings'])}
    return ref


def _edge_cases(args, rng, n):
    """Actions [n, NA, 4], PV and E [n, NA] mixing every edge per (env, agent)."""
    a = rng.uniform(-0.5, 1.5, (n, NA, 4))
    kind = rng.integers(0, 10, (n, NA))
    comp = rng.integers(0, 4, (n, NA))
    pick = lambda k: kind == k
    a[pick(1)] = rng.choice([0.0, 1.0], (int(pick(1).sum()), 4))
    a[pick(2)] = rng.choice([-1e30, 1e30], (int(pick(2).sum()), 4))
    a[pick(3)] = rng.choice([-np.inf, np.inf, 0.5], (int(pick(3).sum()), 4))
    m = pick(4)                                                 # one NaN component, each of the four
    a[m, comp[m]] = np.nan
    m = pick(5)                                                 # charge and discharge both positive, either larger
    a[m, 1] = rng.uniform(0.01, 1.2, int(m.sum())); a[m, 2] = rng.uniform(0.01, 1.2, int(m.sum()))
    m = pick(6)
    a[m, 3] = rng.choice([-np.inf, np.inf], int(m.sum()))      # a3 = +-inf (NaN where PV = 0)
    m = pick(7)
    a[m] = a[m] + 1e-12                                         # fp64 values fp32 cannot hold
    m = pick(8)                                                 # equal charge and discharge
    a[m, 2] = a[m, 1]
    pv = rng.uniform(0.0, 0.3, (n, NA))
    pv[rng.random((n, NA)) < 0.3] = 0.0                         # night
    e = rng.uniform(args["e_min"], args["e_max"], (n, NA))
    r = rng.random((n, NA))
    e[r < 0.15] = args["e_min"]; e[r > 0.85] = args["e_max"]
    return a, pv, e


def _same(x, y):
    """Bit for bit, NaN positions included, up to the sign of a zero: numpy.clip itself returns -0.0 or +0.0 for a -0.0 on
    a zero-width range [-0.0, 0.0] (qpv at PV = 0) depending on whether its bounds are scalars or arrays."""
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    return np.array_equal(np.isnan(x), np.isnan(y)) and np.array_equal(x[~np.isnan(x)], y[~np.isnan(y)])


def test_parse_and_closed_form_equal_the_scalar_oracle(args):
    rng = np.random.default_rng(101)
    a, pv, e = _edge_cases(args, rng, N_ENVS)
    y0 = B.parse_actions(args, pv, e, a)
    G = ieee33.create_network()
    want = np.empty_like(y0)
    for i in range(N_ENVS):
        pct, ch, dis, qpv = safety_ref.parse_actions(_stub(args, pv[i], e[i]), a[i])
        want[i] = [[pct[b], ch[b], dis[b], qpv[b]] for b in G['buildings']]
    assert _same(y0, want)
    # the cases really reach the edges
    assert np.isnan(y0).any(axis=-1).sum() > 1000
    for c in range(4):
        assert np.isnan(y0[..., c]).sum() > 100, c
    assert np.isnan(y0[..., 3][pv == 0]).any() and not np.isnan(y0[..., 3][(pv > 0) & ~np.isnan(a[..., 3])]).any()
    assert ((y0[..., 1] == args["p_ch_max"]) & (e == args["e_min"])).any()
    # the row-sum projection, with sP / sQ negative, zero and positive and demands placing V0 around both limits
    Pd = rng.uniform(0.0, 0.4, (N_ENVS, NA)); Qd = rng.uniform(-0.1, 0.2, (N_ENVS, NA))
    sP = rng.choice([-0.9, -0.3, 0.0, 0.2, 0.7], (N_ENVS, NA)) * rng.uniform(0.5, 1.0, (N_ENVS, NA))
    sQ = rng.choice([-0.6, -0.1, 0.0, 0.1, 0.5], (N_ENVS, NA)) * rng.uniform(0.5, 1.0, (N_ENVS, NA))
    target = rng.choice([0.85, 0.899, 0.95, 1.0, 1.05, 1.101, 1.15, -40.0, 40.0], (N_ENVS, NA))
    with np.errstate(all="ignore"):
        b = target - (sP * (Pd * (1.0 - np.nan_to_num(y0[..., 0])) + np.nan_to_num(y0[..., 1]) - np.nan_to_num(y0[..., 2]))
                      + sQ * (Qd + np.nan_to_num(y0[..., 3])))
    y, slack, lam = B.project_rowsum(y0, Pd, Qd, sP, sQ, b, 0.9, 1.1)
    wy, wslack, wlam = np.empty_like(y), np.empty_like(slack), np.empty_like(lam)
    for i in range(N_ENVS):
        for k in range(NA):
            wy[i, k], wslack[i, k], wlam[i, k] = safety_ref.project_closed_form(y0[i, k], Pd[i, k], Qd[i, k], sP[i, k], sQ[i, k],
                                                                                b[i, k], 0.9, 1.1)
    assert _same(y, wy) and _same(slack, wslack) and _same(lam, wlam)
    assert not (lam[np.isnan(y0).any(axis=-1)] > 0).any() and not slack[np.isnan(y0).any(axis=-1)].any()
    moved = lam > 0
    assert 2000 < moved.sum() < 18000 and (slack > 0).sum() > 500 and (lam == safety_ref.W_SLACK).any()


@pytest.mark.parametrize("pool", [False, True])
def test_affine_batch_equals_the_scalar_restatement(args, pool):
    """Inside, moved, hopeless and NaN envs of one batch: the GEMV classification plus the scalar restatement equal the
    scalar restatement on every env; with worker processes the same."""
    rng = np.random.default_rng(102)
    n, NB = 240, 33
    bus = np.array([4, 9, 14, 19, 24])
    a, pv, e = _edge_cases(args, rng, n)
    y0 = B.parse_actions(args, pv, e, a)
    Pd = rng.uniform(0.02, 0.4, (n, NB)); Qd = rng.uniform(0.01, 0.2, (n, NB)); Pd[:, 0] = Qd[:, 0] = 0.0
    A = -rng.uniform(0.0, 0.02, (NB, 2 * NB))
    A[:, 2 * bus] -= rng.uniform(0.005, 0.06, (NB, 5)); A[:, 2 * bus + 1] -= rng.uniform(0.002, 0.04, (NB, 5))
    c = np.ones(NB)
    V, _ = B.affine_prediction(y0, Pd, Qd, bus, A, c)
    ok = np.isfinite(V).all(axis=1)
    mixed = (float(np.quantile(V[ok].min(1), 0.3)), float(np.quantile(V[ok].max(1), 0.85)))
    hopeless = (float(V[ok].max()) + 50.0, float(V[ok].max()) + 60.0)
    for v_min, v_max in (mixed, hopeless):
        if pool:
            with B.AffinePool(2) as p:
                y, slack, st, n_run = B.project_affine(y0, Pd, Qd, bus, A, c, v_min, v_max, pool=p, chunk=16)
        else:
            y, slack, st, n_run = B.project_affine(y0, Pd, Qd, bus, A, c, v_min, v_max)
        assert 0 < n_run <= ok.sum()
        for i in range(n):
            wy, ws, wst = safety_affine_ref.project_affine(y0[i], Pd[i], Qd[i], bus, A, c, v_min, v_max)
            assert _same(y[i], wy) and _same(slack[i], ws) and st[i] == wst, i
        assert (st[ok] > 0).any() and (v_min > 10.0 or (st[ok] == 0).any())
        nan_env = np.isnan(y0).any(axis=(1, 2))
        assert nan_env.any() and not st[nan_env].any() and not slack[nan_env].any()
        assert not B.bits_moved(y, y0)[nan_env].any()
