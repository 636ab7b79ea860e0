"""GPU: both safety kernels at rollout scale, every row against the fp64 batch restatement (tests/_safety_batch_ref.py,
itself equal to the scalar oracle by tests/test_oracle_safety_batch.py).

  * k_safety_project (row sums, one thread per (env, agent), grid capped at 148 x 16 CTAs of 256 threads = 606 208
    threads): N = 1, 7, 121 241, 121 242 (the first N whose grid-stride loop wraps at five agents), 131 072, 262 147.
  * k_safety_project_affine (one warp per env, 8 envs a CTA): N = 1, 9, 2 367, 2 369 (either side of one resident wave,
    2 CTAs/SM x 148 SMs x 8 envs = 2 368), 131 072; four maps (the reference's fit with its scalers folded in,
    LinDistFlow, the banded row-sum map, LinDistFlow with one building's two columns zeroed) and three limit mixes
    (inside, mixed, hopeless, as tools/bench_safety.py places them).
  * One batch per size holds envs at episode steps 0, 1, 2, mid-episode, 95, 96 and past termination (the row in
    force clamps), envs whose last step failed and rolled back, night rows, and ESS energies driven to and placed at
    e_min and e_max.  Actions mix U(-0.5, 1.5), exact 0 and 1, +-1e30, +-inf (also a3 at PV = 0), one NaN component,
    and fp64 values fp32 cannot hold; fp32 and fp64 actions, both layouts, every optional output left NULL alone and
    in every combination, on a non-default stream.
  * Both layers on five catalogue feeders (one to five agents) at 20 000 envs.
  * Every output sits in a NaN-sentinel allocation with a guard band behind it: every element must be written, the
    guard band must come back untouched.  Two launches are bit-identical; poisoning one env's actions changes only that
    env's outputs.

Bars: setpoints 1e-6 relative (floor 1; fp32 outputs), slack 1e-9, `intervened` and `status == 0` exact, NaN positions
exact, and an env or agent the layer leaves alone is the parsed proposal cast to fp32, equal element for element.
NaN contract (include/flexgpu.h): a proposal that is NaN after parse_actions is returned as parsed; the row-sum layer
does not project that agent, the affine layer not that env (slack 0, status 0, intervened 0).

The affine restatement runs the scalar active-set method on every env not clearly inside the limits, in spawned worker
processes; that dominates this file's wall time: 31 s for the whole file on an NVIDIA B200 (1000 W power limit) host
with 16 CPU cores."""
import ctypes as C
import itertools
import os

import numpy as np
import pytest
import torch

import _feeders as F
import _safety_batch_ref as B
from _env_check import feeder_profiles, make_env, ptr
from oracle import ieee33, safety_ref

pytestmark = pytest.mark.gpu

SENT = {torch.float32: 0x7FA5A5A5, torch.float64: 0x7FF5A5A5A5A5A5A5, torch.uint8: 0xA5, torch.int32: 0x5A5A5A5A}
INT_OF = {torch.float32: torch.int32, torch.float64: torch.int64, torch.uint8: torch.uint8, torch.int32: torch.int32}
GUARD = 256
RS_SIZES = [1, 7, 121241, 121242, 131072, 262147]
AF_SIZES = [1, 9, 2367, 2369, 131072]
MAPS = ["reference_fit", "lindistflow", "banded", "lindistflow_zeroed"]
LIMITS = ["inside", "mixed", "hopeless"]
FEEDERS = ["two_bus", "slack_star", "custom14", "ieee33_4agents", "chain33"]
L_DRIVE = 130                                           # driving iterations: past the row-in-force clamp (121 steps)
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_predictor.npz")


# ------------------------------------------------------------------ sentinel-filled outputs
class _Out:
    """n elements of `dtype` inside an allocation filled with a sentinel bit pattern, GUARD more behind them."""

    def __init__(self, n, dtype, device):
        self.n, self.dtype = n, dtype
        self.buf = torch.empty(n + GUARD, dtype=dtype, device=device)
        self.buf.view(INT_OF[dtype]).fill_(SENT[dtype])
        self.view = self.buf[:n]

    def ptr(self):
        return C.c_void_p(self.view.data_ptr())

    def check(self, what):
        bits = self.buf.view(INT_OF[self.dtype])
        s = SENT[self.dtype]
        assert bool((bits[self.n:] == s).all()), f"{what}: a write past the end of the output"
        assert not bool((bits[:self.n] == s).any()), f"{what}: an element was not written"


@pytest.fixture(scope="module")
def stream(cuda):
    return torch.cuda.Stream(device=cuda)


def _rowsum(env, actions, tm, stream, slack=True, moved=True):
    """fp_safety_project through the C ABI on `stream`; returns the host copies (out [N, na, 4] fp32 in the agent
    layout, slack [N, na] or None, moved [N, na] or None) and the raw buffers."""
    N, na = env.n_envs, env.n_agents
    dev = env.device
    o = _Out(N * na * 4, torch.float32, dev)
    s = _Out(N * na, torch.float64, dev) if slack else None
    m = _Out(N * na, torch.uint8, dev) if moved else None
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        env._check(env._lib.fp_safety_project(env._h, ptr(actions), 1 if actions.dtype == torch.float64 else 0, o.ptr(),
                                              1 if tm else 0, s.ptr() if s else None, m.ptr() if m else None,
                                              C.c_void_p(stream.cuda_stream)), "fp_safety_project")
    stream.synchronize()
    for b, w in ((o, "adjusted"), (s, "slack"), (m, "intervened")):
        if b is not None:
            b.check(w)
    out = o.view.view(N, 4, na).permute(0, 2, 1) if tm else o.view.view(N, na, 4)
    return (out.cpu().numpy(), None if s is None else s.view.view(N, na).cpu().numpy(),
            None if m is None else m.view.view(N, na).cpu().numpy()), (o, s, m)


def _affine(env, actions, tm, stream, slack=True, moved=True, status=True):
    N, na, nb = env.n_envs, env.n_agents, env.n_bus
    dev = env.device
    o = _Out(N * na * 4, torch.float32, dev)
    s = _Out(N * nb, torch.float64, dev) if slack else None
    m = _Out(N * na, torch.uint8, dev) if moved else None
    st = _Out(N, torch.int32, dev) if status else None
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        env._check(env._lib.fp_safety_project_affine(env._h, ptr(actions), 1 if actions.dtype == torch.float64 else 0, o.ptr(),
                                                     1 if tm else 0, s.ptr() if s else None, m.ptr() if m else None,
                                                     st.ptr() if st else None, C.c_void_p(stream.cuda_stream)),
                   "fp_safety_project_affine")
    stream.synchronize()
    for b, w in ((o, "adjusted"), (s, "slack"), (m, "intervened"), (st, "status")):
        if b is not None:
            b.check(w)
    out = o.view.view(N, 4, na).permute(0, 2, 1) if tm else o.view.view(N, na, 4)
    return (out.cpu().numpy(), None if s is None else s.view.view(N, nb).cpu().numpy(),
            None if m is None else m.view.view(N, na).cpu().numpy(), None if st is None else st.view.cpu().numpy()), (o, s, m, st)


# ------------------------------------------------------------------ the batch: every episode position at once
def _roles(N, seed):
    """Role of each env (0: step 0, 1: step 1, 2: step 2, 3: mid-episode, 4: step 95, 5: step 96 or past termination,
    6: last step failed, 7: ESS runs) and the steps since its last reset (-1: only the initial one).  A reset sets the
    record's step counter to 1, so the counter reads steps + 1."""
    rng = np.random.default_rng(seed)
    role = (np.arange(N) * 5 + rng.integers(0, 8)) % 8 if N < 64 else rng.integers(0, 8, N)
    k = np.select([role == 0, role == 1, role == 2, role == 3, role == 4, role == 6, role == 7],
                  [0, 1, 2, rng.integers(3, 95, N), 95, rng.integers(1, 60, N), 45], default=-1)
    k[(role == 5) & (rng.random(N) < 0.3)] = 96                        # done on its last step
    return role, k


def _drive(env, seed):
    """Staggered masked resets and steps: env e ends k_e steps after its last reset (past termination when it never
    resets), the failing envs' last step is a solver failure, the ESS envs charge or discharge at full power."""
    N, na = env.n_envs, env.n_agents
    dev = env.device
    role, k = _roles(N, seed)
    rng = np.random.default_rng(seed + 1)
    charge = rng.random(N) < 0.5
    env.reset(return_obs=False)
    g = torch.Generator(device=dev).manual_seed(seed)
    ess = torch.as_tensor(role == 7, device=dev)
    full = torch.zeros(N, na, 4, dtype=torch.float64, device=dev)
    full[:, :, 1] = torch.as_tensor(charge, device=dev)[:, None].double()
    full[:, :, 2] = 1.0 - full[:, :, 1]
    for t in range(L_DRIVE):
        rs = (k >= 0) & (L_DRIVE - k == t)
        if rs.any():
            env.reset(mask=torch.as_tensor(rs.astype(np.uint8), device=dev), return_obs=False)
        if t == L_DRIVE - 1:
            env.inject_failure(torch.as_tensor((role == 6).astype(np.uint8), device=dev))
        a = torch.rand(N, na, 4, device=dev, generator=g, dtype=torch.float64)
        a = torch.where(ess[:, None, None], full, a)
        env.step(a, want_info=False)
    env.inject_failure(torch.zeros(N, dtype=torch.uint8, device=dev))
    rs = k == 0
    if rs.any():
        env.reset(mask=torch.as_tensor(rs.astype(np.uint8), device=dev), return_obs=False)
    # ESS energies placed exactly at the limits on some agents
    r = torch.as_tensor(rng.random((N, na)), device=dev)
    E = env.ess_energy
    E[r < 0.06] = float(env.args_dict["e_min"]); E[r > 0.94] = float(env.args_dict["e_max"])
    torch.cuda.synchronize()
    return role


def _actions(N, na, pv, seed):
    """fp64 raw actions [N, na, 4] mixing the edges per (env, agent)."""
    rng = np.random.default_rng(seed)
    a = rng.uniform(-0.5, 1.5, (N, na, 4))
    kind = rng.integers(0, 16, (N, na))                       # 9..15: U(-0.5, 1.5) alone
    comp = rng.integers(0, 4, (N, na))
    n_of = lambda m: int(m.sum())
    m = kind == 1; a[m] = rng.choice([0.0, 1.0], (n_of(m), 4))
    m = kind == 2; a[m] = rng.choice([-1e30, 1e30, 0.3], (n_of(m), 4))
    m = kind == 3; a[m] = rng.choice([-np.inf, np.inf, 0.6], (n_of(m), 4))
    m = kind == 4; a[m, comp[m]] = np.nan
    m = kind == 5; a[m] = a[m] + 1e-12 * rng.choice([-1.0, 1.0], (n_of(m), 4))
    m = (kind == 6) | ((kind == 7) & (pv == 0)); a[m, 3] = rng.choice([-np.inf, np.inf], n_of(m))
    m = kind == 8; a[m, 1] = rng.uniform(0.01, 1.2, n_of(m)); a[m, 2] = rng.uniform(0.01, 1.2, n_of(m))
    return a


class Batch:
    def __init__(self, env, role, seed):
        self.env, self.role = env, role
        N, na, nb = env.n_envs, env.n_agents, env.n_bus
        self.state = env.get_state(torch.float64).cpu().numpy()
        self.P, self.Q, self.PV, self.E = B.split_state(self.state, nb, na)
        self.bus = np.array([env.base_powergrid['bus_numbers'].index(b) for b in env.agent_ids])
        self.args = env.args_dict
        a64 = _actions(N, na, self.PV, seed)
        self.act = {torch.float64: torch.as_tensor(a64, device=env.device),
                    torch.float32: torch.as_tensor(a64.astype(np.float32), device=env.device)}
        with np.errstate(all="ignore"):
            self.y0 = {dt: B.parse_actions(self.args, self.PV, self.E, a.cpu().numpy().astype(np.float64))
                       for dt, a in self.act.items()}


_CACHE = {}


def _batch(cuda, profiles, N, net=None, name=None):
    key = (name or "ieee33", N)
    if key not in _CACHE:
        seed = 1000 + N % 977
        env = make_env(cuda, profiles if net is None else feeder_profiles(net), N, net=net, seed=seed)
        role = _drive(env, seed)
        _CACHE[key] = Batch(env, role, seed + 7)
    return _CACHE[key]


@pytest.fixture(scope="module", autouse=True)
def _close_batches():
    yield
    for b in _CACHE.values():
        b.env.close()
    _CACHE.clear()


@pytest.fixture(scope="module")
def pool():
    with B.AffinePool() as p:
        yield p


# ------------------------------------------------------------------ models, maps and limits
def _rowsum_model(b, kind):
    nb = b.env.n_bus
    if nb == 33 and kind == "reference_fit":
        g = np.load(GOLD)
        return g["coef"].astype(np.float64), g["intercept"].astype(np.float64)
    A, _ = F.lindistflow_map(ieee33.tree_arrays(b.env.base_powergrid))
    return np.hstack([A[:, 0::2], A[:, 1::2]]) * 20.0, 1.0 + np.random.default_rng(52).uniform(-0.12, 0.12, nb)


def _affine_map(b, name):
    env = b.env
    g = np.load(GOLD)
    if name == "reference_fit":
        from flexgpu.predictor import VoltagePredictor
        pred = VoltagePredictor.from_linear_model(env, g["coef"], g["intercept"], g["x_scale"], g["x_min"], g["y_scale"], g["y_min"])
        return np.array(pred.A, dtype=np.float64), np.array(pred.c, dtype=np.float64)
    if name == "banded":
        coef = g["coef"].astype(np.float64)
        n = coef.shape[0]
        A = np.zeros((n, 2 * n)); A[np.arange(n), 2 * np.arange(n)] = coef[:, :n].sum(1)
        A[np.arange(n), 2 * np.arange(n) + 1] = coef[:, n:].sum(1)
        return A, g["intercept"].astype(np.float64)
    A, c = F.lindistflow_map(ieee33.tree_arrays(env.base_powergrid))
    if name == "lindistflow_zeroed":
        k = min(1, len(b.bus) - 1)
        A = A.copy(); A[:, 2 * b.bus[k]] = 0.0; A[:, 2 * b.bus[k] + 1] = 0.0
    return A, c


def _limits(V, mix):
    if mix == "inside":
        return float(V.min()) - 10.0, float(V.max()) + 10.0
    if mix == "hopeless":
        return float(V.max()) + 50.0, float(V.max()) + 60.0
    lo, hi = float(np.quantile(V.min(1), 0.3)), float(np.quantile(V.max(1), 0.85))
    return lo, (hi if hi > lo else lo + 1e-3)


def _clear(lims, V0s):
    """Limits moved off every predicted voltage by more than any summation order can change it.  The batch repeats
    profile rows, so a quantile of the predictions can equal one of them exactly; a proposal at zero then puts V(y0) on
    the limit, where the kernel's and the restatement's roundings may classify it differently."""
    V = np.concatenate([np.ravel(v) for v in V0s])
    V = V[np.isfinite(V)]
    out = []
    for lim in lims:
        while V.size and np.abs(V - lim).min() <= 1e-9 * max(1.0, abs(lim)):
            lim += 3e-9 * max(1.0, abs(lim))
        out.append(lim)
    return tuple(out)


def _free_prediction(b, A, c):
    """The map's prediction at the current demands (no proposal applied), for placing the limits."""
    x = np.empty((len(b.P), 2 * b.env.n_bus)); x[:, 0::2] = b.P; x[:, 1::2] = b.Q
    return x @ A.T + c


# ------------------------------------------------------------------ the checks
def _setpoints(got, want, what):
    gn, wn = np.isnan(got), np.isnan(want)
    bad = np.argwhere(gn != wn)
    assert len(bad) == 0, f"{what}: NaN positions differ at (env, agent, value) {bad[:5].tolist()}: got {got[tuple(bad[0])]}, want {want[tuple(bad[0])]}"
    g, w = got[~gn].astype(np.float64), want[~wn]
    err = np.abs(g - w) / np.maximum(1.0, np.abs(w))
    assert err.size == 0 or err.max() < 1e-6, (what, float(err.max()), np.argwhere(~gn)[int(err.argmax())].tolist())


def _as_parsed(got, y0, rows, what):
    """Rows the layer left alone: the proposal cast to fp32, element for element (NaN positions included)."""
    g, w = got[rows], y0[rows].astype(np.float32)
    assert np.array_equal(np.isnan(g), np.isnan(w)), what
    assert np.array_equal(g[~np.isnan(g)], w[~np.isnan(w)]), (what, np.argwhere((g != w) & ~np.isnan(w))[:5].tolist())


def _slack(got, want, what):
    d = np.abs(got - want) > 1e-9 * np.maximum(1.0, np.abs(want))
    assert not d.any(), (what, np.argwhere(d)[:5].tolist(), got[d][:5], want[d][:5])


def _check_rowsum(b, res, ref, what):
    out, slack, moved = res
    y, wslack, lam = ref
    _setpoints(out, y, what)
    _as_parsed(out, b.y0_cur, ~(lam > 0), what + " (unprojected)")
    if slack is not None:
        _slack(slack, wslack, what + " slack")
    if moved is not None:
        bad = np.argwhere(moved.astype(bool) != (lam > 0))
        assert len(bad) == 0, (what + " intervened", bad[:5].tolist())


def _check_affine(b, res, ref, what):
    out, slack, moved, status = res
    y, wslack, wstatus, _ = ref
    _setpoints(out, y, what)
    _as_parsed(out, b.y0_cur, wstatus == 0, what + " (envs left as proposed)")
    if slack is not None:
        _slack(slack, wslack, what + " slack")
    if moved is not None:
        bad = np.argwhere(moved.astype(bool) != B.bits_moved(y, b.y0_cur))
        assert len(bad) == 0, (what + " intervened", bad[:5].tolist())
    if status is not None:
        assert (status >= 0).all(), (what, "iteration cap reached", np.flatnonzero(status < 0)[:5].tolist())
        bad = np.flatnonzero((status == 0) != (wstatus == 0))
        assert len(bad) == 0, (what + " status", bad[:5].tolist(), status[bad[:5]], wstatus[bad[:5]])


def _load_rowsum(b, kind, mix):
    env = b.env
    coef, icpt = _rowsum_model(b, kind)
    sP, sQ, sb = safety_ref.row_sums(coef, icpt)
    V = b.P[:, b.bus] * sP[b.bus] + b.Q[:, b.bus] * sQ[b.bus] + sb[b.bus]
    v_min, v_max = _limits(V, mix) if mix != "env" else (float(env.args_dict["v_min"]), float(env.args_dict["v_max"]))
    v_min, v_max = _clear((v_min, v_max), [B.rowsum_prediction(y0, b.P[:, b.bus], b.Q[:, b.bus], sP[b.bus], sQ[b.bus], sb[b.bus])
                                           for y0 in b.y0.values()])
    env._check(env._lib.fp_safety_load(env._h, coef.ctypes.data_as(C.c_void_p), icpt.ctypes.data_as(C.c_void_p), v_min, v_max,
                                       1000.0), "fp_safety_load")
    torch.cuda.synchronize()
    return lambda y0: B.project_rowsum(y0, b.P[:, b.bus], b.Q[:, b.bus], sP[b.bus], sQ[b.bus], sb[b.bus], v_min, v_max)


def _load_affine(b, name, mix):
    A, c = _affine_map(b, name)
    v_min, v_max = _clear(_limits(_free_prediction(b, A, c), mix),
                          [B.affine_prediction(y0, b.P, b.Q, b.bus, A, c)[0] for y0 in b.y0.values()])
    b.env.load_safety_map(A, c, v_min=v_min, v_max=v_max)
    torch.cuda.synchronize()
    return lambda y0, pool: B.project_affine(y0, b.P, b.Q, b.bus, A, c, v_min, v_max, pool=pool)


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("N", RS_SIZES)
def test_rowsum_every_row(cuda, profiles, stream, N):
    b = _batch(cuda, profiles, N)
    for kind, mix in (("reference_fit", "mixed"), ("lindistflow", "mixed"), ("reference_fit", "env")):
        ref_of = _load_rowsum(b, kind, mix)
        for dt in (torch.float32, torch.float64):
            b.y0_cur = b.y0[dt]
            ref = ref_of(b.y0_cur)
            for tm in (0, 1):
                res, _ = _rowsum(b.env, b.act[dt], tm, stream)
                _check_rowsum(b, res, ref, f"N={N} {kind}/{mix} {dt} type_major={tm}")
            if N >= 100000 and mix == "mixed":
                lam = ref[2]
                assert 0.02 < float((lam > 0).mean()) < 0.98, float((lam > 0).mean())
                assert np.isnan(b.y0_cur).any(-1).sum() > 1000
    if N >= 100000:                                             # the batch reaches every position
        steps = b.env.steps.cpu().numpy() - 1                   # steps since the last reset
        for s in (0, 1, 2, 95, 96, L_DRIVE):
            assert (steps == s).any(), s
        assert ((steps > 2) & (steps < 95)).any() and L_DRIVE > b.env.episode_limit + b.env.history + 1
        assert (b.PV == 0).any() and ((b.PV == 0) & np.isinf(b.act[torch.float64].cpu().numpy()[..., 3])).any()
        assert (b.E == float(b.env.args_dict["e_min"])).any() and (b.E == float(b.env.args_dict["e_max"])).any()
        assert ((b.env.flags.cpu().numpy()[b.role == 6] & 2) != 0).all(), "FP_FLAG_FAILED"


@pytest.mark.parametrize("N", AF_SIZES)
def test_affine_every_row(cuda, profiles, stream, pool, N):
    b = _batch(cuda, profiles, N)
    if N == 131072:                                             # the scalar restatement's cost bounds this size's matrix
        plan = [("reference_fit", "mixed", torch.float32), ("reference_fit", "mixed", torch.float64),
                ("lindistflow_zeroed", "inside", torch.float64)]
    else:
        plan = [(m, x, dt) for m in MAPS for x in LIMITS for dt in (torch.float32, torch.float64)]
    seen = set()
    for name, mix, dt in plan:
        ref_of = _load_affine(b, name, mix)
        b.y0_cur = b.y0[dt]
        ref = ref_of(b.y0_cur, pool)
        for tm in (0, 1):
            res, _ = _affine(b.env, b.act[dt], tm, stream)
            _check_affine(b, res, ref, f"N={N} {name}/{mix} {dt} type_major={tm}")
        st = ref[2]
        seen.update({"moved"} if (st > 0).any() else set())
        if N >= 2367 and mix == "mixed":
            assert 0.02 < float((st > 0).mean()) < 0.98, (name, float((st > 0).mean()))
        if mix == "hopeless":
            assert (ref[1].sum(1) > 0).sum() >= 0.9 * np.isfinite(b.y0_cur).all(axis=(1, 2)).sum()
    if N > 1:
        assert "moved" in seen


def test_optional_outputs_same_bits(cuda, profiles, stream):
    """Every subset of the optional outputs: the outputs that remain hold the same bits as with all of them."""
    b = _batch(cuda, profiles, 121242)
    _load_rowsum(b, "reference_fit", "mixed")
    a = b.act[torch.float64]
    full, _ = _rowsum(b.env, a, 1, stream)
    for sl, mv in itertools.product((True, False), repeat=2):
        res, _ = _rowsum(b.env, a, 1, stream, slack=sl, moved=mv)
        assert np.array_equal(res[0].view(np.int32), full[0].view(np.int32))
        for i, on in ((1, sl), (2, mv)):
            assert (res[i] is None) != on and (res[i] is None or np.array_equal(res[i].view(np.uint8), full[i].view(np.uint8)))
    b = _batch(cuda, profiles, 2369)
    _load_affine(b, "lindistflow", "mixed")
    a = b.act[torch.float32]
    full, _ = _affine(b.env, a, 0, stream)
    assert (full[3] > 0).any()
    for sl, mv, st in itertools.product((True, False), repeat=3):
        res, _ = _affine(b.env, a, 0, stream, slack=sl, moved=mv, status=st)
        assert np.array_equal(res[0].view(np.int32), full[0].view(np.int32))
        for i, on in ((1, sl), (2, mv), (3, st)):
            assert (res[i] is None) != on and (res[i] is None or np.array_equal(res[i].view(np.uint8), full[i].view(np.uint8)))


def test_nan_and_inf_at_night_stay_nan(cuda, profiles, stream, pool):
    """A NaN action component, a3 = +-inf where PV = 0 (numpy: -0 + inf * 0 = NaN), or charge and discharge both +inf
    (inf - inf) is NaN after parse_actions; both layers return it as parsed, unprojected, with no slack, no intervention
    and status 0."""
    b = _batch(cuda, profiles, 2369)
    a64 = b.act[torch.float64].cpu().numpy()
    # NaN after parse_actions: a NaN component; a3 = +-inf at PV = 0; charge and discharge both +inf, where
    # adjust_ess_actions takes dis - ch = inf - inf
    nan_rows = (np.isnan(a64).any(-1) | (np.isinf(a64[..., 3]) & (b.PV == 0))
                | ((a64[..., 1] == np.inf) & (a64[..., 2] == np.inf)))
    assert nan_rows.sum() > 200 and (np.isinf(a64[..., 3]) & (b.PV == 0)).sum() > 20
    for dt in (torch.float32, torch.float64):
        b.y0_cur = b.y0[dt]
        assert np.array_equal(np.isnan(b.y0_cur).any(-1), nan_rows)
        ref = _load_rowsum(b, "reference_fit", "mixed")(b.y0_cur)
        (out, slack, moved), _ = _rowsum(b.env, b.act[dt], 1, stream)
        _setpoints(out, ref[0], f"row-sum NaN proposals {dt}")
        assert not slack[nan_rows].any() and not moved[nan_rows].any()
        ref = _load_affine(b, "reference_fit", "hopeless")(b.y0_cur, pool)
        (out, slack, moved, status), _ = _affine(b.env, b.act[dt], 0, stream)
        _setpoints(out, ref[0], f"affine NaN proposals {dt}")
        nan_env = nan_rows.any(-1)
        assert not slack[nan_env].any() and not moved[nan_env].any() and not status[nan_env].any()
        assert (status[~nan_env] > 0).all()


@pytest.mark.parametrize("layer", ["rowsum", "affine"])
def test_locality_and_determinism(cuda, profiles, stream, pool, layer):
    """Two launches are bit-identical (guard bands included); NaN actions for one env change that env's outputs only."""
    N = 121242 if layer == "rowsum" else 2369
    b = _batch(cuda, profiles, N)
    na, nb = b.env.n_agents, b.env.n_bus
    call = _rowsum if layer == "rowsum" else _affine
    if layer == "rowsum":
        _load_rowsum(b, "reference_fit", "mixed")
    else:
        _load_affine(b, "lindistflow", "mixed")
    a = b.act[torch.float64].clone()
    _, r0 = call(b.env, a, 1, stream)
    _, r1 = call(b.env, a, 1, stream)
    for x, y in zip(r0, r1):
        assert torch.equal(x.buf.view(INT_OF[x.dtype]), y.buf.view(INT_OF[y.dtype]))
    for e in (0, N // 2 + 3, N - 1):
        p = a.clone(); p[e] = float("nan")
        res, rp = call(b.env, p, 1, stream)
        widths = [4 * na, nb if layer == "affine" else na, na, 1]
        for x, y, w in zip(r0, rp, widths):
            xb = x.view.view(INT_OF[x.dtype]).view(N, -1)
            yb = y.view.view(INT_OF[y.dtype]).view(N, -1)
            keep = torch.ones(N, dtype=torch.bool, device=cuda); keep[e] = False
            assert torch.equal(xb[keep], yb[keep]), (layer, e, "another env changed")
            assert torch.equal(x.buf[N * w:].view(INT_OF[x.dtype]), y.buf[N * w:].view(INT_OF[y.dtype]))
        assert np.isnan(res[0][e]).all() and not res[1][e].any() and not res[2][e].any()
        if layer == "affine":
            assert res[3][e] == 0


@pytest.mark.parametrize("name", FEEDERS)
def test_feeders_every_row(cuda, profiles, stream, pool, name):
    net = F.feeder(name)
    b = _batch(cuda, profiles, 20000, net=net, name=name)
    assert b.env.n_agents == {"two_bus": 1, "slack_star": 2, "custom14": 3, "ieee33_4agents": 4, "chain33": 5}[name]
    dt = torch.float64 if name in ("slack_star", "ieee33_4agents") else torch.float32
    b.y0_cur = b.y0[dt]
    ref = _load_rowsum(b, "lindistflow", "mixed")(b.y0_cur)
    for tm in (0, 1):
        res, _ = _rowsum(b.env, b.act[dt], tm, stream)
        _check_rowsum(b, res, ref, f"{name} row-sum {dt} type_major={tm}")
    assert (ref[2] > 0).any()
    ref = _load_affine(b, "lindistflow", "mixed")(b.y0_cur, pool)
    for tm in (0, 1):
        res, _ = _affine(b.env, b.act[dt], tm, stream)
        _check_affine(b, res, ref, f"{name} affine {dt} type_major={tm}")
    assert 0 < (ref[2] > 0).sum() < 20000
