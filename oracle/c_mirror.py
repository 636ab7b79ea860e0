"""ctypes wrapper of oracle/c/flex_oracle.c -- the bit-exact CPU mirror (TEST INFRASTRUCTURE).

PARITY: see oracle/__init__.py (pinned on the reference's Python code, IPOPT excepted).  `MirrorBatch` holds N environments as plain numpy
arrays and advances them with the C restatement of reset/step; `mirror_power_flow` is the
batched power flow.  Used by the GPU parity tests (bit-exact masks, ulp-level floats) and as
bench.py's CPU baseline.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from math import acos, tan

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "_build", "libflex_oracle.so")
NL = 32


def build(force=False):
    """Compiles the mirror into oracle/_build/ if it is missing or older than its source.  A tree that cannot be
    written (a read-only checkout) gets it compiled into a temporary directory instead, removed at exit."""
    global LIB
    src = os.path.join(_HERE, "c", "flex_oracle.c")
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        out_dir = os.path.dirname(LIB)
        if not os.access(out_dir if os.path.isdir(out_dir) else _HERE, os.W_OK):
            out_dir = tempfile.mkdtemp(prefix="flex_oracle_")
            atexit.register(shutil.rmtree, out_dir, True)
        out = os.path.join(out_dir, "libflex_oracle.so")
        subprocess.run(["make", "-C", os.path.join(_HERE, "c"), f"OUT={out}"], check=True, capture_output=True)
        LIB = out
    return LIB


class FoNet(C.Structure):
    _fields_ = [
        ("nb", C.c_int32), ("nl", C.c_int32), ("na", C.c_int32), ("history", C.c_int32),
        ("episode_limit", C.c_int32), ("raw_actions", C.c_int32), ("pf_max_iter", C.c_int32), ("variant", C.c_int32),
        ("pf_f32", C.c_int32), ("pad_", C.c_int32),
        ("pf_tol", C.c_double), ("v_min", C.c_double), ("v_max", C.c_double), ("e_min", C.c_double),
        ("e_max", C.c_double), ("p_ch_max", C.c_double), ("p_dis_max", C.c_double), ("eta_ch", C.c_double),
        ("eta_dis", C.c_double), ("mpr", C.c_double), ("kappa", C.c_double), ("pv_cost", C.c_double),
        ("ess_cost", C.c_double), ("discomfort_coeff", C.c_double), ("voltage_coeff", C.c_double),
        ("delta_t", C.c_double), ("fail_penalty", C.c_double), ("e_next_lb", C.c_double),
        ("R", C.c_double * NL), ("X", C.c_double * NL), ("Z2", C.c_double * NL), ("imax2", C.c_double * NL),
        ("end", C.c_int32 * NL), ("col", C.c_int32 * NL), ("agent", C.c_int32 * NL), ("anc", (C.c_int32 * NL) * 5),
        ("agent_lane", C.c_int32 * 8), ("agent_col", C.c_int32 * 8), ("par", C.c_int32 * NL),
    ]


class FoState(C.Structure):
    _fields_ = [
        ("n", C.c_int64), ("E_init", C.c_void_p), ("E_cur", C.c_void_p), ("cum", C.c_void_p),
        ("start", C.c_void_p), ("steps", C.c_void_p), ("episode", C.c_void_p), ("hist_n", C.c_void_p),
        ("V", C.c_void_p), ("setp", C.c_void_p), ("vmask", C.c_void_p), ("vcount", C.c_void_p),
        ("flags", C.c_void_p), ("iters", C.c_void_p), ("lmask", C.c_void_p),
        ("pfl", C.c_void_p), ("qfl", C.c_void_p), ("isq", C.c_void_p),
    ]


DEFAULT_TOL = {0: 1e-5, 1: 1e-9}     # must match flexgpu.config (pf_tol per kernel variant)
DEFAULT_F32_PASSES = {0: 5, 1: 0}    # must match flexgpu.config.DEFAULT_PF_F32_PASSES
_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        l = C.CDLL(LIB)
        assert l.fo_sizeof_net() == C.sizeof(FoNet), "FoNet layout mismatch"
        assert l.fo_sizeof_state() == C.sizeof(FoState), "FoState layout mismatch"
        _lib = l
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def use_all_cores():
    """Give the OpenMP loops every core this process may run on (torchrun exports OMP_NUM_THREADS=1);
    returns the number of worker threads in force."""
    l = lib()
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    l.fo_set_threads(C.c_int(n))
    return int(l.fo_threads())


VARIANT_THREAD, VARIANT_WARP = 0, 1


def translate_action_f32(x, low=0.0, high=1.0):
    """numpy fp32 restatement of translate_action's continuous branch (utils/util.py:124-128), in
    torch's operation order: clamp, + 1, * 0.5, * (high - low), + low, every step rounded to fp32.
    Pinned on the reference's own function by tests/golden/ref_translate_action.npz."""
    f = np.float32
    x = np.asarray(x, dtype=f)
    c = np.where(x < f(low), f(low), np.where(x > f(high), f(high), x)).astype(f)
    t = (c + f(1.0)).astype(f)
    t = (f(0.5) * t).astype(f)
    t = (t * f(high - low)).astype(f)
    return (t + f(low)).astype(f)


def make_net(tree, args, agent_buses, pf_tol=None, pf_max_iter=32, raw_actions=False,
             fail_penalty=200.0, e_next_lb=-1e-8, variant=VARIANT_THREAD, pf_f32_passes=None):
    """tree: oracle.ieee33.tree_arrays(net); args: dict with the reference's yaml keys.
    variant selects which kernel's floating-point operation order is mirrored (the thread-per-env
    kernel converges on max |dl| <= pf_tol, the warp-per-env kernel on max |dv| <= pf_tol)."""
    if pf_tol is None:
        pf_tol = DEFAULT_TOL[variant]
    l = lib()
    net = FoNet()
    nb = len(tree['parent'])
    parent = np.ascontiguousarray(tree['parent'], dtype=np.int32)
    r = np.ascontiguousarray(tree['R'], dtype=np.float64)
    x = np.ascontiguousarray(tree['X'], dtype=np.float64)
    imax = np.ascontiguousarray(tree['imax'], dtype=np.float64)
    ab = np.ascontiguousarray([tree['pos'][b] for b in agent_buses], dtype=np.int32)
    rc = l.fo_build(C.byref(net), nb, len(agent_buses), _p(parent), _p(r), _p(x), _p(imax), _p(ab))
    if rc != 0:
        raise ValueError(f"fo_build failed: {rc}")
    net.history = args['history']; net.episode_limit = args['episode_limit']
    net.raw_actions = 1 if raw_actions else 0
    net.variant = variant
    net.pf_max_iter = pf_max_iter; net.pf_tol = pf_tol
    net.pf_f32 = DEFAULT_F32_PASSES[variant] if pf_f32_passes is None else int(pf_f32_passes)
    net.v_min, net.v_max = args['v_min'], args['v_max']
    net.e_min, net.e_max = args['e_min'], args['e_max']
    net.p_ch_max, net.p_dis_max = args['p_ch_max'], args['p_dis_max']
    net.eta_ch, net.eta_dis = args['eta_ch'], args['eta_dis']
    net.mpr = args['max_power_reduction']
    net.kappa = tan(acos(args['cos_phi_max']))
    net.pv_cost, net.ess_cost = args['pv_cost'], args['ess_cost']
    net.discomfort_coeff, net.voltage_coeff = args['discomfort_coeff'], args['voltage_coeff']
    net.delta_t = 24 / args['episode_limit']
    net.fail_penalty = fail_penalty; net.e_next_lb = e_next_lb
    return net


def mirror_power_flow(net, p, q, want_flows=True):
    l = lib()
    p = np.ascontiguousarray(p, dtype=np.float64)
    q = np.ascontiguousarray(q, dtype=np.float64)
    n = p.shape[0]
    V = np.empty((n, net.nb))
    Pl = np.empty((n, net.nl)) if want_flows else None
    Ql = np.empty((n, net.nl)) if want_flows else None
    Isq = np.empty((n, net.nl)) if want_flows else None
    iters = np.empty(n, dtype=np.int32)
    fail = np.empty(n, dtype=np.uint8)
    l.fo_power_flow(C.byref(net), C.c_double(net.pf_tol), C.c_int(net.pf_max_iter), C.c_int64(n), _p(p), _p(q),
                    _p(V), _p(Pl), _p(Ql), _p(Isq), _p(iters), _p(fail))
    return dict(V=V, P=Pl, Q=Ql, Isq=Isq, iters=iters, failed=fail.astype(bool))


class MirrorBatch:
    """N environments advanced by the C mirror.  profiles: dict(P, Q, PV, price) fp64 arrays."""

    def __init__(self, net, profiles, n, keep_flows=False):
        self.net, self.n = net, n
        na, nb, nl = net.na, net.nb, net.nl
        self.P = np.ascontiguousarray(profiles['P'], dtype=np.float64)
        self.Q = np.ascontiguousarray(profiles['Q'], dtype=np.float64)
        self.PV = np.ascontiguousarray(profiles['PV'], dtype=np.float64)
        self.price = np.ascontiguousarray(profiles['price'], dtype=np.float64).reshape(-1)
        self.E_init = np.zeros((n, na)); self.E_cur = np.zeros((n, na)); self.cum = np.zeros(n)
        self.start = np.zeros(n, dtype=np.int32); self.steps = np.zeros(n, dtype=np.int32)
        self.episode = np.zeros(n, dtype=np.int32); self.hist_n = np.zeros(n, dtype=np.int32)
        self.V = np.zeros((n, nb)); self.setp = np.zeros((n, 4, na))
        self.vmask = np.zeros(n, dtype=np.uint64); self.vcount = np.zeros(n, dtype=np.int32)
        self.flags = np.zeros(n, dtype=np.int32); self.iters = np.zeros(n, dtype=np.int32)
        self.lmask = np.zeros(n, dtype=np.uint32)
        self.pfl = np.zeros((n, nl)) if keep_flows else None
        self.qfl = np.zeros((n, nl)) if keep_flows else None
        self.isq = np.zeros((n, nl)) if keep_flows else None
        self.reward = np.zeros(n); self.done = np.zeros(n, dtype=np.uint8); self.info = np.zeros((n, 8))
        self.st = FoState(n, *[_p(a) for a in (
            self.E_init, self.E_cur, self.cum, self.start, self.steps, self.episode, self.hist_n, self.V,
            self.setp, self.vmask, self.vcount, self.flags, self.iters, self.lmask, self.pfl, self.qfl, self.isq)])
        T = self.P.shape[0]
        self.start_range = T - (net.episode_limit + net.history + 1) + 1

    def _prof(self):
        return _p(self.P), _p(self.Q), _p(self.PV), _p(self.price)

    def reset(self, start, e0, a0, mask=None):
        start = np.ascontiguousarray(start, dtype=np.int32)
        e0 = np.ascontiguousarray(e0, dtype=np.float64)
        a0 = np.ascontiguousarray(a0, dtype=np.float64)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        lib().fo_env_reset(C.byref(self.net), *self._prof(), C.byref(self.st), _p(start), _p(e0), _p(a0), _p(m))

    def reset_random(self, seed, env_offset=0, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        lib().fo_env_reset_random(C.byref(self.net), *self._prof(), C.byref(self.st), C.c_uint64(seed),
                                  C.c_int64(env_offset), C.c_int32(self.start_range), _p(m))

    def step(self, actions, inject=None, mask=None):
        """actions: fp32 or fp64; fp32 is widened exactly (quirk Q6)."""
        a = np.ascontiguousarray(np.asarray(actions).reshape(self.n, -1), dtype=np.float64)
        inj = None if inject is None else np.ascontiguousarray(inject, dtype=np.uint8)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        lib().fo_env_step(C.byref(self.net), *self._prof(), C.byref(self.st), _p(a), _p(inj), _p(m),
                          _p(self.reward), _p(self.done), _p(self.info))
        return self.reward, self.done.astype(bool), self.info

    # numpy restatement of get_state / get_obs for the batch (flexibility_provision_env.py:358-403)
    def row(self):
        """The profile row in force, clamped to the last row of the episode slice as the kernels clamp it."""
        max_off = self.net.episode_limit + self.net.history
        return self.start.astype(np.int64) + np.where(self.steps > 1, np.minimum(self.steps - 1, max_off), 1)

    def get_state(self):
        r = self.row()
        n = self.n
        z = np.zeros((n, 1))
        return np.hstack([z, self.P[r], z, self.Q[r], self.PV[r], self.V, self.price[r][:, None], self.E_cur])

    def current_obs(self):
        r = self.row()
        cols = np.array(self.net.agent_col[:self.net.na])
        out = np.empty((self.n, self.net.na, 6))
        out[:, :, 0] = self.P[r][:, cols]
        out[:, :, 1] = self.Q[r][:, cols]
        out[:, :, 2] = self.PV[r]
        out[:, :, 3] = self.V[:, cols + 1]
        out[:, :, 4] = self.price[r][:, None]
        out[:, :, 5] = self.E_cur
        return out


def draw_random(net, seed, gid, episode, start_range):
    st = C.c_int32()
    e0 = np.zeros(8)
    a0 = np.zeros(32)
    lib().fo_random_draw(C.byref(net), C.c_uint64(seed), C.c_int64(gid), C.c_int32(episode), C.c_int32(start_range),
                         C.byref(st), _p(e0), _p(a0))
    return st.value, e0[:net.na].copy(), a0[:4 * net.na].copy()
