"""The env kernels against the C mirror: the helpers every env-parity suite shares.

make_env() builds the env and reset_draws() the explicit reset's draws; reset_both() / step_both() drive the env and a
MirrorBatch together.  same() compares a device result with the mirror's bit for bit (NaN and -0.0 included) and names
`where`, the env and the first differing element of a mismatch; check_state() compares the whole env state that way,
field by field.  Pinned on the mirror alone by tests/test_preview_ref.py.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import _feeders as F
from flexgpu._lib import INFO_KEYS, REC_COUNTS, REC_CUM, REC_E_CUR, REC_E_INIT, REC_HIST, REC_LINES, REC_TIME, REC_VMASK
from oracle import c_mirror


@pytest.fixture(scope="module", autouse=True)
def all_cores():
    """The mirror's OpenMP loops on every core: the rollout-scale suites step 10^5 - 10^6 envs on it."""
    c_mirror.use_all_cores()


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


# ------------------------------------------------------------------ envs, profiles, draws and actions
def make_env(cuda, profiles, n, variant="thread", net=None, seed=None, env_offset=0, **args):
    """A BatchedFlexProvisionEnv of n envs: on feeder `net` with _feeders.env_args, else on the built-in IEEE 33-bus
    case with `args`; seed None is the env arguments' seed."""
    from flexgpu import BatchedFlexProvisionEnv
    a = F.env_args(net, variant, **args) if net is not None else {**args, "kernel_variant": variant}
    return BatchedFlexProvisionEnv(a, n_envs=n, device=cuda, network=net, profiles=profiles, seed=seed,
                                   env_offset=env_offset)


def feeder_profiles(net):
    """The synthetic profiles of a catalogue feeder."""
    from flexgpu.network import Network
    from flexgpu.profiles import synthetic_profiles
    return synthetic_profiles(Network(net), len(net['buildings']), T=1500, seed=3)


def scaled_profiles(p, every_other_day):
    """Demand (P and Q) x 2.4: on every row (voltage and line-limit violations throughout), or on every other day of 96
    rows (an episode then runs through a normal and a heavily loaded day)."""
    from flexgpu import Profiles
    f = np.where((np.arange(p.P.shape[0]) // 96) % 2 == 1, 2.4, 1.0)[:, None] if every_other_day else 2.4
    return Profiles(p.P * f, p.Q * f, p.PV, p.price)


def reset_draws(rng, n, na, max_start):
    """(start, e0, a0) of an explicit reset of n envs with na agents, drawn from rng in that order."""
    start = rng.integers(0, max_start, n).astype(np.int32)
    e0 = rng.uniform(0.9 * 0.0125, 1.1 * 0.0125, (n, na))
    a0 = rng.uniform(0, 1, (n, 4 * na))
    return start, e0, a0


def draws(seed, env):
    """reset_draws() for every env of `env` from default_rng(seed)."""
    return reset_draws(np.random.default_rng(seed), env.n_envs, env.n_agents, env.max_start())


def reset_both(env, mb, rng, mask=None):
    """An explicit reset of the env and the mirror from reset_draws(rng) (mask: the envs to reset); returns the draws."""
    start, e0, a0 = reset_draws(rng, env.n_envs, env.n_agents, env.max_start())
    env.reset(start, e0, a0, mask=mask, return_obs=False); mb.reset(start, e0, a0, mask=mask)
    return start, e0, a0


def actions(kind, rng, shape, mean):
    """Actions of one kind: fp32 / fp64 policy outputs N(mean, 0.6), raw fp32 outputs to translate ("policy"), or
    setpoints of a raw-action env ("raw").  A numpy Generator gives a numpy array, a torch Generator a tensor on its
    device."""
    scale = [0.5, 0.01, 0.01, 0.02]
    if isinstance(rng, torch.Generator):
        if kind == "raw":
            return torch.rand(shape, dtype=torch.float64, device=rng.device, generator=rng) * \
                torch.tensor(scale, dtype=torch.float64, device=rng.device)
        dtype = torch.float64 if kind == "f64" else torch.float32
        return torch.randn(shape, dtype=dtype, device=rng.device, generator=rng) * 0.6 + mean
    if kind == "raw":
        return rng.uniform(0, 1, shape) * np.array(scale)
    return rng.normal(mean, 0.6, shape).astype(np.float64 if kind == "f64" else np.float32)


def mirror_actions(kind, a):
    """What the mirror steps with for actions `a` (numpy or torch) of `kind`: "policy" outputs translated in fp32."""
    if isinstance(a, torch.Tensor):
        a = a.cpu().numpy()
    return c_mirror.translate_action_f32(a) if kind == "policy" else a


def step_both(env, mb, a, where, translate=False, inject=None):
    """One committed step of the env and the mirror; reward, done and info compared."""
    r, d, info = env.step(a, translate=translate)
    rr, dd, ii = mb.step(mirror_actions("policy" if translate else None, a), inject=inject)
    same(r, rr, "reward", where); same(d, dd, "done", where)
    same(env._info, ii, "info", where)
    return r, d, info


# ------------------------------------------------------------------ bit comparisons
def bits(t):
    """A tensor whose equality is equality of bits: floats as integers of their width, bool as uint8."""
    t = t.contiguous()
    if t.dtype == torch.float64:
        return t.view(torch.int64)
    if t.dtype == torch.float32:
        return t.view(torch.int32)
    if t.dtype == torch.bool:
        return t.view(torch.uint8)
    return t


def _tensor(x):
    if isinstance(x, torch.Tensor):
        return x
    x = np.ascontiguousarray(x)
    if x.dtype == np.uint64:                                       # torch keeps violation masks as int64
        x = x.view(np.int64)
    return torch.from_numpy(x)


def same(got, want, what, where):
    """got == want bit for bit (NaN and -0.0 included).  Both are indexed by env first ([N, ...]); a mismatch raises an
    AssertionError naming `where` (the leg and the candidate), `what`, the env and the first differing element."""
    want = _tensor(want).to(got.device)
    if want.dtype == torch.int64 and got.dtype == torch.uint64:
        got = got.view(torch.int64)
    assert got.shape == want.shape and got.dtype == want.dtype, \
        f"{where}: {what}: {tuple(got.shape)} {got.dtype} vs {tuple(want.shape)} {want.dtype}"
    d = bits(got) != bits(want)
    if bool(d.any()):
        i = tuple(int(x) for x in torch.nonzero(d)[0])
        raise AssertionError(f"{where}: {what} differs at env {i[0]}, element {i} ({int(d.sum())} elements differ): "
                             f"{got[i].item()!r} vs {want[i].item()!r}")


def same_outputs(got, want, where, info=True, voltage=True, mask=True):
    """One step's outputs against the mirror's (reward [N], done [N], info [N, 8], voltages [N, nb], violation mask [N]).
    got: the same, its info a dict of [N] columns by INFO_KEYS or an [N, 8] tensor; the parts switched off are not
    compared."""
    r, d, inf, V, vm = got
    wr, wd, wi, wV, wm = want
    same(r, wr, "reward", where)
    same(d, wd, "done", where)
    if info:
        for i, key in enumerate(INFO_KEYS):
            same(inf[key] if isinstance(inf, dict) else inf[:, i], wi[:, i], f"info[{key}]", where)
    if voltage:
        same(V, wV, "voltages", where)
    if mask:
        same(vm, wm, "violation mask", where)


def check_state(env, mb, where, pushes=None):
    """The env's record, voltages and setpoints against the mirror's, bit for bit, each field on its own: the record words
    the mirror keeps for its agent count (E_init and E_cur of na agents, the cumulative reward, start, steps, the episode
    counter, the violation mask and count, the flags, the line-limit mask and the power-flow passes) and, when `pushes`
    (every env's push count since its last reset) is given, the push-count half of REC_HIST."""
    rec, na = env.rec, mb.E_init.shape[1]
    half = rec.view(torch.int32)                    # [N, 32]: the low 32 bits of word w at 2 w, the high ones at 2 w + 1
    fields = [("E_init", rec[:, REC_E_INIT:REC_E_INIT + na].view(torch.float64), mb.E_init),
              ("E_cur", rec[:, REC_E_CUR:REC_E_CUR + na].view(torch.float64), mb.E_cur),
              ("cumulative reward", rec[:, REC_CUM].view(torch.float64), mb.cum),
              ("start", half[:, 2 * REC_TIME], mb.start), ("steps", half[:, 2 * REC_TIME + 1], mb.steps),
              ("episode", half[:, 2 * REC_HIST + 1], mb.episode),
              ("violation mask", rec[:, REC_VMASK], mb.vmask),
              ("violation count", half[:, 2 * REC_COUNTS], mb.vcount), ("flags", half[:, 2 * REC_COUNTS + 1], mb.flags),
              ("line-limit mask", half[:, 2 * REC_LINES], mb.lmask.view(np.int32)),
              ("power-flow passes", half[:, 2 * REC_LINES + 1], mb.iters),
              ("voltages", env.voltages, mb.V), ("setpoints", env.setpoints, mb.setp)]
    if pushes is not None:
        fields.append(("push count", half[:, 2 * REC_HIST], torch.as_tensor(pushes).to(torch.int32)))
    for what, got, want in fields:
        same(got, want, what, where)
