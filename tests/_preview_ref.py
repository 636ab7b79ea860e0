"""The step preview's expected outputs from the C mirror, and a bit comparison that names where it fails.

mirror_preview() is what fp_step_preview computes for K candidate actions per env: the mirror steps its batch once per
candidate from the same state and is put back after each, so it is left as it was.  same() compares one candidate's
outputs at a time (no [K, N, 33] host array is built) and names the candidate, the env and the first differing element
of a mismatch.  Pinned on the mirror alone by tests/test_preview_ref.py.
"""
import numpy as np
import torch

from flexgpu._lib import INFO_KEYS
from oracle import c_mirror


def mirror_copy(mb):
    """Copies of every ndarray of a MirrorBatch: its state, its profiles and its last outputs."""
    return {k: v.copy() for k, v in vars(mb).items() if isinstance(v, np.ndarray)}


def mirror_restore(mb, saved):
    """Writes copies from mirror_copy back in place (the C state struct points at these very arrays)."""
    for k, v in saved.items():
        getattr(mb, k)[...] = v


def mirror_preview(mb, candidates, inject=None, translate=False):
    """For each candidate action array ([N, na, 4], numpy or torch) in `candidates`, yields the mirror's (reward [N] f64,
    done [N] bool, info [N, 8] f64, voltages [N, nb] f64, violation mask [N] u64) of one step from the batch's current
    state -- after a failed solve the rolled-back voltages and their mask, as the step leaves them.  translate: the
    candidates are raw fp32 policy outputs (FP_F32_POLICY).  inject is the env-indexed failure mask of every candidate.
    The batch is restored before each yield, so every candidate starts from the same state and the batch ends as it
    began, whenever the caller stops."""
    saved = mirror_copy(mb)
    for a in candidates:
        if isinstance(a, torch.Tensor):
            a = a.cpu().numpy()
        if translate:
            a = c_mirror.translate_action_f32(a)
        r, d, info = mb.step(a, inject=inject)
        out = (r.copy(), d.copy(), info.copy(), mb.V.copy(), mb.vmask.copy())
        mirror_restore(mb, saved)
        yield out


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
    """One candidate's preview outputs against one mirror_preview() tuple.  got: (reward [N], done [N], info: a dict of
    [N] columns by INFO_KEYS or an [N, 8] tensor, voltages [N, nb], mask [N]); the parts switched off are not compared."""
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
