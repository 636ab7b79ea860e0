"""The step preview's expected outputs from the C mirror.

mirror_preview() is what fp_step_preview computes for K candidate actions per env: the mirror steps its batch once per
candidate from the same state and is put back after each, so it is left as it was.  It yields one candidate's outputs
at a time (no [K, N, 33] host array is built), for _env_check.same_outputs() to compare.  Pinned on the mirror alone by
tests/test_preview_ref.py.
"""
import numpy as np
import torch

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
