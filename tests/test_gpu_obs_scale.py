"""GPU: the observation history, the state and the records at rollout scale, every env bit-exact against the C mirror.

The other observation tests run 64 to 1 317 envs, where no kernel loops.  Here N = 131 072 + 19 (4 097 tiles: 3-4 tiles
per warp of the 1 184-CTA step grid, ~14 envs per warp of the 9 472-warp observation grid, 13 pad columns of the
env-minor ring) unless a leg says otherwise.  The expected observation history comes from tests/_obs_ref.py: the mirror's
current_obs() pushed into a test-owned fp64 history on the device.  Observations and states are copies of mirror values
(fp64, or the fp64 value rounded once to fp32), so every comparison is of bits.  A mismatch names the leg, the step and
the first differing element.

  A  fused step + env-minor ring (k_env_t<MODE_STEP, Ieee33, A64, OBS=true>: next-tile row prefetch, push after the
     bulk-store fence, ragged last tile), k_obsr_reset_push on a changing subset, k_obsr_gather's multi-trip tile,
     k_obs_push / k_state's next-env prefetch, the fp64 history ring and the push count
  B  ring-only stepping (DeviceRollout's configuration) and k_hist_from_ring at scale
  C  the window ring (fp_step_obs: k_obs_push, k_obsm_clear, k_obsm_compact twice, rebuild) for both variants; the
     warp variant alternates with return_obs="ring" (its step, push and ring rebuild) -- the warp step beyond 2 048 envs
  D  2^20 + 77 envs: second trips of k_obsr_reset_push / k_obsr_clear / k_obsr_gather, window-ring offsets past 2^31
  F  the row clamp past the end of an episode slice on a NaN-poisoned table, both variants
"""
import time

import numpy as np
import pytest
import torch

from _env_check import actions, check_state, make_env, mirror_actions, reset_draws, same
from _env_check import all_cores  # noqa: F401  (autouse fixture)
from _obs_ref import ObsRef, clamp_tables
from oracle import c_mirror

pytestmark = pytest.mark.gpu
N = 131072 + 19
H, NA = 24, 5
SENT = -7.25e6


def check_outputs(env, r, d, rr, dd, ii, where, info=True, mask=None):
    """reward, done and info of the stepped envs (mask: None = all)."""
    sel = np.ones(len(rr), dtype=bool) if mask is None else mask.astype(bool)
    dsel = torch.from_numpy(sel).to(r.device)
    same(r[dsel], torch.from_numpy(rr[sel]), "reward", where)
    same(d[dsel], torch.from_numpy(dd[sel]), "done", where)
    if info:
        same(env._info[dsel], torch.from_numpy(ii[sel]), "info", where)


def check_ring(ring, ref, slot, where):
    assert ring.slot == slot, f"{where}: ring slot {ring.slot}, expected {slot}"
    n = ref.n
    for lo, hi in ref.chunks():
        same(ring.ring[..., lo:hi], ref.ring(slot, lo, hi), "env-minor ring", f"{where} envs {lo}..")
    same(ring.ring[..., n:], torch.zeros_like(ring.ring[..., n:]), "ring pad columns", where)


def check_history(env, ref, where):
    hist = env._history(False)
    for lo, hi in ref.chunks():
        want, live = ref.history(lo, hi)
        same(torch.where(live, hist[lo:hi], 0.0), torch.where(live, want, 0.0), "fp64 history ring (live entries)",
             f"{where} envs {lo}..")


def check_windows(get, ref, where, cur=None, dtype=torch.float32):
    """get(lo, hi) -> the device's windows of envs lo .. hi-1."""
    for lo, hi in ref.chunks():
        same(get(lo, hi), ref.window(lo, hi, cur).to(dtype), "window", f"{where} envs {lo}..")


def check_reads(env, mb, ref, where, ring=None):
    """get_obs(push=False) and get_state() in fp32 and fp64; the gather of the env-minor ring into a sentinel-filled
    buffer with a guard band after it."""
    cur = torch.from_numpy(mb.current_obs())
    for dt in (torch.float32, torch.float64):
        o = env.get_obs(push=False, dtype=dt)
        check_windows(lambda lo, hi: o[lo:hi], ref, f"{where} get_obs(push=False, {dt})", cur, dt)
        same(env.get_state(dt), torch.from_numpy(mb.get_state()).to(dt), f"get_state({dt})", where)
    if ring is not None:
        n, per = env.n_envs, NA * 6 * H
        buf = torch.full((n * per + 4096,), SENT, dtype=torch.float32, device=env.device)
        out = ring.dense(out=buf[:n * per].view(n, NA, 6 * H))
        check_windows(lambda lo, hi: out[lo:hi], ref, f"{where} ObsRing.dense")
        same(buf[n * per:], torch.full((4096,), SENT, dtype=torch.float32), "guard band after dense()", where)


class Slot:
    """The env-minor ring's slot: H - 1 after a rebuild from the fp64 history (a generic push invalidates the ring), + 1
    per fused push."""

    def __init__(self):
        self.q, self.valid = H - 1, True

    def generic_push(self):
        self.valid = False

    def ring_op(self, push):
        if not self.valid:
            self.q, self.valid = H - 1, True
        if push:
            self.q = (self.q + 1) % H
        return self.q


def act_for(t, g, n):
    """Actions cycling through fp32, fp64 (the fp32 draw widened) and raw fp32 policy outputs (translate=True); what the
    mirror steps with."""
    raw = actions("f32", g, (n, NA, 4), 0.3)
    kind = ("f32", "f64", "policy")[t % 3]
    a = raw.double() if kind == "f64" else raw
    return a, {"translate": kind == "policy"}, mirror_actions(kind, a)


def test_a_fused_ring_step_default_mode(cuda, profiles, fonets):
    """Leg A: ~100 fused ring steps, reset-done-each-step (masked Philox reset + k_obsr_reset_push), one step with injected
    failures, one masked (unfused) step, one generic fp64 push; records, rewards, info, V, setpoints, the whole ring and
    the fp64 history every step, the dense gather, get_obs and get_state every few steps."""
    t0 = time.time()
    env = make_env(cuda, profiles, N, seed=21)
    mb = c_mirror.MirrorBatch(fonets["thread"], profiles.as_dict(), N)
    ref = ObsRef(N, NA, H, cuda)
    slot = Slot()
    ring = env.reset(return_obs="ring", retries=0); mb.reset_random(21)
    ref.push(mb.current_obs()); check_ring(ring, ref, slot.ring_op(False), "A reset")
    g = torch.Generator(device=cuda).manual_seed(5)
    rng = np.random.default_rng(6)
    for t in range(100):
        where = f"A step {t}"
        a, kw, am = act_for(t, g, N)
        want_info = t % 4 != 1
        inj = mask = None
        if t == 37:
            inj = np.zeros(N, dtype=np.uint8); inj[rng.integers(0, N, 300)] = 1
            env.inject_failure(inj)
        if t == 53:
            mask = (rng.uniform(size=N) < 0.7).astype(np.uint8)
        r, d, _, ring = env.step(a, mask=mask, want_info=want_info, return_obs="ring", **kw)
        rr, dd, ii = mb.step(am, inject=inj, mask=mask)
        if inj is not None:
            env.inject_failure(None)
        if mask is not None:                       # unfused: generic push of every env, then a ring rebuild
            slot.generic_push()
        ref.push(mb.current_obs())
        check_outputs(env, r, d, rr, dd, ii, where, info=want_info, mask=mask)
        check_state(env, mb, where, pushes=ref.cnt)
        check_ring(ring, ref, slot.ring_op(True) if mask is None else slot.ring_op(False), where)
        check_history(env, ref, where)
        if t == 37:
            assert int(dd[inj.astype(bool)].sum()) >= 290
        if t == 70:                                # a generic pushing fp64 get_obs detour: the next ring step rebuilds
            o = env.get_obs(dtype=torch.float64)
            ref.push(mb.current_obs()); slot.generic_push()
            check_windows(lambda lo, hi: o[lo:hi], ref, f"{where} get_obs(float64)", dtype=torch.float64)
        if t % 9 == 4:
            check_reads(env, mb, ref, where, ring)
        done = (mb.flags & 1).astype(np.uint8)
        if done.any():                             # DeviceRollout(reset_done_each_step=True)
            ring = env.reset(mask=done, return_obs="ring", retries=0); mb.reset_random(21, mask=done)
            ref.reset(done); ref.push(mb.current_obs(), done)
            check_ring(ring, ref, slot.ring_op(False), where + " reset")
    check_state(env, mb, "A end", pushes=ref.cnt)
    check_reads(env, mb, ref, "A end", env.obs_ring())
    env.close()
    print(f"leg A: {time.time() - t0:.1f} s")


def test_b_ring_only_stepping(cuda, profiles, fonets):
    """Leg B: set_obs_history(False), translate=True, reset-done-each-step -- the fused step pushes the ring alone; three
    fp64 reads restore the history from the ring (k_hist_from_ring): history entries are the mirror values rounded to
    fp32 and widened, the newest entry exact fp64; then back to the default mode with a generic push."""
    t0 = time.time()
    env = make_env(cuda, profiles, N, seed=31)
    mb = c_mirror.MirrorBatch(fonets["thread"], profiles.as_dict(), N)
    ref = ObsRef(N, NA, H, cuda)
    slot = Slot()
    ring = env.reset(return_obs="ring", retries=0); mb.reset_random(31)
    ref.push(mb.current_obs()); slot.ring_op(False)
    env.set_obs_history(False)
    g = torch.Generator(device=cuda).manual_seed(7)
    for t in range(60):
        where = f"B step {t}"
        raw = actions("f32", g, (N, NA, 4), 0.3)
        r, d, _, ring = env.step(raw, translate=True, return_obs="ring")
        rr, dd, ii = mb.step(mirror_actions("policy", raw))
        ref.push(mb.current_obs())
        check_outputs(env, r, d, rr, dd, ii, where)
        check_ring(ring, ref, slot.ring_op(True), where)
        if t in (9, 30, 51):                       # an fp64 read: the history is restored from the ring
            cur = torch.from_numpy(mb.current_obs())
            o = env.get_obs(push=False, dtype=torch.float64)
            ref.round_f32()
            check_windows(lambda lo, hi: o[lo:hi], ref, f"{where} restored get_obs(push=False, float64)", cur, torch.float64)
            check_history(env, ref, where + " restored")
            check_state(env, mb, where, pushes=ref.cnt)
        done = (mb.flags & 1).astype(np.uint8)
        if done.any():
            ring = env.reset(mask=done, return_obs="ring", retries=0); mb.reset_random(31, mask=done)
            ref.reset(done); ref.push(mb.current_obs(), done)
            check_ring(ring, ref, slot.ring_op(False), where + " reset")
    env.set_obs_history(True)
    o = env.get_obs(dtype=torch.float64)           # restore, then a generic push in fp64
    ref.round_f32(); ref.push(mb.current_obs())
    check_windows(lambda lo, hi: o[lo:hi], ref, "B generic push", dtype=torch.float64)
    check_history(env, ref, "B end"); check_state(env, mb, "B end", pushes=ref.cnt)
    env.close()
    print(f"leg B: {time.time() - t0:.1f} s")


@pytest.mark.parametrize("variant", ["thread", "warp"])
def test_c_window_ring(cuda, profiles, fonets, variant):
    """Leg C: 104 steps through the window ring (step(..., return_obs=True)), so that k_obsm_compact runs twice; masked
    Philox resets of the done envs and a random tenth every 4 steps (k_obsm_clear); one generic push (rebuild).  The
    returned strided view and its strides against the reference every step.  The warp variant alternates with
    return_obs="ring" (step, window-ring push, env-minor ring rebuild), which pushes the window ring as well."""
    t0 = time.time()
    env = make_env(cuda, profiles, N, variant, seed=41)
    mb = c_mirror.MirrorBatch(fonets[variant], profiles.as_dict(), N)
    ref = ObsRef(N, NA, H, cuda)
    env.reset(return_obs=False, retries=0); mb.reset_random(41)
    g = torch.Generator(device=cuda).manual_seed(8)
    rng = np.random.default_rng(9)
    for t in range(104):
        where = f"C[{variant}] step {t}"
        a, kw, am = act_for(t, g, N)
        as_ring = variant == "warp" and t % 2 == 1
        r, d, _, o = env.step(a, return_obs="ring" if as_ring else True, **kw)
        rr, dd, ii = mb.step(am)
        ref.push(mb.current_obs())
        check_outputs(env, r, d, rr, dd, ii, where)
        if as_ring:
            check_ring(o, ref, H - 1, where)       # rebuilt from the fp64 history after the window-ring push
        else:
            assert o.stride() == (NA * 3 * H * 6, 3 * H * 6, 1) and o.shape == (N, NA, 6 * H), where
            check_windows(lambda lo, hi: o[lo:hi], ref, where)
        if t % 10 == 3:
            check_state(env, mb, where, pushes=ref.cnt)
        if t == 100:                               # generic push (after the second compaction): rebuilt at the next step
            env.get_obs(dtype=torch.float64); ref.push(mb.current_obs())
        if t % 4 == 2:
            m = ((mb.flags & 1) | (rng.uniform(size=N) < 0.1)).astype(np.uint8)
            env.reset(mask=m, return_obs=False, retries=0); mb.reset_random(41, mask=m); ref.reset(m)
    check_state(env, mb, f"C[{variant}] end", pushes=ref.cnt); check_history(env, ref, f"C[{variant}] end")
    env.close()
    print(f"leg C[{variant}]: {time.time() - t0:.1f} s")


def test_d_two_pow_20_envs(cuda, profiles, fonets):
    """Leg D: 2^20 + 77 envs, 30 steps: fused ring with reset-done-each-step and one masked reset of about half the batch
    (second grid-stride trips of k_obsr_reset_push and k_obsr_clear), the dense gather (multi-trip k_obsr_gather),
    get_state / get_obs(push=False) in fp32 and fp64, a ring-only stretch with one restore, and 6 pushes through the
    window ring, whose element offsets pass 2^31."""
    t0 = time.time()
    n = 2 ** 20 + 77
    env = make_env(cuda, profiles, n, seed=51)
    mb = c_mirror.MirrorBatch(fonets["thread"], profiles.as_dict(), n)
    ref = ObsRef(n, NA, H, cuda)
    slot = Slot()
    ring = env.reset(return_obs="ring", retries=0); mb.reset_random(51)
    ref.push(mb.current_obs()); slot.ring_op(False)
    g = torch.Generator(device=cuda).manual_seed(10)
    rng = np.random.default_rng(11)
    for t in range(30):
        where = f"D step {t}"
        a, kw, am = act_for(t, g, n)
        if t == 12:
            env.set_obs_history(False)
        if t < 24:
            r, d, _, ring = env.step(a, return_obs="ring", **kw)
        else:                                      # the window ring: fp_step_obs
            r, d, _, o = env.step(a, return_obs=True, **kw)
            slot.generic_push()
        rr, dd, ii = mb.step(am)
        ref.push(mb.current_obs())
        check_outputs(env, r, d, rr, dd, ii, where)
        if t < 24:
            check_ring(ring, ref, slot.ring_op(True), where)
        else:
            check_windows(lambda lo, hi: o[lo:hi], ref, where)
        if t == 18:                                # ring-only since step 12: restore through an fp64 read
            cur = torch.from_numpy(mb.current_obs())
            o64 = env.get_obs(push=False, dtype=torch.float64)
            ref.round_f32()
            check_windows(lambda lo, hi: o64[lo:hi], ref, f"{where} restored", cur, torch.float64)
            env.set_obs_history(True)
        if t in (5, 23):
            check_state(env, mb, where, pushes=ref.cnt)
            check_reads(env, mb, ref, where, ring)
        m = (mb.flags & 1).astype(np.uint8)
        if t == 8:
            m |= (rng.uniform(size=n) < 0.5).astype(np.uint8)
        if m.any() and t < 23:
            ring = env.reset(mask=m, return_obs="ring", retries=0); mb.reset_random(51, mask=m)
            ref.reset(m); ref.push(mb.current_obs(), m)
            if t == 8:
                check_ring(ring, ref, slot.ring_op(False), where + " half reset")
            else:
                slot.ring_op(False)
    check_state(env, mb, "D end", pushes=ref.cnt); check_history(env, ref, "D end")
    env.close()
    print(f"leg D: {time.time() - t0:.1f} s")


@pytest.mark.parametrize("variant", ["thread", "warp"])
def test_f_row_clamp_past_the_episode_slice(cuda, profiles, fonets, variant):
    """Leg F: a table whose rows after start + episode_limit + history are NaN for the latest start S0; explicit resets
    with starts in [S0 - 40, S0]; a third of the envs is never reset and steps 130 times, across steps 119-123 where the
    row clamps.  Ring steps (fused for the thread variant), window-ring steps, k_obs and k_state: every value finite and
    bit-exact against the mirror, which clamps as the kernels do."""
    t0 = time.time()
    s0, n = 2000, 40000 + 7
    _, prof = clamp_tables(profiles, s0)
    env = make_env(cuda, prof, n, variant, seed=1)
    mb = c_mirror.MirrorBatch(fonets[variant], prof.as_dict(), n)
    ref = ObsRef(n, NA, H, cuda)
    slot = Slot()
    rng = np.random.default_rng(12)

    def draw():
        back, e0, a0 = reset_draws(rng, n, NA, 41)
        st = (s0 - back).astype(np.int32)
        st[::3] = s0                               # the never-reset subset starts on the last start
        return st, e0, a0

    st, e0, a0 = draw()
    ring = env.reset(st, e0, a0, return_obs="ring"); mb.reset(st, e0, a0)
    ref.push(mb.current_obs()); slot.ring_op(False)
    never = np.zeros(n, dtype=bool); never[::3] = True
    g = torch.Generator(device=cuda).manual_seed(13)
    for t in range(130):
        where = f"F[{variant}] step {t}"
        a, kw, am = act_for(t, g, n)
        as_window = t % 5 == 4
        r, d, info, o = env.step(a, return_obs=True if as_window else "ring", **kw)
        rr, dd, ii = mb.step(am)
        ref.push(mb.current_obs())
        assert bool(torch.isfinite(r).all()) and bool(torch.isfinite(env._info).all()), where
        check_outputs(env, r, d, rr, dd, ii, where)
        check_state(env, mb, where, pushes=ref.cnt)
        if as_window:
            slot.generic_push()
            check_windows(lambda lo, hi: o[lo:hi], ref, where)
        else:
            fused = variant == "thread"
            if not fused:
                slot.generic_push()
            check_ring(o, ref, slot.ring_op(fused), where)
        if t >= 116 or t % 20 == 7:
            check_reads(env, mb, ref, where)
            assert bool(torch.isfinite(env.get_state(torch.float64)).all()), where
        if t % 25 == 24 and t < 110:               # the other envs start new episodes
            st, e0, a0 = draw()
            m = (~never).astype(np.uint8)
            ring = env.reset(st, e0, a0, mask=m, return_obs="ring"); mb.reset(st, e0, a0, mask=m)
            ref.reset(m); ref.push(mb.current_obs(), m)
            check_ring(ring, ref, slot.ring_op(False), where + " reset")
    assert int(mb.steps[never].min()) == 131
    check_history(env, ref, f"F[{variant}] end")
    env.close()
    print(f"leg F[{variant}]: {time.time() - t0:.1f} s")
