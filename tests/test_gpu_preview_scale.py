"""GPU: the step preview (fp_step_preview, env.preview_step) at rollout scale, every candidate of every env bit-exact
against the C mirror (tests/_preview_ref.py).

The other preview tests launch at most 400 tiles, fewer than the thread kernel's resident grid, so no warp of theirs
carries a second preview tile.  Here N = 131 072 + 19 unless a leg says otherwise: 4 097 tiles per candidate, each
candidate ending on a 19-env ragged tile.  Every thread-variant leg with K > 1 asserts K tpk >= 2 x the device's
resident warps, so that every warp loops and its next tile often belongs to another candidate: stage [D] requests
tile i+1's records, fp32 actions and PV rows for a candidate other than tile i's, and the fp64 path loads them in [A].
Candidates differ across k and across neighbouring envs; NaN actions sit at the last env of candidate k, the first env
of candidate k + 1 and at env 31 or 32 (a tile edge inside a candidate).  Profiles carry every other day's demand
x 2.4, so previews meet voltage violations and failed solves.  Each candidate is compared on its own; a mismatch names
the leg, the step, the candidate, the env and the first differing element.

  A  thread variant over a whole episode (done envs stepping on into the row clamp): fp32 K = 16, fp64 K = 5,
     translated K = 8 and K = 1; the last candidate committed through step() returns the preview's bits
  B  raw actions (alg="safemaddpg"): fp64 setpoint candidates, K = 5
  C  warp variant: fp32 K = 16, fp64 K = 4, translated K = 1, 16, 4 (the scratch grows, then is reused), translated step
  D  run-time-shape thread kernels (ieee33_4agents: na = 4; custom14: nb = 14, na = 3), N = 100 000 + 13, K = 7
  E  2^20 + 77 envs, K = 16: a 4.4 GB voltage output (byte offsets past 2^32), k N + e up to 1.7e7
  F  the C ABI into sentinel-filled buffers with guard bands, both variants, every combination of null outputs
"""
import itertools
import time

import numpy as np
import pytest
import torch

import _feeders as F
from _env_check import actions, feeder_profiles, make_env, ptr, reset_both, same, same_outputs, scaled_profiles, step_both
from _env_check import all_cores  # noqa: F401  (autouse fixture)
from _feeders import assert_same_bytes, snapshot
from _preview_ref import mirror_preview
from flexgpu import _lib
from oracle import c_mirror, ieee33

pytestmark = pytest.mark.gpu
N = 131072 + 19
NA = 5


@pytest.fixture(scope="module")
def loaded(profiles):
    """Every other day's demand x 2.4 (an episode spans a normal and a heavily loaded day)."""
    return scaled_profiles(profiles, every_other_day=True)


def loops(cuda, k, n):
    """The thread-variant legs' precondition: K tpk tiles are at least twice the warps the device can hold, so every
    warp of the preview grid carries more than one tile whatever the build's occupancy."""
    p = torch.cuda.get_device_properties(cuda)
    tiles, warps = k * ((n + 31) // 32), p.multi_processor_count * (p.max_threads_per_multi_processor // 32)
    assert tiles >= 2 * warps, f"K = {k}, N = {n}: {tiles} tiles < 2 x {warps} resident warps"


def candidates(g, kind, k, n, na=NA):
    """[K, N, na, 4] candidate actions on the device: fp32 / fp64 policy outputs, raw fp32 outputs to translate
    ("policy") or fp64 setpoints ("raw"); NaN at the candidate boundaries and at a tile edge."""
    a = actions(kind, g, (k, n, na, 4), 0.4)
    for j in range(k):
        if j % 2 == 0:
            a[j, n - 1, j % na, j % 4] = float("nan")                          # last lane of the ragged tile
            if j + 1 < k:
                a[j + 1, 0, (j + 1) % na, (j + 2) % 4] = float("nan")          # first env of the next candidate
        a[j, 31 + j % 2, (j + 2) % na, (j + 1) % 4] = float("nan")              # a tile edge inside the candidate
    return a


def preview(env, cand, translate=False):
    """preview_step with voltages and masks, K = 1 through the [N, na, 4] form; outputs with a leading K."""
    k = cand.shape[0]
    out = env.preview_step(cand if k > 1 else cand[0], translate=translate, want_voltage=True, want_mask=True)
    if k == 1:
        r, d, info, V, vm = out
        out = (r[None], d[None], {key: v[None] for key, v in info.items()}, V[None], vm[None])
    return out


def candidate(out, j):
    r, d, info, V, vm = out
    return r[j], d[j], {key: v[j] for key, v in info.items()}, V[j], vm[j]


def check(out, want, where):
    """Every candidate of a preview against mirror_preview(); returns (failed solves, envs with a violation)."""
    failed = violated = j = 0
    for j, w in enumerate(want):
        same_outputs(candidate(out, j), w, f"{where} candidate {j}")
        failed += int(w[2][:, 7].sum()); violated += int((w[4] != 0).sum())
    assert j + 1 == out[0].shape[0], where
    return failed, violated


def check_commit(env, mb, out, step_out, where):
    """A step committing the preview's last candidate returned its bits and left its voltages and mask, the mirror's."""
    r, d, info = step_out
    k = out[0].shape[0]
    pr, pd, pinfo, pV, pvm = candidate(out, k - 1)
    want = (pr, pd, torch.stack([pinfo[key] for key in _lib.INFO_KEYS], 1), pV, pvm)
    same_outputs((r, d, info, env.voltages, env.violation_mask), want, f"{where}: step after the preview")
    same(env.voltages, mb.V, "voltages", f"{where}: step vs mirror")
    same(env.setpoints, mb.setp, "setpoints", f"{where}: step vs mirror")


def test_a_thread_variant_over_an_episode(cuda, loaded, fonets):
    """Leg A: 30 steps, a reset of a random half (steps differ within a tile), then a 95-step episode whose done envs of
    even index are reset after every step while the odd ones step on past done into the row clamp.  Six steps preview
    before committing: fp32 K = 16 (65 552 tiles), fp64 K = 5 (k_env_t<.., A64>), translated K = 8 with ~300 injected
    failures, K = 1, fp32 K = 16 again and fp64 K = 5 at the last step; the handle's bytes are unchanged by each, and
    the step committing candidate K - 1 returns its bits."""
    t0 = time.time()
    env = make_env(cuda, loaded, N, seed=21)
    mb = c_mirror.MirrorBatch(fonets["thread"], loaded.as_dict(), N)
    env.reset(return_obs=False, retries=0); mb.reset_random(21)
    g = torch.Generator(device=cuda).manual_seed(22)
    rng = np.random.default_rng(23)
    for t in range(30):
        step_both(env, mb, actions("f32", g, (N, NA, 4), 0.4), f"A warm-up step {t}")
    m = (rng.uniform(size=N) < 0.5).astype(np.uint8)
    env.reset(mask=m, return_obs=False, retries=0); mb.reset_random(21, mask=m)
    plan = {0: ("f32", 16), 19: ("f64", 5), 45: ("policy", 8), 60: ("f32", 1), 77: ("f32", 16), 94: ("f64", 5)}
    even = np.arange(N) % 2 == 0
    failed = violated = done = 0
    for t in range(95):
        where = f"A step {t}"
        inj = None
        if t == 45:
            inj = np.zeros(N, dtype=np.uint8); inj[rng.integers(0, N, 300)] = 1
            env.inject_failure(inj)
        kind, k = plan.get(t, ("f32", 0))
        translate = kind == "policy"
        if k:
            if k > 1:
                loops(cuda, k, N)
            cand = candidates(g, kind, k, N)
            before = snapshot(env)
            out = preview(env, cand, translate)
            assert_same_bytes(before, snapshot(env))
            del before
            f, v = check(out, mirror_preview(mb, cand, inject=inj, translate=translate), where)
            failed += f; violated += v
            a = cand[k - 1]
        else:
            a = actions("f32", g, (N, NA, 4), 0.4)
        step = step_both(env, mb, a, where, translate, inj)
        if k:
            check_commit(env, mb, out, step, where)
            del out
        if inj is not None:
            assert int(mb.done[inj.astype(bool)].sum()) == int(inj.sum())
            env.inject_failure(None)
        done += int(mb.done.sum())
        m = (mb.done.astype(bool) & even).astype(np.uint8)
        if m.any():
            env.reset(mask=m, return_obs=False, retries=0); mb.reset_random(21, mask=m)
    assert failed > 300 and violated > 0 and done > 0, (failed, violated, done)
    assert int(mb.steps[1::2].max()) > env.episode_limit + env.history + 1      # odd envs stepped into the row clamp
    env.close()
    print(f"leg A: {time.time() - t0:.1f} s")


def test_b_raw_actions(cuda, loaded, tree, args):
    """Leg B: alg="safemaddpg" (actions are setpoints), fp64 candidates, K = 5, three steps into an episode."""
    t0 = time.time()
    k = 5
    loops(cuda, k, N)
    env = make_env(cuda, loaded, N, seed=1, alg="safemaddpg")
    mb = c_mirror.MirrorBatch(c_mirror.make_net(tree, args, args["buildings"], raw_actions=True), loaded.as_dict(), N)
    rng = np.random.default_rng(31)
    reset_both(env, mb, rng)
    g = torch.Generator(device=cuda).manual_seed(32)
    for t in range(3):
        step_both(env, mb, candidates(g, "raw", 1, N)[0], f"B step {t}")
    cand = candidates(g, "raw", k, N)
    before = snapshot(env)
    out = preview(env, cand)
    assert_same_bytes(before, snapshot(env))
    failed, violated = check(out, mirror_preview(mb, cand), "B")
    check_commit(env, mb, out, step_both(env, mb, cand[k - 1], "B commit"), "B")
    assert failed >= 2 * k
    env.close()
    print(f"leg B: {time.time() - t0:.1f} s")


def test_c_warp_variant(cuda, loaded, fonets):
    """Leg C: the warp kernel over K N virtual envs: fp32 K = 16, fp64 K = 4, then translated candidates with K = 1, 16
    (the FP_F32_POLICY scratch grows) and 4 (it is reused), then a translated step through the same scratch."""
    t0 = time.time()
    env = make_env(cuda, loaded, N, "warp", seed=41)
    mb = c_mirror.MirrorBatch(fonets["warp"], loaded.as_dict(), N)
    env.reset(return_obs=False, retries=0); mb.reset_random(41)
    g = torch.Generator(device=cuda).manual_seed(42)
    for t in range(2):
        step_both(env, mb, candidates(g, "f32", 1, N)[0], f"C step {t}")
    before = snapshot(env)
    failed = violated = 0
    for kind, k in (("f32", 16), ("f64", 4), ("policy", 1), ("policy", 16), ("policy", 4)):
        translate = kind == "policy"
        cand = candidates(g, kind, k, N)
        out = preview(env, cand, translate)
        f, v = check(out, mirror_preview(mb, cand, translate=translate), f"C {kind} K = {k}")
        failed += f; violated += v
        del out
    assert_same_bytes(before, snapshot(env))
    assert failed > 0 and violated > 0
    a = candidates(g, "policy", 1, N)[0]
    step_both(env, mb, a, "C translated step", translate=True)
    same(env.voltages, mb.V, "voltages", "C translated step")
    same(env.violation_mask, mb.vmask, "violation mask", "C translated step")
    env.close()
    print(f"leg C: {time.time() - t0:.1f} s")


@pytest.mark.parametrize("name", ["ieee33_4agents", "custom14"])
def test_d_run_time_shape(cuda, name):
    """Leg D: k_env_t<MODE_PREVIEW, RtShape, ..> with na < 5 (the staged fp32 actions are n_left na 16-byte chunks),
    N = 100 000 + 13 (tpk = 3 126), fp32 and fp64 candidates, K = 7, two steps apart."""
    t0 = time.time()
    net = F.feeder(name)
    prof = scaled_profiles(feeder_profiles(net), every_other_day=True)
    n, k = 100000 + 13, 7
    loops(cuda, k, n)
    env = make_env(cuda, prof, n, net=net, seed=1)
    na = env.n_agents
    assert na < 5
    fonet = c_mirror.make_net(ieee33.tree_arrays(net), F.env_args(net), net['buildings'])
    mb = c_mirror.MirrorBatch(fonet, prof.as_dict(), n)
    rng = np.random.default_rng(51)
    reset_both(env, mb, rng)
    g = torch.Generator(device=cuda).manual_seed(52)
    failed = 0
    for t in range(5):
        where = f"D[{name}] step {t}"
        kind = {1: "f32", 3: "f64"}.get(t)
        if kind is None:
            step_both(env, mb, candidates(g, "f32", 1, n, na)[0], where)
            continue
        cand = candidates(g, kind, k, n, na)
        before = snapshot(env)
        out = preview(env, cand)
        assert_same_bytes(before, snapshot(env))
        failed += check(out, mirror_preview(mb, cand), where)[0]
        check_commit(env, mb, out, step_both(env, mb, cand[k - 1], where), where)
        del out
    assert failed >= 2 * k
    env.close()
    print(f"leg D[{name}]: {time.time() - t0:.1f} s")


def test_e_two_pow_20_envs(cuda, loaded, fonets):
    """Leg E: 2^20 + 77 envs, K = 16 fp32 candidates with voltages and masks: the [K][N][33] voltage output is 4.4 GB,
    so its byte offsets pass 2^32.  Records, voltages and setpoints are unchanged by the preview (the fp64 history of
    this size is not snapshotted)."""
    t0 = time.time()
    n, k = 2 ** 20 + 77, 16
    loops(cuda, k, n)
    env = make_env(cuda, loaded, n, seed=61)
    mb = c_mirror.MirrorBatch(fonets["thread"], loaded.as_dict(), n)
    env.reset(return_obs=False, retries=0); mb.reset_random(61)
    g = torch.Generator(device=cuda).manual_seed(62)
    step_both(env, mb, candidates(g, "f32", 1, n)[0], "E step 0")
    cand = candidates(g, "f32", k, n)
    before = {"rec": env.rec.clone(), "V": env.voltages.clone(), "setp": env.setpoints.clone()}
    out = preview(env, cand)
    assert out[3].numel() * 8 > 2 ** 32 and k * n > 1.6e7
    after = {"rec": env.rec, "V": env.voltages, "setp": env.setpoints}
    for key in before:
        same(after[key], before[key], key, "E: state after the preview")
    del before, after
    failed, violated = check(out, mirror_preview(mb, cand), "E")
    assert failed > 0 and violated > 0
    env.close()
    print(f"leg E: {time.time() - t0:.1f} s")


GUARD = 4096 + 48                                                   # bytes before a payload: 16-byte aligned, not 128


def guarded(count, dtype, fill, dev):
    """A sentinel-filled buffer and its payload of `count` elements, with a guard band before and after."""
    size = torch.tensor([], dtype=dtype).element_size()
    pre = GUARD // size
    buf = torch.full((pre + count + pre,), fill, dtype=dtype, device=dev)
    return buf, buf[pre:pre + count], pre


def guards_intact(buf, pre, count, fill, what, where):
    for band in (buf[:pre], buf[pre + count:]):
        same(band, torch.full_like(band, fill), f"guard band of {what}", where)


SENTINELS = {torch.float64: -7.25e6, torch.uint8: 0xA5, torch.int64: 0x5A5A5A5A5A5A5A5A}


@pytest.mark.parametrize("variant", ["thread", "warp"])
def test_f_outputs_through_the_c_abi(cuda, loaded, fonets, variant):
    """Leg F: fp_step_preview into payloads carved out of sentinel-filled buffers at 16-byte aligned offsets, guard bands
    of 4 KB before and after: the bands unchanged, the payloads the mirror's.  Then every combination of null info /
    voltage / mask writes the requested outputs as the full call did and nothing around them."""
    t0 = time.time()
    k = 5
    if variant == "thread":
        loops(cuda, k, N)
    env = make_env(cuda, loaded, N, variant, seed=71)
    mb = c_mirror.MirrorBatch(fonets[variant], loaded.as_dict(), N)
    env.reset(return_obs=False, retries=0); mb.reset_random(71)
    g = torch.Generator(device=cuda).manual_seed(72)
    step_both(env, mb, candidates(g, "f32", 1, N)[0], f"F[{variant}] step 0")
    cand = candidates(g, "f32", k, N)
    l, h, s = env._lib, env._h, _lib.stream(env.device)
    nb = env.n_bus
    shapes = {"reward": (k * N, torch.float64), "done": (k * N, torch.uint8), "info": (k * N * 8, torch.float64),
              "voltage": (k * N * nb, torch.float64), "mask": (k * N, torch.int64)}
    def call(want, where):
        bufs = {key: guarded(cnt, dt, SENTINELS[dt], cuda) for key, (cnt, dt) in shapes.items()
                if key in ("reward", "done") or key in want}
        pay = {key: b[1] for key, b in bufs.items()}
        rc = l.fp_step_preview(h, k, ptr(cand), _lib.FP_F32, ptr(pay["reward"]), ptr(pay["done"]), ptr(pay.get("info")),
                               ptr(pay.get("voltage")), ptr(pay.get("mask")), s)
        assert rc == 0, (where, l.fp_last_error(h))
        torch.cuda.synchronize()
        for key, (buf, _, pre) in bufs.items():
            guards_intact(buf, pre, shapes[key][0], SENTINELS[shapes[key][1]], key, where)
        return pay

    before = snapshot(env)
    full = call({"info", "voltage", "mask"}, f"F[{variant}] full call")
    assert_same_bytes(before, snapshot(env))
    out = (full["reward"].view(k, N), full["done"].view(torch.bool).view(k, N),
           {key: full["info"].view(k, N, 8)[..., i] for i, key in enumerate(_lib.INFO_KEYS)},
           full["voltage"].view(k, N, nb), full["mask"].view(k, N))
    failed, violated = check(out, mirror_preview(mb, cand), f"F[{variant}] full call")
    assert failed > 0 and violated > 0
    for flags in itertools.product((False, True), repeat=3):
        if all(flags):
            continue
        want = {key for key, on in zip(("info", "voltage", "mask"), flags) if on}
        where = f"F[{variant}] outputs {sorted(want)}"
        got = call(want, where)
        for key in got:
            same(got[key].view(k * N, -1), full[key].view(k * N, -1), key, where)     # indexed by virtual env k N + e
    assert_same_bytes(before, snapshot(env))
    env.close()
    print(f"leg F[{variant}]: {time.time() - t0:.1f} s")
