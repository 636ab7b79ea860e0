"""env.preview_step / fp_step_preview: the step's computation for K candidate actions per env without committing it.

 * equals step bit for bit: reward, done, info, voltages and violation mask of preview_step(a) are those of a following
   step(a) and of env.voltages / env.violation_mask after it, at every step of a whole episode;
 * touches nothing: records, voltages, setpoints, line flows, both observation histories and the statistics partials
   are byte-identical before and after previews, and a step after previews gives the bits of a step without them;
 * K candidates in one launch equal K single-candidate calls;
 * argument and call-sequence checks.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from _env_check import actions, bits, draws, make_env, ptr, scaled_profiles
from _feeders import assert_same_bytes, snapshot
from flexgpu import _lib


def candidates(kind, rng, shape):
    return torch.from_numpy(actions(kind, rng, shape, 0.3))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [500, 3001])
@pytest.mark.parametrize("kind", ["f32", "f64", "policy", "raw"])
def test_preview_equals_the_following_step_over_an_episode(cuda, profiles, variant, kind, n):
    """At every step of a 95-step episode (the first step, the episode limit, done and the row in force included),
    preview_step(a) returns what step(a) then returns, and the voltages / mask that step leaves in the env."""
    env = make_env(cuda, profiles, n, variant, **({"alg": "safemaddpg"} if kind == "raw" else {}))
    env.reset(*draws(1, env), return_obs=False)
    rng = np.random.default_rng(2)
    translate = kind == "policy"
    n_failed = 0
    for t in range(env.episode_limit):
        a = candidates(kind, rng, (n, 5, 4))
        if t == 40:                                                 # NaN actions: the failure path
            a[::97, 1, 2] = float("nan")
        inj = None
        if t == 60:                                                 # injected failures
            inj = torch.zeros(n, dtype=torch.uint8); inj[5::31] = 1
            env.inject_failure(inj)
        r, d, info, V, vm = env.preview_step(a, translate=translate, want_voltage=True, want_mask=True)
        r, d, V, vm = r.clone(), d.clone(), V.clone(), vm.clone()
        info = {k: v.clone() for k, v in info.items()}
        rs, ds, infos = env.step(a, translate=translate)
        assert torch.equal(bits(r), bits(rs)), t
        assert torch.equal(d, ds), t
        assert info.keys() == infos.keys()
        for k in info:
            assert torch.equal(bits(info[k]), bits(infos[k])), (t, k)
        assert torch.equal(bits(V), bits(env.voltages)), t
        assert torch.equal(vm, env.violation_mask), t
        n_failed += int(infos["solver_failed"].sum())
        if inj is not None:
            env.inject_failure(None)
    assert bool(d.all()), "the last step reaches the episode limit"
    assert n_failed > 0, "the episode must exercise the failure path"
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 8])
def test_preview_touches_nothing(cuda, profiles, variant, k):
    """Heavy loading (thousands of violations), injected failures and NaN actions: the handle's state is
    byte-identical before and after previews, and the next step gives the bits of a twin env that never previewed."""
    heavy = scaled_profiles(profiles, every_other_day=False)
    n = 1000
    envs = [make_env(cuda, heavy, n, variant) for _ in range(2)]
    rng = np.random.default_rng(5)
    for env in envs:
        env.keep_line_flows(True)
        env.reset(*draws(3, env), return_obs=False)
    for t in range(3):                                              # some history in both observation rings
        a = candidates("f32", np.random.default_rng(10 + t), (n, 5, 4))
        for env in envs:
            env.step(a, return_obs="ring")
    inj = torch.zeros(n, dtype=torch.uint8); inj[::7] = 1
    envs[0].inject_failure(inj)
    before = snapshot(envs[0])
    violations = 0
    for rep in range(3):
        cand = candidates("f32" if rep != 1 else "f64", rng, (k, n, 5, 4))
        cand[:, ::13, 2, 1] = float("nan")
        for translate in (False, True):
            if translate and cand.dtype != torch.float32:
                continue
            r, d, info, V, vm = envs[0].preview_step(cand if k > 1 else cand[0], translate=translate, want_voltage=True,
                                                     want_mask=True)
            violations += int(((V > 1.1) | (V < 0.9)).sum())
            assert bool(info["solver_failed"].bool().any())
    assert violations > 1000, "the loading must produce violations"
    assert_same_bytes(before, snapshot(envs[0]))
    envs[0].inject_failure(None)
    a = candidates("f32", rng, (n, 5, 4))
    outs = []
    for env in envs:
        r, d, info = env.step(a)
        outs.append((r.clone(), d.clone(), {k_: v.clone() for k_, v in info.items()}))
    assert torch.equal(bits(outs[0][0]), bits(outs[1][0])) and torch.equal(outs[0][1], outs[1][1])
    for k_ in outs[0][2]:
        assert torch.equal(bits(outs[0][2][k_]), bits(outs[1][2][k_])), k_
    assert_same_bytes(snapshot(envs[0]), snapshot(envs[1]))
    for env in envs:
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 5, 16])
@pytest.mark.parametrize("kind", ["f32", "f64"])
def test_k_candidates_equal_k_single_calls(cuda, profiles, variant, kind, k):
    n = 777                                                         # not a multiple of 32
    env = make_env(cuda, profiles, n, variant)
    env.reset(*draws(7, env), return_obs=False)
    rng = np.random.default_rng(8)
    env.step(candidates(kind, rng, (n, 5, 4)))                      # past the first step: the row in force moves
    cand = candidates(kind, rng, (k, n, 5, 4))
    cand[k - 1, 3::50, 0, 0] = float("nan")
    r, d, info, V, vm = env.preview_step(cand, want_voltage=True, want_mask=True)
    assert r.shape == (k, n) and d.shape == (k, n) and V.shape == (k, n, 33) and vm.shape == (k, n)
    assert info["reward"].shape == (k, n)
    for j in range(k):
        r1, d1, info1, V1, vm1 = env.preview_step(cand[j], want_voltage=True, want_mask=True)
        assert torch.equal(bits(r[j]), bits(r1)) and torch.equal(d[j], d1), j
        assert torch.equal(bits(V[j]), bits(V1)) and torch.equal(vm[j], vm1), j
        for key in info:
            assert torch.equal(bits(info[key][j]), bits(info1[key])), (j, key)
    assert bool(info["solver_failed"][k - 1].bool().any())
    # the outputs are fresh: a later call leaves earlier results alone
    r_again = env.preview_step(cand[0] * 0.5)[0]
    assert torch.equal(bits(r[0]), bits(env.preview_step(cand[0])[0])) and not torch.equal(r_again, r[0])
    env.close()


@pytest.mark.gpu
def test_preview_argument_and_state_checks(cuda, profiles, variant):
    from flexgpu import FlexGpuError
    from flexgpu.config import make_fp_config, normalize_args
    n = 40
    env = make_env(cuda, profiles, n, variant)
    env.reset(*draws(1, env), return_obs=False)
    l, h = env._lib, env._h
    a = torch.rand(n, 5, 4, device=cuda)
    r = torch.empty(n, dtype=torch.float64, device=cuda)
    d = torch.empty(n, dtype=torch.uint8, device=cuda)
    s = _lib.stream(env.device)
    assert l.fp_step_preview(h, 1, ptr(a), _lib.FP_F32, ptr(r), ptr(d), None, None, None, s) == 0
    assert l.fp_step_preview(h, 1, None, _lib.FP_F32, ptr(r), ptr(d), None, None, None, s) == -1
    assert l.fp_step_preview(h, 1, ptr(a), _lib.FP_F32, None, ptr(d), None, None, None, s) == -1
    assert l.fp_step_preview(h, 1, ptr(a), _lib.FP_F32, ptr(r), None, None, None, None, s) == -1
    assert l.fp_step_preview(h, 0, ptr(a), _lib.FP_F32, ptr(r), ptr(d), None, None, None, s) == -1
    assert l.fp_step_preview(h, -3, ptr(a), _lib.FP_F32, ptr(r), ptr(d), None, None, None, s) == -1
    assert l.fp_step_preview(h, 1, ptr(a), 7, ptr(r), ptr(d), None, None, None, s) == -1
    assert b"fp_step_preview" in l.fp_last_error(h)
    with pytest.raises(ValueError):
        env.preview_step(torch.rand(n + 1, 5, 4))
    with pytest.raises(ValueError):
        env.preview_step(torch.rand(2, n, 5, 3))
    env.close()
    # before fp_load_profiles: FP_ESTATE, as fp_step
    args = normalize_args({"kernel_variant": variant})
    cfg = make_fp_config(args, env.network)
    hh = C.c_void_p()
    assert l.fp_create(C.byref(cfg), n, 0, C.byref(hh)) == 0
    try:
        assert l.fp_step_preview(hh, 1, ptr(a), _lib.FP_F32, ptr(r), ptr(d), None, None, None, s) == -3
        assert l.fp_step(hh, ptr(a), _lib.FP_F32, ptr(r), ptr(d), None, None, s) == -3
    finally:
        l.fp_destroy(hh)
    env = make_env(cuda, profiles, n, variant)
    with pytest.raises(ValueError):
        env.preview_step(torch.rand(0, n, 5, 4))
    with pytest.raises(FlexGpuError):                                # failures of the entry point surface as FlexGpuError
        env._check(l.fp_step_preview(env._h, 0, ptr(a), _lib.FP_F32, ptr(r), ptr(d), None, None, None, s), "fp_step_preview")
    env.close()


def test_null_handle_preview_is_rejected():
    assert _lib.lib().fp_step_preview(None, 1, None, 0, None, None, None, None, None, None) == -1
