"""CPU: the step preview's reference (tests/_preview_ref.py) and the env-parity comparisons (tests/_env_check.py), on
the C mirror alone.  mirror_preview() leaves the batch byte-identical, gives candidate j what a fresh batch in the same
state gives for one step of candidate j (injected failures, NaN actions, translated actions and voltage violations
included), and permutes with its candidates; same() compares bits and names the candidate and the env of a mismatch;
check_state() names any one field of the state that differs from the mirror's."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from _env_check import check_state, reset_draws, same, same_outputs, scaled_profiles
from _preview_ref import mirror_copy, mirror_preview
from oracle import c_mirror

N, NA, K = 32 * 3 + 5, 5, 6
NAN_ENV = {1: N - 1, 2: 0, 4: 31}                                       # candidate: an env with a NaN action


@pytest.fixture(scope="module")
def heavy(profiles):
    """Every other day's demand x 2.4: voltage violations and some failed solves."""
    return scaled_profiles(profiles, every_other_day=True).as_dict()


def batch(fonet, heavy):
    """A batch a few steps into an episode, the same every call: varied rows in force, energies and setpoints."""
    mb = c_mirror.MirrorBatch(fonet, heavy, N)
    rng = np.random.default_rng(1)
    mb.reset(*reset_draws(rng, N, NA, mb.start_range))
    for _ in range(3):
        mb.step(rng.normal(0.4, 0.6, (N, NA, 4)).astype(np.float32))
    return mb


def candidates(dtype=np.float64, seed=2):
    c = np.random.default_rng(seed).normal(0.4, 0.6, (K, N, NA, 4)).astype(dtype)
    c[1, N - 1, 2, 0] = np.nan                                          # the last env of one candidate, the first of the next
    c[2, 0, 0, 3] = np.nan
    c[4, 31:33, 4, 1] = np.nan
    return c


def inject_mask():
    inj = np.zeros(N, dtype=np.uint8)
    inj[5::17] = 1
    return inj


def as_bytes(saved):
    return {k: v.tobytes() for k, v in saved.items()}


def equal_outputs(a, b):
    return all(x.tobytes() == y.tobytes() for x, y in zip(a, b))


@pytest.mark.parametrize("variant", [c_mirror.VARIANT_THREAD, c_mirror.VARIANT_WARP])
def test_preview_leaves_the_batch_unchanged(tree, args, heavy, variant):
    fonet = c_mirror.make_net(tree, args, args["buildings"], variant=variant)
    mb = batch(fonet, heavy)
    before = as_bytes(mirror_copy(mb))
    outs = list(mirror_preview(mb, candidates(), inject=inject_mask()))
    assert len(outs) == K
    assert as_bytes(mirror_copy(mb)) == before
    for _ in mirror_preview(mb, candidates(np.float32), translate=True):    # a caller that stops after one candidate
        break
    assert as_bytes(mirror_copy(mb)) == before
    # the batch still steps as one that never previewed
    a = candidates(seed=9)[0]
    twin = batch(fonet, heavy)
    assert equal_outputs(mb.step(a), twin.step(a))
    assert as_bytes(mirror_copy(mb)) == as_bytes(mirror_copy(twin))


@pytest.mark.parametrize("kind", ["f64", "f32", "policy"])
def test_candidate_j_equals_one_step_of_a_fresh_batch(fonet, heavy, kind):
    cand = candidates(np.float64 if kind == "f64" else np.float32)
    translate = kind == "policy"
    inj = inject_mask()
    mb = batch(fonet, heavy)
    outs = list(mirror_preview(mb, cand, inject=inj, translate=translate))
    failed = violated = 0
    for j in range(K):
        fresh = batch(fonet, heavy)
        a = c_mirror.translate_action_f32(cand[j]) if translate else cand[j]
        r, d, info = fresh.step(a, inject=inj)
        assert equal_outputs(outs[j], (r, d, info, fresh.V, fresh.vmask)), j
        assert outs[j][1].dtype == bool and outs[j][4].dtype == np.uint64
        failed += int(info[:, 7].sum()); violated += int((fresh.vmask != 0).sum())
        if j in NAN_ENV:
            assert info[NAN_ENV[j], 7] == 1.0, j                           # a NaN action fails its env
        assert (info[inj.astype(bool), 7] == 1.0).all(), j
        bad = info[:, 7] == 1.0                                         # a failed solve reports the rolled-back voltages
        assert np.array_equal(outs[j][3][bad], mb.V[bad]), j
    assert failed > K * int(inj.sum()) and violated > 0
    # torch candidates (what the GPU tests hand over) give the same
    assert all(equal_outputs(x, y) for x, y in zip(outs, mirror_preview(mb, torch.from_numpy(cand), inject=inj,
                                                                         translate=translate)))


def test_permuted_candidates_permute_the_outputs(fonet, heavy):
    cand = candidates()
    mb = batch(fonet, heavy)
    outs = list(mirror_preview(mb, cand))
    perm = np.random.default_rng(3).permutation(K)
    for j, out in enumerate(mirror_preview(mb, cand[perm])):
        assert equal_outputs(out, outs[perm[j]]), j
    assert not equal_outputs(outs[0], outs[1])                          # the candidates differ


def test_same_compares_bits_and_names_the_candidate_and_the_env():
    x = torch.tensor([[1.0, float("nan")], [0.0, 2.0], [3.0, 4.0]], dtype=torch.float64)
    same(x, x.clone().numpy(), "voltages", "leg candidate 3")                   # NaN equals itself
    y = x.clone(); y[1, 0] = -0.0
    with pytest.raises(AssertionError, match=r"leg candidate 3: voltages differs at env 1, element \(1, 0\)"):
        same(y, x.numpy(), "voltages", "leg candidate 3")
    y = x.clone(); y[2, 1] = np.nextafter(4.0, 5.0)
    with pytest.raises(AssertionError, match="at env 2"):
        same(y, x, "voltages", "")
    m = np.array([0, 1 << 63, 5], dtype=np.uint64)                              # masks: the mirror's u64, torch's i64
    same(torch.from_numpy(m.view(np.int64)), m, "violation mask", "")
    with pytest.raises(AssertionError, match="at env 1"):
        same(torch.tensor([0, 1, 5]), m, "violation mask", "")
    with pytest.raises(AssertionError, match="float32"):                        # dtypes must agree
        same(x.float(), x, "reward", "")
    d = np.array([True, False, True])
    same(torch.from_numpy(d), d, "done", "")
    with pytest.raises(AssertionError, match="done differs at env 2"):
        same(torch.tensor([True, False, False]), d, "done", "")


def test_same_outputs_checks_every_part(fonet, heavy):
    mb = batch(fonet, heavy)
    want = next(mirror_preview(mb, candidates()[:1]))
    got = [torch.from_numpy(np.ascontiguousarray(w)) for w in want[:3]] + [torch.from_numpy(want[3]),
                                                                          torch.from_numpy(want[4].view(np.int64))]
    info = {k: got[2][:, i] for i, k in enumerate(("reward", "revenue", "der_cost", "ess_cost", "discomfort_penalty",
                                                   "voltage_penalty", "cumulative_reward", "solver_failed"))}
    same_outputs(got, want, "x")
    same_outputs((got[0], got[1], info, got[3], got[4]), want, "x")
    for part, what in ((2, r"info\[voltage_penalty\]"), (3, "voltages"), (4, "violation mask")):
        bad = [g.clone() for g in got]
        bad[part].view(-1)[5 if part != 2 else 7 * 8 + 5] += 1
        with pytest.raises(AssertionError, match=f"{what} differs at env 7" if part == 2 else what):
            same_outputs(bad, want, "x")
        same_outputs(bad, want, "x", info=part != 2, voltage=part != 3, mask=part != 4)


# ------------------------------------------------------------------ check_state
FLIPS = [("E_init", 4, 0), ("E_cur", 5, 51), ("cumulative reward", 10, 62), ("start", 11, 2), ("steps", 11, 33),
         ("push count", 12, 4), ("episode", 12, 40), ("violation mask", 13, 32), ("violation count", 14, 1),
         ("flags", 14, 34), ("line-limit mask", 15, 31), ("power-flow passes", 15, 32)]    # (field, record word, bit)


def test_check_state_names_every_field(fonet, heavy):
    """check_state() passes on a stand-in env whose record, voltages and setpoints are the mirror's state, and names the
    field and the env of any one flipped bit: each field of the 16 record words, the voltages and the setpoints.  The
    push count is compared only when it is given."""
    mb = batch(fonet, heavy)
    mb.step(candidates()[0], inject=inject_mask())                      # failed envs: flags and rolled-back voltages
    pushes = np.arange(N) % 25

    def u64(lo, hi):
        return (lo.astype(np.uint32).astype(np.uint64) | (hi.astype(np.uint32).astype(np.uint64) << np.uint64(32))).view(
            np.int64)

    def stand_in():
        rec = np.empty((N, 16), dtype=np.int64)
        rec[:, 0:5] = mb.E_init.view(np.int64); rec[:, 5:10] = mb.E_cur.view(np.int64); rec[:, 10] = mb.cum.view(np.int64)
        rec[:, 11] = u64(mb.start, mb.steps); rec[:, 12] = u64(pushes, mb.episode); rec[:, 13] = mb.vmask.view(np.int64)
        rec[:, 14] = u64(mb.vcount, mb.flags); rec[:, 15] = u64(mb.lmask, mb.iters)
        return SimpleNamespace(rec=torch.from_numpy(rec), voltages=torch.from_numpy(mb.V.copy()),
                               setpoints=torch.from_numpy(mb.setp.copy()))

    assert (mb.flags != 0).any() and (mb.vmask != 0).any() and (mb.lmask != 0).any()
    check_state(stand_in(), mb, "pin", pushes=pushes)
    for k, (field, word, bit) in enumerate(FLIPS):
        env, e = stand_in(), (37 * k + 5) % N
        env.rec[e, word] ^= 1 << bit
        with pytest.raises(AssertionError, match=f"pin: {field} differs at env {e},"):
            check_state(env, mb, "pin", pushes=pushes)
        if field == "push count":
            check_state(env, mb, "pin")
    for k, field in enumerate(("voltages", "setpoints")):
        env, e = stand_in(), 3 + k
        getattr(env, field).view(torch.int64).view(N, -1)[e, 7] ^= 1
        with pytest.raises(AssertionError, match=f"pin: {field} differs at env {e},"):
            check_state(env, mb, "pin")
