"""GPU parity of the device rollout path (SURVEY 8f ranks 1-2) through the C ABI:

  * fp_policy_act (tcgen05) against the reference's own RNNAgent + Model.policy + select_action run on CPU torch
    (tests/golden/ref_policy.npz, written by tests/golden/make_ref_policy_golden.py from the reference's code; loaded
    through tests/_golden.py, which rebuilds the seeded inputs and keeps the hidden states of a fixed subset of envs).
    Tolerances (fp32 arithmetic, stated): the device holds the weight MATRICES as TF32 and keeps activations at fp32
    accuracy, so against the reference evaluated with the same TF32-rounded matrices means / hidden states / actions
    agree to 2e-5 (observed ~2e-6) and log-probabilities to 2e-4 (the tanh correction log(1 - a^2 + 1e-6) amplifies
    rounding near |a| = 1); against the reference with its unrounded fp32 initialisation the bound is 5e-4.
  * Transition fields written by DeviceRollout against the env's own dense observations / rewards and the policy outputs
    (bit-exact: pure data movement).
  * learner_batch against the reference's TransReplayBuffer.get_batch + Model.unpack_data + MADDPG.value's critic input."""
import os

import numpy as np
import pytest
import torch
from _golden import load_ref_policy
from _rollout_ref import KEYS, mlp_critic_torch, ring_from_windows, torch_mats

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_policy.npz")


@pytest.fixture(scope="module")
def gold():
    return load_ref_policy()


def hidden_rows(gold, n):
    """[n, 5, 64] hidden-state inputs: the reference's step-0 hidden states (TF32 weights) of the stored envs, repeated."""
    return np.resize(gold["t_hid0"], (n, 5, 64))


@pytest.mark.parametrize("tag,tol,tol_lp", [("t_", 2e-5, 2e-4), ("", 5e-4, 5e-3)])
def test_policy_matches_reference_rnn_agent(gold, cuda, tag, tol, tol_lp):
    from flexgpu.policy import DevicePolicy
    prefix = "wt_" if tag == "t_" else "w_"
    pol = DevicePolicy({k: gold[prefix + k] for k in KEYS}, device=cuda, std=1.0)
    n = gold["obs0"].shape[0]
    hid = None
    worst = {}
    rows = torch.from_numpy(gold["hid_rows"]).to(cuda)           # the envs whose hidden states the fixture keeps
    for t, slot in enumerate((7, 23, 0)):                       # three recurrent steps, three rotations of the ring
        ring = ring_from_windows(gold[f"obs{t}"], slot).to(cuda)
        hid_out = torch.empty(n, 5, 64, device=cuda)
        act, logp, hid_new, mean = pol.act(ring, slot=slot, n_envs=n, hid_in=hid, explore=True, eps=torch.from_numpy(gold[f"eps{t}"]),
                                           hid_out=hid_out, want_mean=True)
        for name, got, bound in (("mean", mean, tol), ("hid", hid_new[rows], tol), ("action", act, tol), ("logp", logp, tol_lp)):
            err = float(np.max(np.abs(got.cpu().numpy() - gold[f"{tag}{name}{t}"])))
            worst[name] = max(worst.get(name, 0.0), err)
            assert err < bound, (name, t, err)
        act_t, lp_t, _, _ = pol.act(ring, slot=slot, n_envs=n, hid_in=hid, explore=False, hid_out=torch.empty_like(hid_out))
        assert np.max(np.abs(act_t.cpu().numpy() - gold[f"{tag}action_test{t}"])) < tol          # status 'test': tanh(mean)
        hid = hid_new
    print("max abs errors vs reference", tag or "fp32-weights", worst)
    pol.close()


def test_policy_rows_are_independent_and_ragged_sizes(gold, cuda):
    """Any n (tail blocks, n not a multiple of 128 or 32): every row depends on its own inputs only."""
    from flexgpu.policy import DevicePolicy
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda)
    obs = gold["obs1"]
    h0 = hidden_rows(gold, 160)
    full = None
    for n in (160, 129, 128, 33, 1):
        ring = ring_from_windows(obs[:n], 5).to(cuda)
        h_in = torch.from_numpy(h0[:n]).to(cuda).contiguous()
        act, _, hid, mean = pol.act(ring, slot=5, n_envs=n, hid_in=h_in, explore=False, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))
        got = (mean.cpu().numpy().copy(), hid.cpu().numpy().copy())
        if full is None:
            full = got
        else:
            assert np.array_equal(got[0], full[0][:n]) and np.array_equal(got[1], full[1][:n])
    # the env-minor hidden-state layout [5, 64, n_pad] (the kernel's native one) gives the same bits
    n = 160
    ring = ring_from_windows(obs, 5).to(cuda)
    h_rows = torch.from_numpy(h0).to(cuda).contiguous()
    h_em = torch.zeros(5, 64, 160, device=cuda); h_em[:, :, :n] = h_rows.permute(1, 2, 0)
    out_em = torch.empty(5, 64, 160, device=cuda)
    _, _, hid_em, mean_em = pol.act(ring, slot=5, n_envs=n, hid_in=h_em.contiguous(), explore=False, want_mean=True, hid_out=out_em,
                                    hid_layout="env_minor")
    assert np.array_equal(mean_em.cpu().numpy(), full[0]) and np.array_equal(hid_em[:, :, :n].permute(2, 0, 1).cpu().numpy(), full[1])
    # reset mask: the masked envs act from a zero hidden state
    n = 160
    ring = ring_from_windows(obs, 5).to(cuda)
    h_in = torch.from_numpy(h0).to(cuda).contiguous()
    mask = torch.zeros(n, dtype=torch.uint8, device=cuda); mask[::3] = 1
    _, _, hid_m, mean_m = pol.act(ring, slot=5, n_envs=n, hid_in=h_in, reset=mask, explore=False, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))
    mean_m = mean_m.cpu().numpy().copy()
    _, _, _, mean_z = pol.act(ring, slot=5, n_envs=n, hid_in=None, explore=False, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))
    mean_z = mean_z.cpu().numpy()
    assert np.array_equal(mean_m[::3], mean_z[::3]) and np.array_equal(np.delete(mean_m, np.s_[::3], 0), np.delete(full[0], np.s_[::3], 0))
    pol.close()


def test_policy_saturated_gates_stay_finite(gold, cuda):
    """GRU weights x 32 (still TF32-exact): gate pre-activations of +-100 and more.  The kernel takes its reciprocals four
    at a time from the reciprocal of a product and clamps the gate arguments to keep that product finite -- the result
    must stay finite and agree with a plain fp64 evaluation (bound 1e-4: the x 32 amplifies fc1's fp32 rounding)."""
    from flexgpu.policy import DevicePolicy
    w = {k: np.array(gold["wt_" + k], dtype=np.float32) for k in KEYS}
    for k in ("rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh"):
        w[k] = w[k] * np.float32(32.0)
    pol = DevicePolicy(w, device=cuda)
    obs = gold["obs1"]
    n = obs.shape[0]
    h0 = (np.random.default_rng(3).uniform(-1, 1, (n, 5, 64))).astype(np.float32)
    ring = ring_from_windows(obs, 11).to(cuda)
    _, _, hid, mean = pol.act(ring, slot=11, n_envs=n, hid_in=torch.from_numpy(h0).to(cuda), explore=False, want_mean=True,
                              hid_out=torch.empty(n, 5, 64, device=cuda))
    t = {k: torch.from_numpy(v).double() for k, v in w.items()}
    x = torch.cat([torch.from_numpy(obs).double(), torch.eye(5, dtype=torch.float64).expand(n, 5, 5)], dim=-1)
    a = torch.relu(torch.nn.functional.layer_norm(x @ t["fc1.weight"].T + t["fc1.bias"], (64,), t["layernorm.weight"], t["layernorm.bias"]))
    gi = a @ t["rnn.weight_ih"].T + t["rnn.bias_ih"]
    gh = torch.from_numpy(h0).double() @ t["rnn.weight_hh"].T + t["rnn.bias_hh"]
    assert float((gi + gh).abs().max()) > 40.0                   # the clamps are exercised
    r = torch.sigmoid(gi[..., :64] + gh[..., :64]); z = torch.sigmoid(gi[..., 64:128] + gh[..., 64:128])
    nn_ = torch.tanh(gi[..., 128:] + r * gh[..., 128:])
    h1 = (1 - z) * nn_ + z * torch.from_numpy(h0).double()
    m = h1 @ t["fc2.weight"].T + t["fc2.bias"]
    got_h, got_m = hid.cpu().double(), mean.cpu().double()
    assert bool(torch.isfinite(got_h).all()) and bool(torch.isfinite(got_m).all())
    assert float((got_h - h1).abs().max()) < 1e-4 and float((got_m - m).abs().max()) < 1e-4
    pol.close()


def test_policy_nan_observation_poisons_its_row_only(gold, cuda):
    """A NaN in one (env, agent) observation window reaches that row's outputs as NaN (the clamps of the gate arguments
    propagate it, as torch would) and leaves every other row's bits untouched."""
    from flexgpu.policy import DevicePolicy
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda)
    obs = np.array(gold["obs1"], dtype=np.float32)
    n = obs.shape[0]
    outs = []
    for poison in (False, True):
        o = obs.copy()
        if poison:
            o[37, 2, 100] = np.nan
        ring = ring_from_windows(o, 5).to(cuda)
        _, _, hid, mean = pol.act(ring, slot=5, n_envs=n, hid_in=None, explore=False, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))
        outs.append((hid.cpu().numpy().copy(), mean.cpu().numpy().copy()))
    (h0, m0), (h1, m1) = outs
    assert np.isnan(h1[37, 2]).all() and np.isnan(m1[37, 2]).all()
    keep = np.ones((n, 5), dtype=bool); keep[37, 2] = False
    assert np.array_equal(h0[keep], h1[keep]) and np.array_equal(m0[keep], m1[keep])
    pol.close()


def test_policy_philox_sampling(gold, cuda):
    """Device-side exploration noise: N(0, 1) draws keyed by (seed, row, step) -- reproducible, step-dependent."""
    from flexgpu.policy import DevicePolicy
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda, std=1.0, seed=1234)
    n = 4096
    obs = np.tile(gold["obs0"], (26, 1, 1))[:n]
    ring = ring_from_windows(obs, 3).to(cuda)
    a1, lp1, _, m1 = pol.act(ring, slot=3, n_envs=n, explore=True, step=7, want_mean=True)
    a1, lp1, m1 = a1.double().cpu().numpy().copy(), lp1.cpu().numpy().copy(), m1.double().cpu().numpy().copy()
    a2, _, _, _ = pol.act(ring, slot=3, n_envs=n, explore=True, step=7)
    assert np.array_equal(a1, a2.double().cpu().numpy())
    a3, _, _, _ = pol.act(ring, slot=3, n_envs=n, explore=True, step=8)
    assert not np.array_equal(a1, a3.double().cpu().numpy())
    ok = np.abs(a1) < 0.999
    z = (np.arctanh(np.where(ok, a1, 0.0)) - m1)[ok]
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1.0) < 0.03 and abs(np.mean(z ** 3)) < 0.08
    # log_prob consistent with the draws (utils/util.py:56-61)
    want = -0.5 * z ** 2 - 0.9189385332046727 - np.log(1.0 - a1[ok] ** 2 + 1e-6)
    assert np.max(np.abs(lp1[ok] - want)) < 2e-2 and np.median(np.abs(lp1[ok] - want)) < 1e-5
    pol.close()


@pytest.fixture()
def small_env(cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv
    e = BatchedFlexProvisionEnv(None, n_envs=300, device=cuda, profiles=profiles, seed=3)
    yield e
    e.close()


def test_rollout_writes_the_transition_fields(gold, cuda, small_env):
    """DeviceRollout = train_process's loop body (model.py:213-254): what lands in the replay ring is exactly what the
    env and the policy produced at that step."""
    from flexgpu.policy import DevicePolicy, DeviceRollout, TRANSITION_FIELDS
    from flexgpu.predictor import DeviceReplayBuffer
    env = small_env
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda, seed=9)
    R = 200
    buf = DeviceReplayBuffer(3 * R + 50, TRANSITION_FIELDS, device=cuda)
    ro = DeviceRollout(env, pol, replay=buf, record_envs=R)
    ro.reset()
    steps = []
    for t in range(4):                                          # the fourth step wraps the FIFO
        pre = ro.ring.dense().clone()
        last_hid = ro.hidden()
        reward, done = ro.step()
        steps.append(dict(state=pre[:R].reshape(R, -1), next_state=ro.ring.dense()[:R].reshape(R, -1).clone(),
                          last_hid=last_hid[:R].reshape(R, -1), hid=ro.hidden()[:R].reshape(R, -1),
                          action=pol._bufs["action"][:R].reshape(R, -1).clone(), log_prob_a=pol._bufs["logp"][:R].reshape(R, -1).clone(),
                          reward=reward[:R, None].float().repeat(1, 5).clone(), done=done[:R, None].float().clone()))
    assert len(buf) == 3 * R + 50
    got = buf.get_batch(3 * R + 50, start=0)                    # oldest first: the last 50 rows of step 0, then steps 1..3
    want = {k: torch.cat([steps[0][k][R - 50:]] + [s[k] for s in steps[1:]]) for k in steps[0]}
    for k, w in want.items():
        assert torch.equal(got[k], w), k
    assert torch.equal(got["last_step"], got["done"]) and bool((got["action_avail"] == 1).all())
    assert bool((got["value"] == 0).all()) and bool((got["next_value"] == 0).all())
    # the hidden state is carried: last_hid of step t + 1 is hid of step t
    assert torch.equal(steps[2]["last_hid"], steps[1]["hid"])
    pol.close(); buf.close()


def test_rollout_episode_boundary_resets_hidden_state(gold, cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv
    from flexgpu.policy import DevicePolicy, DeviceRollout
    env = BatchedFlexProvisionEnv(None, n_envs=64, device=cuda, profiles=profiles, seed=4)
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda, seed=2)
    ro = DeviceRollout(env, pol)
    ro.reset()
    for t in range(95):
        reward, done = ro.step()
    assert bool(done.all()) and ro.t == 0 and ro._reset_mask is not None       # 95 steps: every env terminated and was reset
    assert int(env.steps.min()) == 1 and int(env.steps.max()) == 1
    # the first action of the new episode comes from a zero hidden state
    ring = ro.ring
    _, _, _, mean_z = pol.act(ring, hid_in=None, explore=False, want_mean=True, hid_out=torch.empty(64, 5, 64, device=cuda))
    mean_z = mean_z.cpu().numpy().copy()
    _, _, _, mean_r = pol.act(ring, hid_in=ro._hid[ro._cur], reset=ro._reset_mask, explore=False, want_mean=True,
                              hid_out=torch.empty_like(ro._hid[ro._cur]), hid_layout="env_minor")
    assert np.array_equal(mean_z, mean_r.cpu().numpy())
    stats = env.episode_stats()
    assert float(stats["env_steps"]) == 64 * 95 and float(stats["episodes"]) == 64
    pol.close(); env.close()


def test_learner_batch_matches_reference_unpack_data(gold, cuda):
    """TransReplayBuffer(64) fed 80 transitions, get_batch(32) with the reference's np.random draw, Model.unpack_data
    and the critic input MADDPG.value builds -- against DeviceReplayBuffer + learner_batch on the same transitions."""
    from flexgpu.policy import DevicePolicy, TRANSITION_FIELDS, learner_batch
    from flexgpu.predictor import DeviceReplayBuffer
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda)
    buf = DeviceReplayBuffer(64, TRANSITION_FIELDS, device=cuda)
    n_tr = gold["tr_state"].shape[0]
    for lo in range(0, n_tr, 7):                                 # add_experience in uneven chunks
        hi = min(n_tr, lo + 7)
        buf.add_experience({k: torch.from_numpy(gold["tr_" + k][lo:hi]).to(cuda) for k in TRANSITION_FIELDS})
    assert len(buf) == 64
    out = learner_batch(pol, buf, 32, start=int(gold["batch_start"]))
    for k in ("state", "action", "log_prob_a", "value", "next_value", "next_state", "done", "last_step", "action_avail", "last_hid", "hid"):
        want = gold["up_" + k]
        assert tuple(out[k].shape) == want.shape, k
        assert np.array_equal(out[k].cpu().numpy(), want.astype(np.float32)), k
    assert np.array_equal(out["log_prob_a"].cpu().numpy(), gold["up_action"])            # the reference's quirk (model.py:313)
    assert np.max(np.abs(out["reward"].cpu().numpy() - gold["up_reward"])) < 1e-5        # BatchNorm1d over the batch
    assert tuple(out["critic_in"].shape) == gold["critic_in"].shape == (160, 745)
    assert np.array_equal(out["critic_in"].cpu().numpy(), gold["critic_in"])
    raw = learner_batch(pol, buf, 32, start=int(gold["batch_start"]), reward_normalisation=False, critic_input=False)
    assert "critic_in" not in raw and float(raw["reward"].abs().max()) > 0
    pol.close(); buf.close()


@pytest.mark.parametrize("critic", ["torch", "native"])
def test_rollout_matches_reference_train_process(cuda, critic):
    """End to end against the reference's own loop: tests/golden/ref_rollout.npz holds the 8 Transitions that
    Model.train_process (madrl/models/model.py:198-267) wrote into a TransReplayBuffer -- reference env (on the Pyomo
    stand-in), reference MADDPG / RNNAgent / select_action, the recorded exploration draws.  The device loop (tcgen05
    policy -> fused translate_action + step + get_obs) from the same start row, E0, reset actions, weights and draws
    must write the same Transition fields.  Tolerances: the policy differs from torch fp32 by ~1e-6 (fp32 arithmetic in a
    different order), which the env turns into ~1e-7 relative on setpoints and rewards; observations are fp32 here
    and fp64 -> fp32 in the reference (prep_obs).  value / next_value: the reference's own MLPCritic weights, either as a
    torch module on the library's critic-input rows (2e-5) or through k_critic (critic="native": fc1 / fc2 held as TF32,
    a weight perturbation of 2^-12 on 745-term rows: bound 1e-3, observed ~1e-4)."""
    from flexgpu import BatchedFlexProvisionEnv, Profiles
    from flexgpu.policy import DevicePolicy, DeviceRollout, TRANSITION_FIELDS
    from flexgpu.predictor import DeviceReplayBuffer
    g = np.load(os.path.join(os.path.dirname(GOLD), "ref_rollout.npz"))
    T = g["tr_reward"].shape[0]
    env = BatchedFlexProvisionEnv(None, n_envs=1, device=cuda, profiles=Profiles(g["P"], g["Q"], g["PV"], g["price"]))
    pol = DevicePolicy({k: g["w_" + k] for k in KEYS}, device=cuda, std=1.0)
    buf = DeviceReplayBuffer(64, TRANSITION_FIELDS, device=cuda)
    # the critic (madrl/critics/mlp_critic.py::MLPCritic, as MADDPG.value feeds it, maddpg.py:29-76) in plain torch on the
    # library's critic-input rows: fills the Transition's value / next_value like model.py:217, :225-226
    from flexgpu.policy import critic_input
    wc = {k[3:]: torch.from_numpy(g[k]).to(cuda) for k in g.files if k.startswith("wc_")}
    F = torch.nn.functional

    def value_fn(obs, act):
        x = F.linear(critic_input(pol, obs, act), wc["fc1.weight"], wc["fc1.bias"])
        x = torch.relu(F.layer_norm(x, (64,), wc["layernorm.weight"], wc["layernorm.bias"], 1e-5))
        h = torch.relu(F.linear(x, wc["fc2.weight"], wc["fc2.bias"]))
        return F.linear(h, wc["fc3.weight"], wc["fc3.bias"]).view(obs.shape[0], 5, 1)
    prev_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    if critic == "native":
        pol.load_critic({k[3:]: g[k] for k in g.files if k.startswith("wc_")})
    ro = DeviceRollout(env, pol, replay=buf, max_steps=T, value_fn="native" if critic == "native" else value_fn)
    env.reset([0], g["e0"][None], g["a0"][None], return_obs=False)          # trainer.env.reset() (model.py:208) with the reference's draws
    assert np.max(np.abs(env.voltages[0].cpu().numpy() - g["V0"])) < 1e-8
    env._check(env._lib.fp_obs_ring_reset_push(env._h, None, None), "fp_obs_ring_reset_push")    # the get_obs inside reset() (:155)
    ro.ring = env.obs_ring(); ro.t = 0
    ro._hid[ro._cur].zero_()
    rewards = []
    for t in range(T):
        reward, done = ro.step(eps=torch.from_numpy(g["eps"][2 * t][None].astype(np.float32)),
                               eps_next=torch.from_numpy(g["eps"][2 * t + 1][None].astype(np.float32)))   # draw 2t + 1: the next-value action
        rewards.append(float(reward[0]))
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in buf.get_batch(T, start=0).items()}
    torch.backends.cuda.matmul.allow_tf32 = prev_tf32
    tol = dict(state=2e-6, next_state=2e-6, action=5e-6, log_prob_a=2e-4, reward=None, done=0, last_step=0, action_avail=0,
               last_hid=5e-6, hid=5e-6, value=2e-5 if critic == "torch" else 1e-3, next_value=2e-5 if critic == "torch" else 1e-3)
    for k, bound in tol.items():
        want = g["tr_" + k]
        assert got[k].shape == want.shape, k
        if bound is None:
            assert np.max(np.abs(got[k] - want) / np.abs(want)) < 1e-5, (k, got[k][:, 0], want[:, 0])     # fp32 field of an fp64 reward
        else:
            assert np.max(np.abs(got[k] - want)) <= bound, (k, float(np.max(np.abs(got[k] - want))))
    assert np.max(np.abs(np.array(rewards) - g["tr_reward"][:, 0]) / np.abs(g["tr_reward"][:, 0])) < 1e-6        # the fp64 reward itself
    assert got["last_step"][-1, 0] == 1.0 and got["done"][-1, 0] == 0.0           # done_ = t == max_steps - 1 (model.py:229)
    # the reference's statistic counts the reward TWICE: info carries a 'reward' key (:697) that lands in the same
    # 'mean_train_reward' slot as the step's reward (model.py:247-252), then the sum is divided by t + 1 (:261-264)
    assert abs(2.0 * np.sum(rewards) / T - float(g["mean_train_reward"])) < 1e-6 * abs(float(g["mean_train_reward"]))
    pol.close(); buf.close(); env.close()


def test_rollout_resets_early_terminations_each_step(gold, cuda, profiles):
    """An env whose power flow fails terminates there (:314-337): the reference ends its episode and starts a new one with a
    zero hidden state.  The device loop does the same with a masked reset after the step (no host round trip)."""
    from flexgpu import BatchedFlexProvisionEnv
    from flexgpu.policy import DevicePolicy, DeviceRollout, TRANSITION_FIELDS
    from flexgpu.predictor import DeviceReplayBuffer
    n = 96
    env = BatchedFlexProvisionEnv(None, n_envs=n, device=cuda, profiles=profiles, seed=6)
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda, seed=5)
    buf = DeviceReplayBuffer(8 * n, TRANSITION_FIELDS, device=cuda)
    ro = DeviceRollout(env, pol, replay=buf, reset_done_each_step=True)
    ro.reset()
    for _ in range(3):
        ro.step()
    fail = torch.zeros(n, dtype=torch.uint8, device=cuda); fail[5] = 1; fail[40] = 1
    env.inject_failure(fail)
    reward, done = ro.step()                                     # step 4: envs 5 and 40 fail -> -200, terminated, reset
    env.inject_failure(None)
    assert done[5] and done[40] and int(done.sum()) == 2 and float(reward[5]) < -199.0
    steps = env.steps.cpu().numpy()
    assert steps[5] == 1 and steps[40] == 1 and (np.delete(steps, [5, 40]) == 5).all()
    hid_before = ro.hidden().clone()
    ro.step()                                                    # step 5 of the others, step 1 of the two new episodes
    got = buf.get_batch(n, start=len(buf) - n)                   # the transitions of that step
    lh = got["last_hid"].view(n, 5, 64)
    assert bool((lh[5] == 0).all()) and bool((lh[40] == 0).all())                     # they acted from init_hidden
    keep = [i for i in range(n) if i not in (5, 40)]
    assert torch.equal(lh[keep], hid_before[keep])
    prev = buf.get_batch(n, start=len(buf) - 2 * n)              # the failing step's transitions: done and last_step set
    assert float(prev["done"][5]) == 1.0 and float(prev["last_step"][40]) == 1.0 and float(prev["done"][6]) == 0.0
    assert int(env.steps[5]) == 2 and int(env.steps[6]) == 6
    pol.close(); buf.close(); env.close()


@pytest.mark.parametrize("n", [300, 40, 1, 2 * 148 * 128 + 77])
def test_native_critic_matches_torch(cuda, n):
    """fp_critic_value (k_critic, tcgen05) against plain torch fp32 with the same TF32-rounded fc1 / fc2 matrices (the
    device holds them as TF32, activations keep fp32 accuracy; bound 2e-5, observed ~1e-6): the TMA path with a ragged last
    tile, the LDGSTS path of rings narrower than a tile, a single env, and several tiles per CTA (weight blocks cycling
    through their three buffers); three ring rotations."""
    from flexgpu.policy import DevicePolicy
    rng = np.random.default_rng(11)
    sd = {"fc1.weight": rng.normal(0, 0.05, (64, 745)), "fc1.bias": rng.uniform(-0.04, 0.04, 64), "layernorm.weight": 1 + rng.normal(0, 0.1, 64),
          "layernorm.bias": rng.normal(0, 0.1, 64), "fc2.weight": rng.uniform(-0.125, 0.125, (64, 64)), "fc2.bias": rng.uniform(-0.125, 0.125, 64),
          "fc3.weight": rng.uniform(-0.125, 0.125, (1, 64)), "fc3.bias": rng.uniform(-0.125, 0.125, 1)}
    sd = {k: v.astype(np.float32) for k, v in sd.items()}
    pol = DevicePolicy(None, device=cuda)
    pol.load_critic(sd)
    w = torch_mats(sd, cuda, critic=True)
    g = torch.Generator(device=cuda).manual_seed(3)
    for slot in (0, 9, 23):
        obs = torch.rand(n, 5, 144, device=cuda, generator=g) * 2 - 0.5
        act = torch.tanh(torch.randn(n, 5, 4, device=cuda, generator=g))
        got = pol.value(ring_from_windows(obs, slot), act, slot=slot, n_envs=n).clone()
        want = mlp_critic_torch(w, obs, act)
        err = float((got - want).abs().max())
        assert got.shape == (n, 5, 1) and err < 2e-5, (slot, err)
    pol.close()
