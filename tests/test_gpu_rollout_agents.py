"""The device rollout at one to four agents: k_policy, k_sample, k_critic, the Transition writers and the learner feed of
a DevicePolicy built for n_agents = na, every row against the fp64 references and within the error model of
tests/_rollout_ref.py, DeviceRollout on the catalogue feeders of each agent count, and the rejection of every agent-count
or history mismatch."""
import ctypes as C

import pytest
import torch

import _feeders as F
import _rollout_ref as R
from _env_check import feeder_profiles, make_env

pytestmark = pytest.mark.gpu
AGENTS = [1, 2, 3, 4]


def _policy(na, seed=21, **kw):
    from flexgpu.policy import DevicePolicy
    sd = R.realistic_policy(seed + na, na)
    return DevicePolicy(sd, device="cuda:0", std=1.0, seed=(5 << 32) + 77, **kw), sd


CONFIGS = [("rows", "none", 0), ("env_minor", "given", 11), ("rows", "reset", 23), ("env_minor", "reset", 5)]


@pytest.mark.parametrize("n", [77, 129, 3917, 131149])
@pytest.mark.parametrize("na", AGENTS)
def test_policy_every_row_against_fp64(cuda, na, n):
    """k_policy at na agents: both hidden layouts, a reset mask, caller eps / Philox / test mode and three ring slots, every
    row within the per-element bound; n = 77 takes the LDGSTS path (n_pad < 128), the others the TMA path."""
    pol, sd = _policy(na)
    M = R.policy_mats(sd, cuda)
    step = (1 << 40) + 3
    n_pad = (n + 31) // 32 * 32
    wst = R.Worst(f"k_policy na={na} n={n}")
    for ci, (layout, hkind, slot) in enumerate(CONFIGS):
        ring, whole = R.random_ring(n, na, 100 * na + ci, cuda)
        hid_in, reset, h_ref = R.hidden_input(n, na, n_pad, hkind, layout, cuda, ci + n)
        eps = torch.randn(n, na, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(ci))
        outs = {mode: R.run_policy(pol, ring, slot, n, hid_in, reset, layout, mode, eps, step) for mode in ("eps", "philox", "test")}
        R.check_policy(wst, pol, M, ring, slot, n, h_ref, eps, step, outs, rms=n >= 3917)
        del whole
    wst.report()
    pol.close()


@pytest.mark.parametrize("na", AGENTS)
def test_sample_bit_identical_to_act(cuda, na):
    """fp_policy_sample on act's mean: act's own action and log-probability bit for bit (Philox, caller eps, test mode)."""
    pol, _ = _policy(na)
    n = 131149
    ring, _ = R.random_ring(n, na, 7, cuda)
    eps = torch.randn(n, na, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(4))
    for step in (0, (1 << 40) + 6):
        for explore, e in ((True, None), (True, eps), (False, None)):
            a1, lp1, _, m1 = pol.act(ring, slot=5, n_envs=n, explore=explore, eps=e, step=step, want_mean=True,
                                     hid_out=torch.empty(n, na, 64, device=cuda))
            a1, lp1, m1 = a1.clone(), lp1.clone(), m1.clone()
            a2, lp2 = pol.sample(m1, explore=explore, eps=e, step=step)
            assert torch.equal(a1, a2) and torch.equal(lp1, lp2), (step, explore, e is None)
    pol.close()


@pytest.mark.parametrize("n", [77, 131072, 131149])
@pytest.mark.parametrize("na", AGENTS)
def test_critic_every_row_against_fp64(cuda, na, n):
    """k_critic at na agents, every row within the bound with kappa = 1 + 2 (18 na + 3) / 4 for fc1; outputs past n keep
    their sentinels."""
    from flexgpu.policy import DevicePolicy
    sd = R.realistic_critic(5 + na, na)
    M = R.critic_mats(sd, cuda)
    pol = DevicePolicy(None, device=cuda, n_agents=na)
    pol.load_critic(sd)
    act = torch.tanh(torch.randn(n, na, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(n)))
    wst = R.Worst(f"k_critic na={na} n={n}")
    for slot in (0, 11, 23):
        ring, whole = R.random_ring(n, na, 7 + slot, cuda)
        R.critic_rows(wst, pol, M, ring, slot, n, act, f"[slot {slot}]", rms=n > 77)
        del whole
    wst.report()
    pol.close()


# ------------------------------------------------------------------------------------------------ DeviceRollout on feeders
ROLLOUT_CASES = [("two_bus", "thread"), ("slack_star", "thread"), ("custom14", "thread"), ("ieee33_4agents", "thread"),
                 ("custom14", "warp")]


def _feeder_env(cuda, name, variant, n, seed=1, **extra):
    net = F.feeder(name)
    return make_env(cuda, feeder_profiles(net), n, variant, net=net, seed=seed, **extra)


@pytest.mark.parametrize("value_kind", ["native", "torch"])
@pytest.mark.parametrize("name,variant", ROLLOUT_CASES)
def test_rollout_on_feeders(cuda, name, variant, value_kind):
    """DeviceRollout on a feeder of na agents with a replay ring: every recorded Transition field equals its source, the
    actions a torch fp32 RNNAgent with obs + na inputs, value / next_value a torch MLPCritic, and each step's reward and
    done those of a twin env stepped with the same actions -- across an episode boundary and one early termination."""
    from flexgpu.policy import DeviceRollout, transition_fields
    from flexgpu.predictor import DeviceReplayBuffer
    n = 200
    env, twin = _feeder_env(cuda, name, variant, n), _feeder_env(cuda, name, variant, n)
    na = env.n_agents
    pol, sd = _policy(na, seed=40)
    csd = R.realistic_critic(50 + na, na)
    pol.load_critic(csd)
    wp, wc = R.torch_mats(sd, cuda), R.torch_mats(csd, cuda, critic=True)
    fields = transition_fields(na)
    assert fields["state"] == 144 * na and fields["hid"] == 64 * na
    buf = DeviceReplayBuffer(8 * n, fields, device=cuda)
    value_fn = "native" if value_kind == "native" else (lambda o, a: R.mlp_critic_torch(wc, o, a))
    ro = DeviceRollout(env, pol, replay=buf, max_steps=3, reset_done_each_step=True, value_fn=value_fn)
    ro.reset()
    twin.reset()
    captured = {}
    orig_step = env.step

    def spy(*a, **kw):
        out = orig_step(*a, **kw)
        captured["ring"], captured["slot"], captured["action"] = out[3].ring.clone(), out[3].slot, a[0].clone()
        return out
    env.step = spy
    head, boundary, restarts = 0, False, 0
    try:
        for t in range(6):
            fail = torch.zeros(n, dtype=torch.uint8, device=cuda)
            if t == 1:
                fail[7::29] = 1
            env.inject_failure(fail); twin.inject_failure(fail)
            pre_ring, pre_slot = ro.ring.ring.clone(), ro.ring.slot
            last_hid = ro.hidden().clone()
            reset = None if ro._reset_mask is None else ro._reset_mask.bool().clone()
            if reset is not None:
                last_hid[reset] = 0
                restarts += int(reset.sum())
            explore = t % 2 == 1
            reward, done = ro.step(explore=explore)
            torch.cuda.synchronize()
            action = captured["action"].view(n, na, 4)
            # the twin env: same actions, same resets
            r2, d2, _ = twin.step(action, translate=True)
            assert torch.equal(reward, r2) and torch.equal(done, d2), t
            if ro.t == 0:
                boundary = True
                twin.reset(mask=ro._reset_mask)
            elif ro._reset_mask is not None:
                twin.reset(mask=ro._reset_mask, retries=0)
            # Transition fields against their sources
            got = buf.get_batch(n, start=head)
            head += n
            pre_obs = R.windows(pre_ring, pre_slot, 0, n)
            post_obs = R.windows(captured["ring"], captured["slot"], 0, n)
            last_step = torch.ones_like(done) if ro.t == 0 else done         # every env at the max_steps boundary
            want = {"state": pre_obs.reshape(n, -1), "next_state": post_obs.reshape(n, -1), "action": action.reshape(n, -1),
                    "log_prob_a": pol._bufs["logp"].reshape(n, -1), "last_hid": last_hid.reshape(n, -1),
                    "hid": ro._hid[ro._cur][:, :, :n].permute(2, 0, 1).reshape(n, -1),
                    "reward": reward[:, None].float().repeat(1, na), "done": done[:, None].float(),
                    "last_step": last_step[:, None].float(), "action_avail": torch.ones(n, na * 4, device=cuda)}
            assert torch.equal(action, pol._bufs["action"])
            if t == 1:
                assert int(done.sum()) == len(range(7, n, 29)), "the injected failures end their episodes"
            for k, w in want.items():
                assert torch.equal(got[k], w), (t, k)
            # hid: the policy's new hidden state, from last_hid by the torch RNNAgent
            m_t, h_t = R.rnn_agent_torch(wp, pre_obs, last_hid)
            assert float((got["hid"].view(n, na, 64) - h_t).abs().max()) < 5e-5, t
            if not explore:
                assert float((action - torch.tanh(m_t)).abs().max()) < 5e-5, t
            v_t = R.mlp_critic_torch(wc, pre_obs, action).view(n, na)
            assert float((got["value"] - v_t).abs().max()) < 2e-4, (t, "value")
            a2 = pol._bufs["action2"].view(n, na, 4)
            nv_t = R.mlp_critic_torch(wc, post_obs, a2).view(n, na)
            assert float((got["next_value"] - nv_t).abs().max()) < 2e-4, (t, "next_value")
            env.inject_failure(None); twin.inject_failure(None)
    finally:
        env.step = orig_step
    assert boundary and restarts > 0
    assert tuple(ro.hidden().shape) == (n, na, 64)
    pol.close(); buf.close(); env.close(); twin.close()


# ------------------------------------------------------------------------------------------------ learner feed
@pytest.mark.parametrize("na", AGENTS + [5])
def test_learner_batch(cuda, na):
    """learner_batch at na agents: critic_in bit for bit against torch.cat, reward_normalisation against BatchNorm1d(na)."""
    from flexgpu.policy import DevicePolicy, learner_batch, transition_fields
    from flexgpu.predictor import DeviceReplayBuffer
    pol = DevicePolicy(None, device=cuda, n_agents=na)
    fields = transition_fields(na)
    buf = DeviceReplayBuffer(300, fields, device=cuda)
    g = torch.Generator(device=cuda).manual_seed(na)
    buf.add_experience({k: torch.randn(300, w, device=cuda, generator=g) for k, w in fields.items()})
    B = 256
    out = learner_batch(pol, buf, B, start=10)
    raw = learner_batch(pol, buf, B, start=10, reward_normalisation=False, critic_input=False)
    assert torch.equal(out["critic_in"], R.critic_input_torch(raw["state"], raw["action"]))
    bn = torch.nn.BatchNorm1d(na).to(cuda).train()
    with torch.no_grad():
        want = bn(raw["reward"].view(B, na))
    assert float((out["reward"] - want).abs().max()) < 1e-5
    assert tuple(out["last_hid"].shape) == (B, na, 64) and tuple(out["value"].shape) == (B, na, 1)
    buf.close(); pol.close()


# ------------------------------------------------------------------------------------------------ rejections
def test_create_agents_rejects_out_of_range(cuda):
    from flexgpu import _lib
    from flexgpu.policy import DevicePolicy
    lib = _lib.lib()
    for na in (0, 6, -1):
        p = C.c_void_p()
        assert lib.fp_policy_create_agents(0, na, C.byref(p)) == -1          # FP_EINVAL
        assert b"n_agents" in lib.fp_policy_last_error(None)
        with pytest.raises(ValueError):
            DevicePolicy(None, device=cuda, n_agents=na)
    p = C.c_void_p()
    assert lib.fp_policy_create_agents(0, 3, C.byref(p)) == 0
    lib.fp_policy_destroy(p)


def test_five_agents_via_create_agents_equals_create(cuda):
    """fp_policy_create_agents(d, 5) and fp_policy_create give the same bits on the same inputs."""
    from flexgpu import _lib
    from flexgpu.policy import DevicePolicy
    sd = R.realistic_policy(3, 5)
    a = DevicePolicy(sd, device=cuda, seed=9)                               # fp_policy_create_agents(d, 5)
    b = DevicePolicy(sd, device=cuda, seed=9)
    lib = _lib.lib()
    lib.fp_policy_destroy(b._p)
    b._p = C.c_void_p()
    assert lib.fp_policy_create(0, C.byref(b._p)) == 0
    b.load_state_dict(sd)
    n = 3000
    ring, _ = R.random_ring(n, 5, 1, cuda)
    ra = [v.clone() for v in a.act(ring, slot=4, n_envs=n, step=2, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))]
    rb = [v.clone() for v in b.act(ring, slot=4, n_envs=n, step=2, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))]
    for x, y in zip(ra, rb):
        assert torch.equal(x, y)
    a.close(); b.close()


def test_mismatches_raise(cuda):
    from flexgpu.policy import DevicePolicy, DeviceRollout, TRANSITION_FIELDS, transition_fields
    from flexgpu.predictor import DeviceReplayBuffer
    env4 = _feeder_env(cuda, "ieee33_4agents", "thread", 130)
    env3 = _feeder_env(cuda, "custom14", "thread", 130)
    pol5, _ = _policy(5)
    pol4, sd4 = _policy(4)
    pol3, _ = _policy(3)
    # 5-agent policy on a 4-agent env / ring, and the reverse
    with pytest.raises(ValueError, match="agents"):
        DeviceRollout(env4, pol5)
    ring4 = env4.reset(return_obs="ring")
    for fn in (lambda: pol5.act(ring4), lambda: pol5.act(ring4.ring, slot=ring4.slot, n_envs=130),
               lambda: pol5.value(ring4, torch.zeros(130, 5, 4, device=cuda)),
               lambda: pol5.gather_windows(ring4, 130, torch.empty(130, 720, device=cuda), 720)):
        with pytest.raises(ValueError, match="ring"):
            fn()
    ring5 = torch.zeros(24, 5, 6, 160, device=cuda)
    with pytest.raises(ValueError, match="ring"):
        pol4.act(ring5, slot=0, n_envs=130)
    # hidden and action tensors of the wrong agent count
    with pytest.raises(ValueError, match="hidden"):
        pol4.act(ring4, hid_in=torch.zeros(130, 5, 64, device=cuda))
    with pytest.raises(ValueError, match="hidden"):
        pol4.act(ring4, hid_layout="env_minor", hid_out=torch.zeros(5, 64, ring4.ring.shape[-1], device=cuda))
    with pytest.raises(ValueError, match="mean"):
        pol4.sample(torch.zeros(130, 5, 4, device=cuda))
    # state dicts: a conflicting n_agents, and mismatched critic / policy widths
    with pytest.raises(ValueError, match="conflicts"):
        DevicePolicy(sd4, device=cuda, n_agents=5)
    with pytest.raises(ValueError, match=r"\(64, 148\)"):
        pol4.load_state_dict(R.realistic_policy(1, 5))
    with pytest.raises(ValueError, match=r"\(64, 596\)"):
        pol4.load_critic(R.realistic_critic(1, 5))
    # a replay buffer of 5-agent fields under a 3-agent rollout
    buf5 = DeviceReplayBuffer(400, TRANSITION_FIELDS, device=cuda)
    with pytest.raises(ValueError, match="transition_fields"):
        DeviceRollout(env3, pol3, replay=buf5)
    buf3 = DeviceReplayBuffer(400, transition_fields(3), device=cuda)
    DeviceRollout(env3, pol3, replay=buf3)                                 # the matching one is accepted
    # history 12
    env12 = _feeder_env(cuda, "custom14", "thread", 130, history=12)
    with pytest.raises(ValueError, match="history"):
        DeviceRollout(env12, pol3)
    for x in (pol5, pol4, pol3, buf5, buf3, env4, env3, env12):
        x.close()
