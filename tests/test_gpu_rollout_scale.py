"""The device rollout's kernels at rollout scale (five agents, up to 2^20 envs), every row: k_policy, k_sample and
k_critic against the fp64 references of tests/_rollout_ref.py within its per-element error model, the Philox exploration
draws against its numpy port, the Transition writers bit for bit, and the LayerNorm's invariance to a common offset of its
input.  The rings carry the golden observation windows.  Each test prints max(err / bound) per quantity and size."""
import numpy as np
import pytest
import torch
from _golden import load_ref_policy
from _rollout_ref import (C_TANH, CHUNK, KAPPA_FC1, KEYS, SENT, U, Worst, action_bound, check_policy, critic_mats,
                          critic_reference, critic_rows, hidden_input, layernorm_bound, logp_bound, philox_normals,
                          policy_mats, policy_reference, realistic_critic, realistic_policy, run_policy, ulp, windows)

pytestmark = pytest.mark.gpu
BIG = 131072


def make_ring(n, slot_seed, cuda, obs_src):
    """[24, 5, 6, n_pad] ring from the golden observation windows: env e carries window e % n_src times (1 + 0.05 N(0, 1)),
    so rows differ; columns past n are zeros, as the env leaves them."""
    n_pad = (n + 31) // 32 * 32
    src = torch.from_numpy(np.ascontiguousarray(obs_src, dtype=np.float32)).to(cuda)           # [n_src, 5, 144]
    g = torch.Generator(device=cuda).manual_seed(slot_seed)
    ring = torch.zeros(24, 5, 6, n_pad, device=cuda)
    for e0 in range(0, n, CHUNK):
        e1 = min(n, e0 + CHUNK)
        idx = torch.arange(e0, e1, device=cuda) % src.shape[0]
        w = src[idx] * (1 + 0.05 * torch.randn(e1 - e0, 5, 144, device=cuda, generator=g))
        ring[:, :, :, e0:e1] = w.view(e1 - e0, 5, 24, 6).permute(2, 1, 3, 0)      # slot order = window order; rotated below
    return ring


def rotate(ring, slot):
    """A ring whose window order is its slot order, re-laid so that its newest entry sits in `slot`."""
    idx = torch.tensor([(r - slot - 1) % 24 for r in range(24)], device=ring.device)
    return ring[idx].contiguous()


# ------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def gold():
    return load_ref_policy()


@pytest.fixture(scope="module")
def policies(gold, cuda):
    from flexgpu.policy import DevicePolicy
    sds = {"real": realistic_policy(21, 5), "gold": {k: np.asarray(gold["wt_" + k], dtype=np.float32) for k in KEYS}}
    pols = {k: (DevicePolicy(sd, device=cuda, std=1.0, seed=(5 << 32) + 77), policy_mats(sd, cuda)) for k, sd in sds.items()}
    yield pols
    for p, _ in pols.values():
        p.close()


# ------------------------------------------------------------------------------------------------ k_policy, every row
# per size, configurations that together cover both hidden layouts, the three hidden inputs, slots 0 / 11 / 23 and both
# weight sets; each runs explore with caller eps, explore with Philox and test mode
CONFIGS = [("rows", "none", 0, "real"), ("env_minor", "given", 11, "gold"), ("rows", "reset", 23, "gold"),
           ("env_minor", "reset", 0, "real"), ("rows", "given", 11, "real")]
SIZES = [129, 3840, BIG, BIG + 77, 1 << 20]


@pytest.mark.parametrize("n", SIZES)
def test_policy_every_row_against_fp64(policies, gold, cuda, n):
    step = (1 << 40) + 3
    n_pad = (n + 31) // 32 * 32
    base = make_ring(n, n, cuda, gold["obs0"])
    wst = Worst(f"k_policy n={n}")
    configs = CONFIGS if n < (1 << 20) else CONFIGS[:3]
    for ci, (layout, hkind, slot, wname) in enumerate(configs):
        pol, M = policies[wname]
        ring = rotate(base, slot)
        hid_in, reset, h_ref = hidden_input(n, 5, n_pad, hkind, layout, cuda, ci + n)
        eps = torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(ci))
        outs = {mode: run_policy(pol, ring, slot, n, hid_in, reset, layout, mode, eps, step) for mode in ("eps", "philox", "test")}
        check_policy(wst, pol, M, ring, slot, n, h_ref, eps, step, outs, rms=True)
        # the log-probability formula alone, at the kernel's own fp32 a and x (caller eps), on the first chunk
        e1 = min(n, CHUNK)
        mk = outs["eps"][3][:e1].double()
        xk = (mk + eps[:e1].double()).float().double()                # fma(1, z, m): exact sum, one rounding
        ak = outs["eps"][0][:e1].double()
        wk = 1 - ak * ak + 1e-6
        dw = 2.0 ** -23                                               # a^2, 1 - a^2, + 1e-6 in fp32
        gauss = 0.5 * (xk - mk) ** 2
        lp_self = -gauss - 0.5 * np.log(2 * np.pi) - torch.log(wk)
        logf = torch.where(wk >= 0.5, torch.full_like(wk, 2.0 ** -21.41), 3 * ulp(torch.log(wk)))
        bound = dw / (wk - dw).clamp(min=0.99e-6) + logf + (xk - mk).abs() * ulp(xk - mk) + 4 * U * (xk - mk) ** 2 + \
            ulp(lp_self) + ulp(gauss + 0.92) + 2 * U
        wst.check("logp_formula", outs["eps"][1][:e1], lp_self, bound)
    wst.report()


# ------------------------------------------------------------------------------------------------ Philox and k_sample
def test_sample_philox_against_port_and_bit_identical_to_act(policies, gold, cuda):
    """k_sample's Philox draws at 131 072 envs against the numpy port (seed >= 2^32; step 2^40 + t differs from step t: the
    counter's high step word is live), the 5.77-sigma truncation of the design, and fp_policy_sample on act's mean equal to
    act's action and logp bit for bit, with Philox and with eps, explore and test."""
    pol, M = policies["real"]
    n = BIG
    ring = rotate(make_ring(n, 3, cuda, gold["obs0"]), 5)
    eps = torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(4))
    wst = Worst("k_sample n=131072")
    rows = np.arange(n * 5, dtype=np.uint64)
    for t in (0, 6):
        step = (1 << 40) + t
        for explore, e in ((True, None), (True, eps), (False, None)):
            a1, lp1, _, m1 = pol.act(ring, slot=5, n_envs=n, explore=explore, eps=e, step=step, want_mean=True,
                                     hid_out=torch.empty(n, 5, 64, device=cuda))
            a1, lp1, m1 = a1.clone(), lp1.clone(), m1.clone()
            a2, lp2 = pol.sample(m1, explore=explore, eps=e, step=step)
            assert torch.equal(a1, a2) and torch.equal(lp1, lp2), (t, explore, e is None)
        m = m1.double()
        a_s, lp_s = [v.clone() for v in pol.sample(m1, explore=True, step=step)]
        zp, ezp = philox_normals(rows, pol.seed, step)
        z = torch.from_numpy(zp).to(cuda).view(n, 5, 4); ez = torch.from_numpy(ezp).to(cuda).view(n, 5, 4)
        a, e_a, x, _ = action_bound(m, torch.zeros_like(m), z, ez, pol.std, True)
        wst.check("action", a_s, a, e_a)
        lp, e_lp = logp_bound(a, e_a, z, ez, x, pol.std)
        wst.check("logp", lp_s, lp, e_lp)
        # the low-step draws are different numbers: dropping the counter's high word would make them equal
        z_low, _ = philox_normals(rows, pol.seed, t)
        assert np.mean(z_low == zp) < 1e-6
        a_low, _ = pol.sample(m1, explore=True, step=t)
        assert float((a_low != a_s).float().mean()) > 0.99
        # u0 in (0, 1]: |z| <= sqrt(-2 ln 2^-24) = 5.768 by construction (a 5.77-sigma truncation of the normals)
        zmax = np.sqrt(-2 * np.log(2.0 ** -24))
        assert np.abs(zp).max() <= zmax and np.abs(zp).max() > 4.5
        # from the kernel's own action: |x - m| = |atanh(a) - m| never exceeds the truncation (where a is not saturated)
        ok = a_s.abs() < 0.999
        zk = (torch.atanh(a_s.double()) - m)[ok]
        assert float(zk.abs().max()) <= zmax + 1e-3
    wst.report()


# ------------------------------------------------------------------------------------------------ k_critic, every row
@pytest.fixture(scope="module")
def critic(cuda):
    from flexgpu.policy import DevicePolicy
    sd = realistic_critic(5, 5)
    pol = DevicePolicy(None, device=cuda)
    pol.load_critic(sd)
    yield pol, critic_mats(sd, cuda)
    pol.close()


@pytest.mark.parametrize("n", [BIG, BIG + 77, 1 << 20])
def test_critic_every_row_against_fp64(critic, gold, cuda, n):
    pol, M = critic
    base = make_ring(n, 7 + n, cuda, gold["obs1"])
    act = torch.tanh(torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(n)))
    wst = Worst(f"k_critic n={n}")
    for slot in (0, 11, 23):
        critic_rows(wst, pol, M, rotate(base, slot), slot, n, act, f"[slot {slot}]", rms=True)
    if n == BIG:                                        # DeviceRollout's native-value call: record_envs < n_pad, TMA path
        critic_rows(wst, pol, M, rotate(base, 11), 11, 40000, act, "[n_envs 40000]", rms=True)
    wst.report()


# ------------------------------------------------------------------------------------------------ LayerNorm offset invariance
OFFSETS = (0.0, 1.0, 4.0, 16.0, 64.0)


def probe_policy(gold, C):
    """The golden fc1 / LayerNorm with fc1.bias + C, under a GRU that exposes the LayerNorm: W_ih's n block = I, every other
    gate weight 0, the z bias -40 (z = sigmoid(-20) after the kernel's clamp, 2e-9), so h' = tanh(relu(LN(v))) per unit."""
    sd = {k: np.asarray(gold["wt_" + k], dtype=np.float32).copy() for k in KEYS}
    sd["fc1.bias"] = (sd["fc1.bias"] + np.float32(C)).astype(np.float32)
    sd["rnn.weight_ih"] = np.zeros((192, 64), np.float32); sd["rnn.weight_ih"][128:] = np.eye(64, dtype=np.float32)
    sd["rnn.weight_hh"] = np.zeros((192, 64), np.float32)
    sd["rnn.bias_ih"] = np.zeros(192, np.float32); sd["rnn.bias_ih"][64:128] = -40.0
    sd["rnn.bias_hh"] = np.zeros(192, np.float32)
    return sd


def test_layernorm_offset_invariance_policy(gold, cuda):
    """fc1.bias + C leaves the network unchanged.  (a) mean and hid of the golden network against the C = 0 fp64 reference,
    inside the error model evaluated at the shifted pre-activation (the offset enters through ulp(v) and the sums' rounding:
    linear in C).  (b) The sharp check: the fc1 accumulator is bit-identical for every C (the bias is added after the MMA),
    so on the probe network the difference of the C and C = 0 runs is the LayerNorm's alone: per unit at most the sum of
    both runs' LayerNorm bounds with exact inputs (e1 = ulp(v)), times tanh', plus both runs' rounding after it."""
    from flexgpu.policy import DevicePolicy
    n = BIG
    slot = 11
    ring = rotate(make_ring(n, 19, cuda, gold["obs0"]), slot)
    h_in = 0.9 * (2 * torch.rand(n, 5, 64, device=cuda, generator=torch.Generator(device=cuda).manual_seed(2)) - 1)
    wst = Worst("LayerNorm offset, k_policy n=131072")
    ref0 = policy_mats({k: np.asarray(gold["wt_" + k], dtype=np.float32) for k in KEYS}, cuda)
    probe = {}
    for C in OFFSETS:
        sd = {k: np.asarray(gold["wt_" + k], dtype=np.float32).copy() for k in KEYS}
        sd["fc1.bias"] = (sd["fc1.bias"] + np.float32(C)).astype(np.float32)
        pol = DevicePolicy(sd, device=cuda)
        _, _, hid, mean = pol.act(ring, slot=slot, n_envs=n, hid_in=h_in, explore=False, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))
        MC = policy_mats(sd, cuda)
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            obs = windows(ring, slot, e0, e1)
            m0, _, h0, _ = policy_reference(ref0, obs, h_in[e0:e1].double())
            mc, e_m, hc, e_h = policy_reference(MC, obs, h_in[e0:e1].double())          # the model at the shifted v
            # + what the fp32 folding of fc1.bias + C + one-hot column changes exactly (the pre-activation's representation)
            wst.check("mean", mean[e0:e1], m0, e_m + (mc - m0).abs(), f"[C={C:g}]")
            wst.check("hid", hid[e0:e1], h0, e_h + (hc - h0).abs(), f"[C={C:g}]")
        pol.load_state_dict(probe_policy(gold, C))
        _, _, hp, _ = pol.act(ring, slot=slot, n_envs=n, hid_in=None, explore=False, hid_out=torch.empty(n, 5, 64, device=cuda))
        probe[C] = (hp.clone(), MC["b1a"])
        pol.close()

    def probe_ref(acc, b1a, e_acc=0.0):               # tanh(relu(LN(acc + b1a))) with input error e_acc + ulp(v), and its bound
        v = acc + b1a[None]
        y, e_y = layernorm_bound(v, e_acc + ulp(v), ref0["g"], ref0["b"])
        n_ = torch.tanh(torch.relu(y))
        return n_, (1 - n_ * n_ + e_y).clamp(max=1) * (e_y + 2.0 ** -20 * y.abs()) + C_TANH + 2.0 ** -22 * y.abs() + 3e-9 + ulp(n_)
    for C in OFFSETS[1:]:
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            x = windows(ring, slot, e0, e1).double()
            acc = x @ ref0["W1"].T
            (r0, b0), (rc, bc) = probe_ref(acc, probe[0.0][1]), probe_ref(acc, probe[C][1])
            wst.check("probe_hid_diff", probe[C][0][e0:e1].double() - probe[0.0][0][e0:e1].double(), rc - r0, b0 + bc, f"[C={C:g}]")
            if C == OFFSETS[1]:                         # the probe itself against fp64, fc1's error included
                r0f, b0f = probe_ref(acc, probe[0.0][1], KAPPA_FC1 * 2.0 ** -20 * (x.abs() @ ref0["W1"].abs().T))
                wst.check("probe_hid", probe[0.0][0][e0:e1], r0f, b0f, "[C=0]")
    wst.report()


def test_layernorm_offset_invariance_critic(gold, cuda):
    """As for the policy: the critic's fc1.bias + C against the C = 0 fp64 reference within the model, and on a probe
    critic (fc2 = I, fc2.bias = 0, fc3 = unit j) whose value is relu(LN(v))_j, the C run against the C = 0 run."""
    from flexgpu.policy import DevicePolicy
    n = BIG
    slot = 23
    ring = rotate(make_ring(n, 23, cuda, gold["obs1"]), slot)
    act = torch.tanh(torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(8)))
    sd0 = realistic_critic(9, 5)
    M0 = critic_mats(sd0, cuda)
    j = int(np.argmax(np.abs(sd0["layernorm.weight"])))
    wst = Worst("LayerNorm offset, k_critic n=131072")
    probe = {}
    pol = DevicePolicy(None, device=cuda)
    for C in OFFSETS:
        sd = {k: v.copy() for k, v in sd0.items()}
        sd["fc1.bias"] = (sd["fc1.bias"] + np.float32(C)).astype(np.float32)
        pol.load_critic(sd)
        val = pol.value(ring, act, slot=slot, n_envs=n).clone()
        MC = critic_mats(sd, cuda)
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            obs, ac = windows(ring, slot, e0, e1).reshape(e1 - e0, 720), act[e0:e1].reshape(e1 - e0, 20)
            v0, _ = critic_reference(M0, obs, ac)
            vc, e_v = critic_reference(MC, obs, ac)
            wst.check("value", val[e0:e1, :, 0], v0, e_v + (vc - v0).abs(), f"[C={C:g}]")
        sd["fc2.weight"] = np.eye(64, dtype=np.float32); sd["fc2.bias"] = np.zeros(64, np.float32)
        sd["fc3.weight"] = np.zeros((1, 64), np.float32); sd["fc3.weight"][0, j] = 1.0; sd["fc3.bias"] = np.zeros(1, np.float32)
        pol.load_critic(sd)
        probe[C] = (pol.value(ring, act, slot=slot, n_envs=n).clone()[:, :, 0], MC["b1a"])
    pol.close()

    def probe_ref(acc, b1a):                           # relu(LN(acc + b1a))_j with exact input and its bound
        v = acc + b1a[None]
        y, e_y = layernorm_bound(v, ulp(v), M0["g"], M0["b"])
        return torch.relu(y[..., j]), e_y[..., j] + 2.0 ** -20 * y[..., j].abs() + ulp(y[..., j])
    for C in OFFSETS[1:]:
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            obs, ac = windows(ring, slot, e0, e1).reshape(e1 - e0, 720).double(), act[e0:e1].reshape(e1 - e0, 20).double()
            acc = (obs @ M0["Wo"].T + ac @ M0["Wa"].T)[:, None, :]
            (r0, b0), (rc, bc) = probe_ref(acc, probe[0.0][1]), probe_ref(acc, probe[C][1])
            wst.check("probe_value_diff", probe[C][0][e0:e1].double() - probe[0.0][0][e0:e1].double(), rc - r0, b0 + bc, f"[C={C:g}]")
    wst.report()


# ------------------------------------------------------------------------------------------------ Transition writers
@pytest.fixture(scope="module")
def big_env(cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv
    e = BatchedFlexProvisionEnv(None, n_envs=BIG, device=cuda, profiles=profiles, seed=12)
    yield e
    e.close()


def dense_rows(ring, slot, n):
    return torch.cat([windows(ring, slot, e0, min(n, e0 + CHUNK)) for e0 in range(0, n, CHUNK)]).reshape(n, 720)


@pytest.mark.parametrize("record,variant", [(BIG, "plain"), (50000, "plain"), (50000, "native"), (BIG, "failures")])
def test_rollout_transition_writers_at_scale(big_env, gold, cuda, record, variant):
    """DeviceRollout on 131 072 envs: every field of every recorded row against plain torch indexing of the ring before and
    after the step, the hidden states and the step's outputs (bit for bit); the reserved window wraps in the middle of a
    128-env tile, and the replay rows outside it keep their sentinels."""
    from flexgpu.policy import DevicePolicy, DeviceRollout, TRANSITION_FIELDS
    from flexgpu.predictor import DeviceReplayBuffer
    env = big_env
    N = env.n_envs
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda, seed=(3 << 32) + 1)
    if variant == "native":
        pol.load_critic(realistic_critic(13, 5))
    cap = record + 500 if record == N else 60000
    pos0 = cap - ((record // 2) // 128 * 128 + 64)                       # the first step's window wraps 64 envs into a tile
    buf = DeviceReplayBuffer(cap, TRANSITION_FIELDS, device=cuda)
    buf.reserve(cap)
    for k, w in TRANSITION_FIELDS.items():
        buf.write(k, 0, torch.full((cap, w), SENT, device=cuda))
    buf.reserve(pos0)
    head = pos0
    ro = DeviceRollout(env, pol, replay=buf, record_envs=record, reset_done_each_step=variant == "failures",
                       value_fn="native" if variant == "native" else None)
    ro.reset()
    R = ro.R
    captured = {}
    orig_step = env.step

    def spy(*a, **kw):
        out = orig_step(*a, **kw)
        captured["ring"], captured["slot"] = out[3].ring.clone(), out[3].slot
        return out
    env.step = spy
    try:
        for t in range(2):
            if variant == "failures":
                fail = torch.zeros(N, dtype=torch.uint8, device=cuda)
                if t == 0:
                    fail[5::997] = 1
                env.inject_failure(fail)
            pre_ring, pre_slot = ro.ring.ring.clone(), ro.ring.slot
            last_hid = ro._hid[ro._cur][:, :, :N].permute(2, 0, 1).clone()
            reset = None if ro._reset_mask is None else ro._reset_mask.bool().clone()
            reward, done = ro.step()
            torch.cuda.synchronize()
            pos = head
            head = (head + R) % cap
            got = buf.get_batch(cap, start=0)                             # logical order: physical row p = (p - head) mod cap
            phys = {k: torch.roll(v, shifts=head, dims=0) for k, v in got.items()}
            rows = (pos + torch.arange(R, device=cuda)) % cap
            want = {"state": dense_rows(pre_ring, pre_slot, R), "next_state": dense_rows(captured["ring"], captured["slot"], R),
                    "hid": ro._hid[ro._cur][:, :, :R].permute(2, 0, 1).reshape(R, 320),
                    "action": pol._bufs["action"][:R].reshape(R, 20), "log_prob_a": pol._bufs["logp"][:R].reshape(R, 20),
                    "reward": reward[:R, None].float().repeat(1, 5), "done": done[:R, None].float(),
                    "last_step": done[:R, None].float(), "action_avail": torch.ones(R, 20, device=cuda)}
            lh = last_hid[:R].reshape(R, 320).clone()
            if reset is not None:
                lh[reset[:R]] = 0
                assert int(reset[:R].sum()) > 0
            want["last_hid"] = lh
            if variant == "native":
                want["value"] = pol._bufs["value"].view(R, 5); want["next_value"] = pol._bufs["next_value"].view(R, 5)
            else:
                want["value"] = want["next_value"] = torch.zeros(R, 5, device=cuda)
            for k, w in want.items():
                assert torch.equal(phys[k][rows], w), (t, k)
            outside = torch.ones(cap, dtype=torch.bool, device=cuda)
            outside[rows] = False
            if t == 0 and bool(outside.any()):
                for k in TRANSITION_FIELDS:
                    assert bool((phys[k][outside] == SENT).all()), ("row outside the window written", k)
            if variant == "failures":
                if t == 0:
                    assert int(done.sum()) == len(range(5, N, 997))
                else:                                              # the restarted envs acted from a zero hidden state
                    h_zero = pol.act(pre_ring, slot=pre_slot, n_envs=N, hid_in=None, explore=False,
                                     hid_out=torch.empty(N, 5, 64, device=cuda))[2]
                    assert torch.equal(want["hid"][reset[:R]], h_zero[:R][reset[:R]].reshape(-1, 320))
                env.inject_failure(None)
    finally:
        env.step = orig_step
        pol.close(); buf.close()

