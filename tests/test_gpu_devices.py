"""GPU, two devices in one process: the env, predictor, replay ring, policy and critic handles created on cuda:1 while
torch's current device is 0 compute, bit for bit, what the same seeded sequence computes on cuda:0, and no call leaves
torch's current device switched (include/flexgpu.h: a handle's work runs on its own device and the caller's current
device is unchanged on return)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def run_sequence(device, profiles, after_call):
    """One seeded sequence of calls on `device`; after_call() runs after each of them.  Returns every output on the host."""
    from flexgpu import BatchedFlexProvisionEnv
    from flexgpu.policy import _CRITIC_KEYS, _CRITIC_SHAPES, _WEIGHT_KEYS, _WEIGHT_SHAPES, DevicePolicy
    from flexgpu.predictor import DeviceReplayBuffer, VoltagePredictor

    g = torch.Generator().manual_seed(0)
    n = 300
    out = {}
    env = BatchedFlexProvisionEnv(None, n_envs=n, device=device, profiles=profiles, seed=4)
    after_call()
    env.reset(return_obs="ring")
    after_call()
    reward, done, _, ring = env.step(torch.rand(n, 5, 4, generator=g).to(device), return_obs="ring")
    after_call()
    out.update(reward0=reward.cpu(), done0=done.cpu(), obs0=ring.dense().cpu())
    after_call()
    env.set_obs_history(False)                       # ring-only steps: the fp64 history is rebuilt on the read below
    after_call()
    reward, done, _, ring = env.step(torch.rand(n, 5, 4, generator=g).to(device), return_obs="ring")
    after_call()
    out.update(reward1=reward.cpu(), done1=done.cpu())
    sd = env.state_dict()                            # fp_history_ptr's read path
    after_call()
    out.update(rec=sd["rec"], voltage=sd["voltage"], history=sd["history"])

    rng = np.random.default_rng(1)
    pred = VoltagePredictor(env, rng.normal(0, 0.05, (33, 66)), np.full(33, 1.0))
    after_call()
    buf = DeviceReplayBuffer(2 * n, {"v_pred": 33, "safety_penalty": 1, "x": 7}, device=device)
    after_call()
    vhat, pen = pred.predict(torch.rand(n, 66, generator=g).to(device), sink=buf)
    after_call()
    out.update(vhat=vhat.cpu(), penalty=pen.cpu())
    buf.add_experience({"x": torch.rand(n, 7, generator=g).to(device)})
    after_call()
    batch = buf.get_batch(2 * n, start=0)
    after_call()
    out.update({"replay_" + k: v.cpu() for k, v in batch.items()})

    pol = DevicePolicy({k: torch.randn(s, generator=g) * 0.1 for k, s in zip(_WEIGHT_KEYS, _WEIGHT_SHAPES)}, device=device, seed=5)
    after_call()
    pol.load_critic({k: torch.randn(s, generator=g) * 0.05 for k, s in zip(_CRITIC_KEYS, _CRITIC_SHAPES)})
    after_call()
    action, logp, hid, mean = pol.act(ring, want_mean=True, step=3)
    after_call()
    value = pol.value(ring, action)
    after_call()
    out.update(action=action.cpu(), logp=logp.cpu(), hid=hid.cpu(), mean=mean.cpu(), value=value.cpu())
    torch.cuda.synchronize(device)
    for h in (pol, buf, env):
        h.close()
        after_call()
    return out


def test_handles_on_a_second_device_match_the_first_and_keep_the_current_device(profiles):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible CUDA devices")
    torch.cuda.set_device(0)

    def current_device_is_0():
        assert torch.cuda.current_device() == 0

    ref = run_sequence(torch.device("cuda:0"), profiles, current_device_is_0)
    got = run_sequence(torch.device("cuda:1"), profiles, current_device_is_0)
    assert ref.keys() == got.keys()
    for k in ref:
        assert ref[k].dtype == got[k].dtype and ref[k].shape == got[k].shape, k
        assert ref[k].numpy().tobytes() == got[k].numpy().tobytes(), k
