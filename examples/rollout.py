"""Batched rollout in the shape of the reference's train_process (madrl/models/model.py:198-267), with the
four host<->device crossings per step removed: observations, actions, rewards and the transition sink stay
on the GPU; only the episode statistics leave it (one all-reduce when several ranks run).

    python examples/rollout.py --envs 65536 --steps 95
    python examples/rollout.py --buildings 5,10,15,20                      # IEEE-33 with four agents
    torchrun --nproc-per-node 8 examples/rollout.py --envs 1048576      # 2^20 envs sharded over 8 GPUs

The policy is the reference's shared-parameter RNNAgent (madrl/agents/rnn_agent.py) evaluated by the tcgen05 policy
kernel straight from the env's observation ring; pass --weights model.pt (a checkpoint written by train_agent.py:
{"model_state_dict": ...}, train_agent.py:144-147) or let the script initialise it like the reference does
(init_std 0.1).  With --record N the Transition fields (model.py:230-242) of the first N envs go into a device replay
ring, from which `learner_batch` hands the learner the unpack_data tensors; with --critic the Transition's value /
next_value are filled by the reference's MLPCritic on the tcgen05 critic kernel (MADDPG.value, model.py:217, :225-226).
"""
import argparse
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "safe-marl_b200")]
from flexgpu import BatchedFlexProvisionEnv, sharding  # noqa: E402


def reference_init(seed=0, n_agents=5):
    """RNNAgent weights as the reference initialises them: nn.Linear weights ~ N(0, init_std = 0.1) (model.py:185-190),
    everything else torch's defaults (uniform(-1/sqrt(fan), 1/sqrt(fan)); LayerNorm 1 / 0); fc1 takes 144 + n_agents inputs."""
    g = torch.Generator().manual_seed(seed)
    u = lambda shape, k: (torch.rand(shape, generator=g) * 2 - 1) * k
    k1 = 144 + n_agents
    return {"fc1.weight": torch.randn(64, k1, generator=g) * 0.1, "fc1.bias": u((64,), k1 ** -0.5),
            "layernorm.weight": torch.ones(64), "layernorm.bias": torch.zeros(64),
            "rnn.weight_ih": u((192, 64), 0.125), "rnn.weight_hh": u((192, 64), 0.125), "rnn.bias_ih": u((192,), 0.125),
            "rnn.bias_hh": u((192,), 0.125), "fc2.weight": torch.randn(4, 64, generator=g) * 0.1, "fc2.bias": u((4,), 0.125)}


def reference_critic_init(seed=1, n_agents=5):
    """MLPCritic weights (madrl/critics/mlp_critic.py, input n_agents x 149: 745 for five agents) initialised like
    reference_init."""
    g = torch.Generator().manual_seed(seed)
    u = lambda shape, k: (torch.rand(shape, generator=g) * 2 - 1) * k
    k1 = 149 * n_agents
    return {"fc1.weight": torch.randn(64, k1, generator=g) * 0.1, "fc1.bias": u((64,), k1 ** -0.5), "layernorm.weight": torch.ones(64),
            "layernorm.bias": torch.zeros(64), "fc2.weight": torch.randn(64, 64, generator=g) * 0.1, "fc2.bias": u((64,), 0.125),
            "fc3.weight": torch.randn(1, 64, generator=g) * 0.1, "fc3.bias": u((1,), 0.125)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536, help="total environments over all ranks")
    ap.add_argument("--steps", type=int, default=95)
    ap.add_argument("--weights", default=None, help="checkpoint with the policy's state_dict (policy_dicts.0.* keys)")
    ap.add_argument("--record", type=int, default=1024, help="envs per rank whose transitions go into the device replay ring")
    ap.add_argument("--critic", action="store_true", help="fill value / next_value with the critic kernel (value_dicts.0.* of --weights, or the reference's initialisation)")
    ap.add_argument("--buildings", default="5,10,15,20,25", help="IEEE-33 buses of the agents' buildings (one to five)")
    args = ap.parse_args()
    from flexgpu.policy import DevicePolicy, DeviceRollout, learner_batch, transition_fields
    from flexgpu.predictor import DeviceReplayBuffer
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", 1), ("RANK", 0), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    offset, count = sharding.shard(args.envs, rank, world)             # env index range of this rank
    buildings = [int(b) for b in args.buildings.split(",")]
    env_args = {"buildings": buildings, "pv_nodes": buildings, "ess_nodes": buildings}
    env = BatchedFlexProvisionEnv(env_args, n_envs=count, device=dev, seed=0, env_offset=offset)
    na = env.n_agents
    if args.weights:
        ckpt = torch.load(args.weights, map_location="cpu")
        ckpt = ckpt.get("model_state_dict", ckpt)
        sd = {k.split("policy_dicts.0.", 1)[1]: v for k, v in ckpt.items() if k.startswith("policy_dicts.0.")} or ckpt
        csd = {k.split("value_dicts.0.", 1)[1]: v for k, v in ckpt.items() if k.startswith("value_dicts.0.")} or reference_critic_init(n_agents=na)
    else:
        sd, csd = reference_init(n_agents=na), reference_critic_init(n_agents=na)
    policy = DevicePolicy(sd, device=dev, std=1.0, seed=1 + rank)      # fixed_policy_std 1.0 (default.yaml)
    if args.critic:
        policy.load_critic(csd)
    rec = min(args.record, count)
    replay = DeviceReplayBuffer(max(rec * 8, 5000), transition_fields(na), device=dev) if rec else None    # replay_buffer_size 5000
    rollout = DeviceRollout(env, policy, replay=replay, record_envs=rec, value_fn="native" if (args.critic and rec) else None)
    rollout.reset()                                                    # env.reset() + init_hidden (model.py:208-211)
    rollout.step()                                                     # warm-up: allocations, module load
    env.episode_stats(reset=True)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for t in range(args.steps):
        reward, done = rollout.step()                                  # policy -> translate_action + step + get_obs -> Transition
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    stats = env.episode_stats()                                        # the one collective (NCCL all-reduce of 16 doubles)
    if rank == 0:
        means = sharding.episode_means(stats)
        print(f"{args.envs} envs x {args.steps} steps on {world} GPU(s): {args.envs * args.steps / dt:.3e} env-steps/s "
              f"(tcgen05 policy + fused step/get_obs" + (f" + {rec} transitions/step/rank" if rec else "") + ")")
        for k in ("mean_train_reward", "mean_train_revenue", "mean_train_voltage_penalty", "mean_train_solver_failed"):
            print(f"  {k:32s} {means[k]: .6f}")
        if replay is not None and len(replay) >= 32:
            batch = learner_batch(policy, replay, 32)                  # replay.get_batch(32) + unpack_data, on the device
            print("  learner batch:", {k: tuple(v.shape) for k, v in batch.items()})
    policy.close(); env.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
