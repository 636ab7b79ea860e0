"""k_critic alone: python tools/bench_critic.py [ENVS] [ITERS] -- CUDA events, L2 flushed before every launch.
NA=1..5 (default 5): agents per env."""
import json, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "safe-marl_b200")]
from flexgpu.policy import DevicePolicy

E = int(sys.argv[1]) if len(sys.argv) > 1 else 131072
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 20
dev = torch.device("cuda:0")
rng = np.random.default_rng(7)
NA = int(os.environ.get("NA", "5"))
sd = {"fc1.weight": rng.normal(0, 0.05, (64, 149 * NA)), "fc1.bias": rng.uniform(-0.04, 0.04, 64), "layernorm.weight": np.ones(64),
      "layernorm.bias": np.zeros(64), "fc2.weight": rng.uniform(-0.125, 0.125, (64, 64)), "fc2.bias": rng.uniform(-0.125, 0.125, 64),
      "fc3.weight": rng.uniform(-0.125, 0.125, (1, 64)), "fc3.bias": rng.uniform(-0.125, 0.125, 1)}
pol = DevicePolicy(None, device=dev, n_agents=NA)
pol.load_critic(sd)
n_pad = (E + 31) // 32 * 32
ring = torch.rand(24, NA, 6, n_pad, device=dev)
act = torch.tanh(torch.randn(E, NA, 4, device=dev))
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
ts = []
for k in range(iters + 3):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); pol.value(ring, act, slot=k % 24, n_envs=E); b.record()
    torch.cuda.synchronize()
    if k >= 3:
        ts.append(a.elapsed_time(b) * 1e3)
us = float(np.median(ts))
bytes_env = 4 * NA * (24 * 6 + 4 + 1)                            # the ring, the actions, the values
flop_env = 2 * 2 * (NA * 148 * 64 + NA * 64 * 64) + NA * 2 * 64  # two products per term (hi, lo) on the tensor cores + fc3
print(json.dumps({"envs": E, "agents": NA, "us_median": round(us, 1), "env_rows_per_s": round(NA * E / us * 1e6 / 1e9, 3), "bytes_per_env": bytes_env,
                  "hbm_frac": round(bytes_env * E / (us * 1e-6) / 6553.3e9, 4), "tf32_tflops": round(flop_env * E / (us * 1e-6) / 1e12, 1)}))
