"""k_policy alone: python tools/bench_policy.py [ENVS] [ITERS] -- CUDA events, L2 flushed before every launch.
NA=1..5 (default 5): agents per env; HID_EM=0: hidden states in rows instead of the env-minor layout."""
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
sd = {"fc1.weight": rng.normal(0, 0.1, (64, 144 + NA)), "fc1.bias": rng.uniform(-0.08, 0.08, 64), "layernorm.weight": np.ones(64),
      "layernorm.bias": np.zeros(64), "rnn.weight_ih": rng.uniform(-0.125, 0.125, (192, 64)),
      "rnn.weight_hh": rng.uniform(-0.125, 0.125, (192, 64)), "rnn.bias_ih": rng.uniform(-0.125, 0.125, 192),
      "rnn.bias_hh": rng.uniform(-0.125, 0.125, 192), "fc2.weight": rng.normal(0, 0.1, (4, 64)), "fc2.bias": rng.uniform(-0.125, 0.125, 4)}
pol = DevicePolicy(sd, device=dev)
n_pad = (E + 31) // 32 * 32
ring = torch.rand(24, NA, 6, n_pad, device=dev)
EM = bool(os.environ.get("HID_EM", "1") != "0")
h = [torch.rand(NA, 64, n_pad, device=dev) - 0.5, torch.empty(NA, 64, n_pad, device=dev)] if EM else [torch.rand(E, NA, 64, device=dev) - 0.5, torch.empty(E, NA, 64, device=dev)]
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
ts = []
NOHID = bool(os.environ.get("NOHID")); NOFLUSH = bool(os.environ.get("NOFLUSH"))
for k in range(iters + 3):
    if not NOFLUSH:
        flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); pol.act(ring, slot=k % 24, n_envs=E, hid_in=None if NOHID else h[k % 2], hid_out=h[1 - k % 2], step=k, hid_layout="env_minor" if EM else "rows"); b.record()
    torch.cuda.synchronize()
    if k >= 3:
        ts.append(a.elapsed_time(b) * 1e3)
us = float(np.median(ts))
# algorithmic bytes per env: the whole ring (24 x NA x 6 floats) + hidden in/out (2 x NA x 64) + action / log-prob out (2 x NA x 4)
bytes_env = 4 * NA * (24 * 6 + 2 * 64 + 2 * 4)
flop_env = NA * 2 * 2 * (144 * 64 + 2 * 64 * 192 + 64 * 16)     # 2 products per term (hi, lo)
print(json.dumps({"envs": E, "agents": NA, "us_median": round(us, 1), "rows_per_s": round(NA * E / us * 1e6 / 1e9, 3), "bytes_per_env": bytes_env,
                  "hbm_frac": round(bytes_env * E / (us * 1e-6) / 6553.3e9, 4), "tf32_tflops": round(flop_env * E / (us * 1e-6) / 1e12, 1)}))
