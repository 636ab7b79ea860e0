"""Config-4 microbenchmark of the MLP voltage predictor: k_predict_mlp against k_predict (the affine model), timed
alternately in the same process (CUDA events, median of the timed passes, the 256 MiB L2 flush between passes untimed),
penalty and Vhat written into the replay ring.  One JSON line per (envs, hidden shape); the first line names the card.

usage: bench_predictor_mlp.py [iters=50] [warmup=5]"""
import json, os, subprocess, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "safe-marl_b200")]
from flexgpu import BatchedFlexProvisionEnv, DEFAULT_ENV_ARGS, Network, create_network, synthetic_profiles
from flexgpu.predictor import DeviceReplayBuffer, MLPVoltagePredictor, VoltagePredictor

iters = int(sys.argv[1]) if len(sys.argv) > 1 else 50
warmup = int(sys.argv[2]) if len(sys.argv) > 2 else 5
SIZES = (262144, 1 << 20)
SHAPES = ((64,), (100,), (128,), (64, 64))
HBM_GBS = 6650.0           # the project's measured B200 HBM read+write rate (tools/bench_predictor.py uses the same)
TF32_TFLOPS = 1125.0       # NVIDIA data sheet, dense TF32, one HGX B200 GPU at 1000 W

dev = torch.device("cuda:0")
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True)
print(json.dumps({"card": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown",
                  "torch": torch.__version__, "iters": iters, "warmup": warmup}), flush=True)

network = Network(create_network(DEFAULT_ENV_ARGS))
env = BatchedFlexProvisionEnv(None, n_envs=8, device=dev, profiles=synthetic_profiles(network, 5, T=2000))
g = np.load(os.path.join(ROOT, "tests", "golden", "predictor_golden.npz"))
affine = VoltagePredictor.from_linear_model(env, g["coef"], g["intercept"], g["x_scale"], g["x_min"], g["y_scale"], g["y_min"])
base = torch.from_numpy(np.stack([network.base_p, network.base_q], axis=1).reshape(-1)).to(dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def mlp_model(hidden, seed=0):
    """A relu MLP whose output stays near 1 p.u. on config-4 inputs (random weights: timing does not depend on them)."""
    rng = np.random.default_rng(seed)
    widths = (66,) + hidden + (33,)
    W = [rng.normal(0, 1.0 / np.sqrt(i), (o, i)) for i, o in zip(widths[:-1], widths[1:])]
    b = [rng.normal(0, 0.1, o) for o in widths[1:]]
    W[-1] *= 0.01; b[-1] = np.ones(33)
    return W, b


def timed(fn):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record()
    return a, b


for n in SIZES:
    # config 4 (SURVEY 8d): X = interleaved [p_n, q_n] of load scenarios, base loads x U(0.7, 1.3)
    X = (base[None, :] * (0.7 + 0.6 * torch.rand(n, 66, device=dev, dtype=torch.float64))).float().contiguous()
    buf = DeviceReplayBuffer(2 * n, {"v_pred": 33, "safety_penalty": 1}, device=dev)
    for hidden in SHAPES:
        W, b = mlp_model(hidden)
        mlp = MLPVoltagePredictor(env, W, b, activation="relu")
        run_m = lambda: mlp.predict(X, want_vhat=False, want_penalty=False, sink=buf)
        run_a = lambda: affine.predict(X, want_vhat=False, want_penalty=False, sink=buf)
        for _ in range(warmup):
            run_m(); run_a()
        ev_m, ev_a = [], []
        for _ in range(iters):                                   # alternate, so both see the same machine state
            ev_m.append(timed(run_m)); ev_a.append(timed(run_a))
        torch.cuda.synchronize()
        ms_m = float(np.median([a.elapsed_time(b) for a, b in ev_m]))
        ms_a = float(np.median([a.elapsed_time(b) for a, b in ev_a]))
        widths = (66,) + hidden + (33,)
        kp = [72] + [(h + 15) // 16 * 16 for h in hidden]
        np_ = [(h + 15) // 16 * 16 for h in hidden] + [48]
        bytes_alg = n * (66 * 4 + 33 * 4 + 4)
        useful = 2.0 * n * sum(i * o for i, o in zip(widths[:-1], widths[1:]))
        issued = 6.0 * n * sum(k * m for k, m in zip(kp, np_))
        hbm_ms = bytes_alg / (HBM_GBS * 1e9) * 1e3
        tf32_ms = issued / (TF32_TFLOPS * 1e12) * 1e3
        bound_ms = max(hbm_ms, tf32_ms)
        print(json.dumps({"workload": f"MLP predictor+penalty->replay, {n} envs, hidden {list(hidden)} relu (config 4)",
                          "envs": n, "hidden": list(hidden), "ms": ms_m, "envs_per_s": n / ms_m * 1e3,
                          "affine_ms_same_call": ms_a, "ratio_to_affine": ms_m / ms_a,
                          "bytes_per_env": bytes_alg / n, "useful_flop": useful, "issued_tf32_flop": issued,
                          "hbm_bound_ms": hbm_ms, "tf32_bound_ms": tf32_ms,
                          "bound": "hbm" if hbm_ms >= tf32_ms else "tf32", "share_of_bound": bound_ms / ms_m,
                          "useful_tflops": useful / ms_m / 1e9, "issued_tf32_tflops": issued / ms_m / 1e9}), flush=True)
    buf.close()
env.close()
