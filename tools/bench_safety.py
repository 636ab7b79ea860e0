"""Safety-layer microbenchmark: the row-sum projection (fp_safety_project, closed form) and the full affine map
(fp_safety_project_affine, active set) over N envs, CUDA events, L2 overwritten before every timed call, median.

    python tools/bench_safety.py [--sizes 131072,1048576] [--iters 30]

Mixes: "inside" (limits no prediction reaches: the no-op path), "mixed" (limits on the spread of the predictions, part
of the envs pushed out on either side), "hopeless" (v_min above every reachable voltage).  Maps: the reference's own fit
(tests/golden/ref_predictor.npz) with its scalers folded in for the affine form, its row sums for fp_safety_project.
Prints one JSON line per (size, mix, form) and one header line with the card and its power limit."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "safe-marl_b200")]
from flexgpu import BatchedFlexProvisionEnv, DEFAULT_ENV_ARGS, Network, create_network, synthetic_profiles  # noqa: E402
from flexgpu.predictor import VoltagePredictor  # noqa: E402


def card():
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out["power_limit"], out["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                           # report, do not guess
        out["power_limit"] = f"unavailable ({e.__class__.__name__})"
    return out


def timed(fn, flush, iters):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize(); ts.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="131072,1048576")
    ap.add_argument("--iters", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_safety.py needs a CUDA device")
    dev = torch.device("cuda:0")
    print(json.dumps({"card": card()}), flush=True)
    network = Network(create_network(DEFAULT_ENV_ARGS))
    prof = synthetic_profiles(network, 5, T=4000, seed=0)
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_predictor.npz"))
    coef, icpt = g["coef"].astype(np.float64), g["intercept"].astype(np.float64)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)        # > 126 MB of L2
    for n in [int(s) for s in args.sizes.split(",")]:
        env = BatchedFlexProvisionEnv(None, n_envs=n, device=dev, profiles=prof, seed=21)
        env.reset(return_obs=False)
        gen = torch.Generator(device=dev).manual_seed(3)
        for _ in range(3):
            env.step(torch.rand(n, 5, 4, device=dev, generator=gen), want_info=False)
        actions = (torch.randn(n, 5, 4, device=dev, generator=gen) * 0.6 + 0.4).float()
        pred = VoltagePredictor.from_linear_model(env, coef, icpt, g["x_scale"], g["x_min"], g["y_scale"], g["y_min"])
        A, c = pred.A, pred.c
        st = env.get_state(torch.float64).cpu().numpy()
        x = np.empty((n, 66)); x[:, 0::2] = st[:, :33]; x[:, 1::2] = st[:, 33:66]
        V = x @ A.T + c
        mixes = {"inside": (float(V.min()) - 10.0, float(V.max()) + 10.0),
                 "mixed": (float(np.quantile(V.min(1), 0.3)), float(np.quantile(V.max(1), 0.85))),
                 "hopeless": (float(V.max()) + 50.0, float(V.max()) + 60.0)}
        out = torch.empty(n, 20, dtype=torch.float32, device=dev)
        slack_a = torch.empty(n, 33, dtype=torch.float64, device=dev); slack_r = torch.empty(n, 5, dtype=torch.float64, device=dev)
        moved = torch.empty(n, 5, dtype=torch.uint8, device=dev); status = torch.empty(n, dtype=torch.int32, device=dev)
        lib, h, s = env._lib, env._h, lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
        p = lambda t: C.c_void_p(t.data_ptr())
        for mix, (v_min, v_max) in mixes.items():
            env.load_safety_map(A, c, v_min=v_min, v_max=v_max)
            env._check(lib.fp_safety_load(h, coef.ctypes.data_as(C.c_void_p), icpt.ctypes.data_as(C.c_void_p), v_min, v_max, 1000.0),
                       "fp_safety_load")
            affine = lambda: env._check(lib.fp_safety_project_affine(h, p(actions), 0, p(out), 1, p(slack_a), p(moved), p(status), s()),
                                        "fp_safety_project_affine")
            rowsum = lambda: env._check(lib.fp_safety_project(h, p(actions), 0, p(out), 1, p(slack_r), p(moved), s()), "fp_safety_project")
            for form, fn in (("rowsum", rowsum), ("affine", affine)):
                med, lo, hi = timed(fn, flush, args.iters)
                fn(); torch.cuda.synchronize()
                rec = {"n_envs": n, "mix": mix, "form": form, "us_median": round(med, 2), "us_min": round(lo, 2), "us_max": round(hi, 2),
                       "projections_per_s": n / med * 1e6, "frac_envs_intervened": float(moved.bool().any(1).double().mean())}
                if form == "affine":
                    it = status.double()
                    rec.update({"iters_mean": float(it.clamp(min=0).mean()), "iters_max": int(status.max()),
                                "iters_mean_intervened": float(it[status > 0].mean()) if bool((status > 0).any()) else 0.0,
                                "n_capped": int((status < 0).sum())})
                print(json.dumps(rec), flush=True)
        env.close()


if __name__ == "__main__":
    main()
