"""Host-buffer step (fp_step_host) microbenchmark: microseconds per BatchedFlexProvisionEnv.step_host call at one env
count, for fp32 and fp64 actions, each in pinned and in pageable host buffers.

    python tools/bench_e2e.py [--envs 131072] [--iters 60]

step_host synchronises the stream before it returns, so a host clock around each call times the whole step: copies,
kernel and synchronisation.  The library is the in-tree build, or FLEXGPU_LIB when set, so that two builds can be
compared by alternating runs.  Prints one header line with the card, its power limit and the library, then one JSON
line per (actions dtype, host memory)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "safe-marl_b200")]
from flexgpu import BatchedFlexProvisionEnv, DEFAULT_ENV_ARGS, Network, create_network, synthetic_profiles  # noqa: E402
from flexgpu import _lib  # noqa: E402

RESET_EVERY = 80          # untimed reset before the 95-step episodes run out


def card():
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out["power_limit"], out["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                           # report, do not guess
        out["power_limit"] = f"unavailable ({e.__class__.__name__})"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--iters", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    E = args.envs
    dev = torch.device("cuda:0")
    print(json.dumps({**card(), "lib": _lib.LIB_PATH, "envs": E}), flush=True)
    network = Network(create_network(DEFAULT_ENV_ARGS))
    env = BatchedFlexProvisionEnv(None, n_envs=E, device=dev, profiles=synthetic_profiles(network, 5, T=105216), seed=5)
    for dtype in (torch.float32, torch.float64):
        for memory in ("pinned", "pageable"):
            acts = torch.rand(4, E, 20, dtype=dtype, generator=torch.Generator().manual_seed(7))
            if memory == "pinned":
                acts = acts.pin_memory()
            host = [acts[k].numpy() for k in range(4)]
            ts = []
            for k in range(args.warmup + args.iters):
                if k % RESET_EVERY == 0:
                    env.reset(return_obs=False)
                    torch.cuda.synchronize()
                t0 = time.perf_counter()
                env.step_host(host[k % 4])
                if k >= args.warmup:
                    ts.append(time.perf_counter() - t0)
            med = statistics.median(ts)
            print(json.dumps({"actions": str(dtype).replace("torch.", ""), "memory": memory, "envs": E,
                              "us_per_step_median": round(med * 1e6, 1), "us_per_step_min": round(min(ts) * 1e6, 1),
                              "env_steps_per_s": round(E / med)}), flush=True)
    env.close()


if __name__ == "__main__":
    main()
