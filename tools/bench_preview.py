"""Step-preview benchmark: fp_step_preview (K candidate actions per env, nothing committed) against the plain step and
against the only alternative the library had before it, state_dict() -> step -> load_state_dict(); then an audit of the
safety layer against the exact power flow.  CUDA events, L2 overwritten before every timed call, medians.

    python tools/bench_preview.py [--iters 30] [--variant thread]

Timings: the preview at 131 072 envs for K = 1, 4, 16 and at 8 192 envs for K = 16 (per call and per candidate solve),
the plain step at 131 072 envs, and the state_dict round trip (host clock around a synchronised round trip, fewer runs).
Audit: a raw_actions (SAFEMADDPG) env, the reference's fitted voltage map (tests/golden/ref_predictor.npz, scalers
folded in) loaded with the "mixed" limits of tools/bench_safety.py; policy-like actions are projected with
safety_project_affine(layout="agent"), the projected setpoints are previewed through the exact step, and the line reports
which fraction of the envs the layer calls safe (inside the band, no slack left) still has a bus outside [v_min, v_max]
under the exact DistFlow solve.  Prints one JSON line per measurement after a header line naming the card."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "safe-marl_b200")]
from flexgpu import BatchedFlexProvisionEnv, DEFAULT_ENV_ARGS, Network, create_network, synthetic_profiles  # noqa: E402
from flexgpu import _lib  # noqa: E402
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


def ptr(t):
    return C.c_void_p(t.data_ptr())


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


def make_env(n, prof, variant, dev, **args):
    env = BatchedFlexProvisionEnv(dict(args, kernel_variant=variant), n_envs=n, device=dev, profiles=prof, seed=21)
    env.reset(return_obs=False)
    gen = torch.Generator(device=dev).manual_seed(3)
    for _ in range(3):
        env.step(torch.rand(n, 5, 4, device=dev, generator=gen), want_info=False)
    return env, gen


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--variant", default="thread", choices=("thread", "warp"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_preview.py needs a CUDA device")
    dev = torch.device("cuda:0")
    print(json.dumps({"card": card(), "variant": args.variant, "iters": args.iters}), flush=True)
    network = Network(create_network(DEFAULT_ENV_ARGS))
    prof = synthetic_profiles(network, 5, T=4000, seed=0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)        # > 126 MB of L2

    # ---- timings
    for n, ks in ((131072, (1, 4, 16)), (8192, (16,))):
        env, gen = make_env(n, prof, args.variant, dev)
        if n == 131072:
            a = torch.rand(n, 5, 4, device=dev, generator=gen)
            sd = env.state_dict()
            step = lambda: env.step(a, want_info=True)
            med, lo, hi = timed(step, flush, args.iters)
            env.load_state_dict(sd)
            print(json.dumps({"what": "step", "n_envs": n, "us_median": round(med, 2), "us_min": round(lo, 2),
                              "us_max": round(hi, 2)}), flush=True)
            ts = []
            for _ in range(5):                                       # the pre-preview way to ask "what would a do?"
                torch.cuda.synchronize(); t0 = time.perf_counter()
                s = env.state_dict(); env.step(a, want_info=True); env.load_state_dict(s)
                torch.cuda.synchronize(); ts.append((time.perf_counter() - t0) * 1e6)
            print(json.dumps({"what": "state_dict_step_load_state_dict", "n_envs": n, "us_median": round(float(np.median(ts)), 1),
                              "us_min": round(float(np.min(ts)), 1), "us_max": round(float(np.max(ts)), 1)}), flush=True)
        for k in ks:
            cand = torch.rand(k, n, 5, 4, device=dev, generator=gen)
            out = [torch.empty(k, n, dtype=torch.float64, device=dev), torch.empty(k, n, dtype=torch.uint8, device=dev),
                   torch.empty(k, n, 8, dtype=torch.float64, device=dev)]
            st = _lib.stream(dev)
            call = lambda: env._check(env._lib.fp_step_preview(env._h, k, ptr(cand), _lib.FP_F32, ptr(out[0]), ptr(out[1]),  # noqa: E731
                                                               ptr(out[2]), None, None, st), "fp_step_preview")
            med, lo, hi = timed(call, flush, args.iters)
            print(json.dumps({"what": "preview", "n_envs": n, "k": k, "us_median": round(med, 2), "us_min": round(lo, 2),
                              "us_max": round(hi, 2), "ns_per_candidate_solve": round(med / (k * n) * 1e3, 3)}), flush=True)
        env.close()

    # ---- audit: the safety layer's "safe" actions under the exact power flow
    n = 131072
    env, gen = make_env(n, prof, args.variant, dev, alg="safemaddpg")
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_predictor.npz"))
    pred = VoltagePredictor.from_linear_model(env, g["coef"].astype(np.float64), g["intercept"].astype(np.float64),
                                              g["x_scale"], g["x_min"], g["y_scale"], g["y_min"])
    A, c = pred.A, pred.c
    st = env.get_state(torch.float64).cpu().numpy()
    x = np.empty((n, 66)); x[:, 0::2] = st[:, :33]; x[:, 1::2] = st[:, 33:66]
    V = x @ A.T + c
    v_min, v_max = float(np.quantile(V.min(1), 0.3)), float(np.quantile(V.max(1), 0.85))     # bench_safety's "mixed"
    env.load_safety_map(A, c, v_min=v_min, v_max=v_max)
    actions = (torch.randn(n, 5, 4, device=dev, generator=gen) * 0.6 + 0.4).float()
    adj, slack, moved, status = env.safety_project_affine(actions, layout="agent", want_info=True)

    def outside(Vx):
        return ((Vx > v_max) | (Vx < v_min)).any(1)

    _, _, info_raw, V_raw = env.preview_step(actions, want_voltage=True)
    _, _, info_adj, V_adj = env.preview_step(adj, want_voltage=True)
    safe = (status >= 0) & (slack.amax(1) == 0)
    bad = outside(V_adj) & safe
    print(json.dumps({"what": "audit", "n_envs": n, "v_min": v_min, "v_max": v_max,
                      "frac_envs_outside_band_raw_actions": float(outside(V_raw).double().mean()),
                      "frac_envs_called_safe": float(safe.double().mean()),
                      "frac_safe_envs_outside_band_exact": float(bad.sum()) / max(1, int(safe.sum())),
                      "max_violation_of_safe_envs_pu": float(torch.clamp(torch.maximum(V_adj - v_max, v_min - V_adj), min=0)
                                                             .amax(1)[safe].max()) if bool(safe.any()) else 0.0,
                      "frac_solver_failed_projected": float(info_adj["solver_failed"].mean())}), flush=True)
    env.close()


if __name__ == "__main__":
    main()
