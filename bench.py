#!/usr/bin/env python
"""bench.py -- 33-bus env-steps/s (incl. power flow) of the fused flex_provision step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu E] [--impl reference] [--dump-outputs DIR]

A "step" is one fused env step (action application, injections, DistFlow power flow,
constraint masks, reward/penalty, ESS update, bookkeeping: flexibility_provision_env.py:241-356)
over the E environments resident on each GPU.  Workload: E = 131 072 envs per GPU -- one GPU's
shard of BASELINE config 5 (2^20 envs over 8 B200), the configuration the 1/2/4/8-GPU metric is
quoted on; at N = 8 the run IS config 5.  Every rank holds its own E envs (weak scaling, no
collective on the step path; one NCCL all-reduce of the 16-double statistics vector after the
timed region).  Config 3 (65 536 envs on one B200) is measured in the same run at N = 1 and
reported as `config3`.  Episodes are 95 steps long (quirk Q1), so a Philox auto-reset launch runs
inside the timed region every 94 steps -- it is part of a rollout and is counted.

Timing: W untimed steps, then K steps, each bracketed by CUDA events on the launching stream
with an L2 flush (256 MiB memset, untimed) before it -- a good part of the per-GPU working set
would otherwise sit in the 126 MB L2.  value = total envs * K / max-over-ranks(sum of step times).
e2e: the same step through fp_step_host (pinned host actions in, reward+done out, copies and
the stream sync inside the timed region), wall-clocked.

Beside the headline (N = 1 only unless noted): `config2` (BASELINE config 2: 4096 power-flow-only
solves, both kernel variants, 776 B/solve), `config3` (65 536 envs), `config4` (predictor -> replay
ring, 262 144 envs), `config5_strong` (every N: 2^20 envs IN TOTAL split over the N GPUs -- strong
scaling of config 5), `step_plus_get_obs` (fused step + observation push into the env-minor ring,
the rollout loop's env cost), `roofline_fp64` (the step kernel against the fp64 pipe).

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned to its caller
(reward, terminated, the eight info fields; one value per env) as DIR/<name>.npy in float64 (terminated in
float32), at most 64 MB in all: above that, the same fixed seeded sample of envs from every array, with its
env indices in DIR/env_index.npy.  Inputs are seeded, so two builds run with the same arguments can be
compared output for output.

--impl reference: the CPU arm.  The reference's own implementation (Pyomo + IPOPT) is probed for
(`import pyomo`, `which ipopt`: utils/pf.py:101) but is not installable here (SURVEY 8c), so this
times the oracle port: oracle/c/flex_oracle.c (OpenMP, all host cores) on the same workload (same
envs per step, same steps and warm-up), plus the single-core Python restatement (oracle/env_ref.py)
for scale.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "safe-marl_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "33-bus env-steps/sec (incl. power flow)"
UNIT = "env-steps/s"
B_ALG = 1256            # algorithmic bytes per env-step (SURVEY 8d; DESIGN.md "Roofline")
EPISODE_STEPS = 94      # steps between auto-resets (an episode terminates at its 95th step)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_mirror(n, prof, seed):
    from oracle import c_mirror, env_ref, ieee33
    fonet = c_mirror.make_net(ieee33.tree_arrays(ieee33.create_network()), env_ref.DEFAULT_ARGS,
                              env_ref.DEFAULT_ARGS["buildings"])
    mb = c_mirror.MirrorBatch(fonet, prof.as_dict(), n)
    mb.reset_random(seed)
    return mb


def cpu_port_rate(prof, n_envs, budget_s, seed=5):
    """The C port (OpenMP, all cores) on a bounded sample: `n` envs stepped until budget_s."""
    import numpy as np
    from oracle import c_mirror
    cores = c_mirror.use_all_cores()
    n = n_envs
    mb = make_mirror(n, prof, seed)
    rng = np.random.default_rng(0)
    acts = rng.uniform(0, 1, (4, n, 20)).astype(np.float32)
    mb.step(acts[0])                                           # warm-up (page faults, thread pool)
    t0 = time.perf_counter(); k = 0
    while True:
        mb.step(acts[k % 4]); k += 1
        el = time.perf_counter() - t0
        if el >= budget_s or k >= 90:
            break
    return n * k / el, cores, f"{n} envs x {k} steps of the C port (oracle/c/flex_oracle.c, OpenMP) in {el:.2f} s"


def python_restatement_rate(prof, budget_s=5.0):
    """Single-core Python restatement (env_ref + sweep power flow): the reference's structure
    (per-env Python objects) minus Pyomo/IPOPT, i.e. a generous stand-in for its per-env step."""
    import numpy as np
    from oracle import env_ref, ieee33
    env = env_ref.RefFlexEnv(dict(env_ref.DEFAULT_ARGS), ieee33.create_network(), prof.as_dict(),
                             rng=np.random.RandomState(0), pf_method='sweep')
    rng = np.random.RandomState(1)
    t0 = time.perf_counter(); k = 0
    while time.perf_counter() - t0 < budget_s:
        _, done, _ = env.step(rng.uniform(0, 1, 20))
        k += 1
        if done:
            env.reset()
    return k / (time.perf_counter() - t0)


def ncu_capture(envs_per_gpu):
    """Counters of one k_env_t<STEP> launch from the committed `ncu --set full` capture
    (profiles/r2_step_kernel_traffic.json), if it was taken at this launch size: DRAM bytes
    (dram__bytes_read.sum + dram__bytes_write.sum) and fp64 / fp32 lane-operations."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_step_kernel_traffic.json")) as f:
            d = json.load(f)
        return d if int(d["envs"]) == int(envs_per_gpu) else None
    except (OSError, ValueError, KeyError):
        return None


FP64_PEAK_LANE_OPS_PER_CLK_SM = 59.0    # measured on B200 (profiles/r1_ubench_fp64_b200.txt; nominal 64)


def workload_name(envs_per_gpu):
    return (f"fused_env_step_{envs_per_gpu}_envs_per_gpu (one GPU's shard of BASELINE config 5 = 2^20 envs over 8 GPUs; "
            f"N=8 is config 5)")


def make_config(args, world, auto_reset):
    """The `config` object: identical for the GPU arm and the reference arm of the same command line."""
    c = {"workload": workload_name(args.envs_per_gpu), "envs_per_gpu": args.envs_per_gpu,
         "total_envs": args.envs_per_gpu * world, "profile_rows": args.rows,
         "actions": "fp32 uniform(0,1), one [envs, 5, 4] array per step",
         "episode": "Philox reset before the warm-up; 95-step episodes (quirk Q1)"}
    if auto_reset:
        c["auto_reset_every"] = EPISODE_STEPS
    return c


DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir, reward, done, info):
    """What one env.step(..., want_info=True) returned, as DIR/<name>.npy (see --dump-outputs)."""
    import numpy as np
    import torch
    arrays = {"reward": reward.double(), "terminated": done.float()}
    arrays.update({f"info_{k}": v.double() for k, v in info.items()})
    n = reward.shape[0]
    per_env = sum(t.element_size() for t in arrays.values())
    if n * per_env > DUMP_MAX_BYTES:
        k = (DUMP_MAX_BYTES - 4096) // (per_env + 8)               # + 8: the float64 env index; 4096: the .npy headers
        sel = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, k, replace=False))).to(reward.device)
        arrays = {name: t.index_select(0, sel) for name, t in arrays.items()}
        arrays["env_index"] = sel.double()
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def probe_reference_solver():
    """BASELINE.md 4.1: is the reference's own power flow (Pyomo + the ipopt binary, utils/pf.py:101) runnable here?"""
    try:
        import pyomo  # noqa: F401
        have_pyomo = True
    except Exception:
        have_pyomo = False
    return {"pyomo": have_pyomo, "ipopt": shutil.which("ipopt") is not None}


def run_reference(args):
    """--impl reference: the CPU arm (rank 0 only) on the GPU arm's workload: the same number of envs per step
    (all N GPUs' shards), the same steps and warm-up."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from flexgpu import DEFAULT_ENV_ARGS, Network, create_network, synthetic_profiles
    network = Network(create_network(DEFAULT_ENV_ARGS))
    prof = synthetic_profiles(network, 5, T=args.rows, seed=0)
    import numpy as np
    from oracle import c_mirror
    probe = probe_reference_solver()
    cores = c_mirror.use_all_cores()                             # torchrun exports OMP_NUM_THREADS=1
    W = max(args.warmup, 3); K = args.steps
    total = args.envs_per_gpu * args.gpus
    # bounded: at most ~1.5e9 env-steps of CPU work (a few minutes on 16 cores); otherwise step a sample of the envs
    n = total if total * (K + W) <= 1.5e9 else max(1024, int(1.5e9 / (K + W)) // 32 * 32)
    mb = make_mirror(n, prof, 5)
    rng = np.random.default_rng(0)
    acts = rng.uniform(0, 1, (4, n, 20)).astype(np.float32)
    t_in_ep = 0
    resets = 0
    def one(k):
        nonlocal t_in_ep, resets
        if t_in_ep == EPISODE_STEPS:
            mb.reset_random(5); t_in_ep = 0; resets += 1        # same Philox key, next episode counter
        mb.step(acts[k % 4]); t_in_ep += 1
    for w in range(W):
        one(w)
    resets = 0
    t0 = time.perf_counter()
    for k in range(K):
        one(W + k)
    el = time.perf_counter() - t0
    value = n * K / el
    py = python_restatement_rate(prof, 5.0)
    kind = "port"                                                # the true reference needs pyomo + ipopt AND /root/reference
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": 1e3 * el / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(args, args.gpus, resets > 0),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{n} envs per step x {K} steps (+{W} warm-up) of the C port of the step (oracle/c/flex_oracle.c, "
                                   f"OpenMP, {cores} threads)" + ("" if n == total else f" -- a sample of the {total} envs") +
                                   f"; single-core Python restatement: {py:.0f} env-steps/s",
                         "reference_solver_probe": probe,
                         "note": "the reference's own step is Pyomo + an ipopt subprocess per env-step; neither is installed "
                                 "(and /root/reference does not exist on the GPU box), so the arm runs the port"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--envs-per-gpu", type=int, default=131072)
    ap.add_argument("--rows", type=int, default=105216, help="profile dataset rows (bundled-data shape)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config3", action="store_true", help="skip the extra 65 536-env (config 3) measurement at N=1")
    ap.add_argument("--no-flush", action="store_true", help="skip the L2 flush (diagnostics only)")
    ap.add_argument("--no-config4", action="store_true", help="skip the extra predictor (config 4) measurement at N=1")
    ap.add_argument("--no-obs", action="store_true", help="skip the extra step+get_obs measurement (rollout-loop cost)")
    ap.add_argument("--no-config2", action="store_true", help="skip the extra power-flow-only (config 2) measurement at N=1")
    ap.add_argument("--no-strong", action="store_true", help="skip the extra strong-scaling (2^20 envs in total) measurement")
    ap.add_argument("--no-rollout", action="store_true", help="skip the extra device-rollout measurement (policy + step + get_obs [+ Transition writes])")
    ap.add_argument("--variant", default="thread", choices=["thread", "warp"], help="kernel variant (see include/flexgpu.h)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy "
                    "(rank 0's envs only when several GPUs run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the GPU path; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from flexgpu import BatchedFlexProvisionEnv, DEFAULT_ENV_ARGS, Network, create_network, synthetic_profiles

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3); K = args.steps; E = args.envs_per_gpu

    network = Network(create_network(DEFAULT_ENV_ARGS))
    prof = synthetic_profiles(network, 5, T=args.rows, seed=0)
    env = BatchedFlexProvisionEnv({"kernel_variant": args.variant}, n_envs=E, device=dev, profiles=prof, seed=5,
                                  env_offset=rank * E)
    env.reset(return_obs=False)
    n_act = 8
    g = torch.Generator(device=dev).manual_seed(2 + rank)
    acts = torch.rand(n_act, E, 5, 4, device=dev, dtype=torch.float32, generator=g)     # resident in HBM
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    state = {"t": 0, "timed_resets": 0}

    def one_step(k, timed):
        if state["t"] == EPISODE_STEPS:
            env.reset(return_obs=False)                       # Philox auto-reset, one launch
            state["t"] = 0
            state["timed_resets"] += 1 if timed else 0
        out = env.step(acts[k % n_act], want_info=True)
        state["t"] += 1
        return out

    for k in range(W):
        if not args.no_flush:
            flush.zero_()
        one_step(k, False)
    barrier()
    env.episode_stats(reduce=False, reset=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    barrier()
    launches0 = env.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    t_wall0 = time.perf_counter()
    for k in range(K):
        if not args.no_flush:
            flush.zero_()
        ev[k][0].record(stream)
        last = one_step(W + k, True)
        ev[k][1].record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = env.launch_count() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    # kernel-only duration of the dominant kernel (k_env<STEP>): steps without a reset in them
    step_ms = sorted(a.elapsed_time(b) for a, b in ev)
    kern_ms = statistics.median(step_ms)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)        # before the measurements below step or reset this env again

    # ---- e2e: through fp_step_host with pinned HOST buffers (copies + sync inside)
    h_act = torch.rand(4, E, 20, dtype=torch.float32).pin_memory()
    Ke = max(10, min(K, 100))
    env.reset(return_obs=False); state["t"] = 0
    for k in range(3):
        env.step_host(h_act[k % 4].numpy())
    barrier()
    t0 = time.perf_counter()
    for k in range(Ke):
        if 3 + k == EPISODE_STEPS:
            env.reset(return_obs=False)
        r_h, d_h, _ = env.step_host(h_act[k % 4].numpy())
    barrier()
    e2e_s = time.perf_counter() - t0

    obs_extra = None
    if not args.no_obs:
        # the rollout loop's env cost: step + pushing get_obs (model.py:220-223) in ONE launch, observation
        # history in its native env-minor ring (what the device policy reads)
        env.reset(return_obs="ring")
        for k in range(3):
            env.step(acts[k % n_act], want_info=False, return_obs="ring")
        Ko = 40
        evo = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Ko)]
        barrier()
        for k in range(Ko):
            if not args.no_flush:
                flush.zero_()
            evo[k][0].record(stream); env.step(acts[k % n_act], want_info=False, return_obs="ring"); evo[k][1].record(stream)
        barrier()
        obs_ms = sum(a.elapsed_time(b) for a, b in evo)
        # the same with ring-only stepping (set_obs_history(False): the fp64 history ring behind get_obs() is not pushed;
        # what the device rollout uses)
        env.set_obs_history(False)
        for k in range(3):
            env.step(acts[k % n_act], want_info=False, return_obs="ring")
        barrier()
        for k in range(Ko):
            if not args.no_flush:
                flush.zero_()
            evo[k][0].record(stream); env.step(acts[k % n_act], want_info=False, return_obs="ring"); evo[k][1].record(stream)
        barrier()
        obs_ring_ms = sum(a.elapsed_time(b) for a, b in evo)
        env.set_obs_history(True)
        obs_extra = (E * Ko, obs_ms, obs_ring_ms)

    # ---- the rollout loop on the device (model.py:213-254): tcgen05 policy -> fused translate_action + step + get_obs
    #      [-> Transition fields into the device replay ring]; nothing crosses PCIe (only the statistics, afterwards)
    rollout = None
    if not args.no_rollout and args.variant == "thread":
        from flexgpu.policy import DevicePolicy, DeviceRollout, TRANSITION_FIELDS
        from flexgpu.predictor import DeviceReplayBuffer
        rngp = np.random.default_rng(7)
        sd = {"fc1.weight": rngp.normal(0, 0.1, (64, 149)), "fc1.bias": rngp.uniform(-0.08, 0.08, 64), "layernorm.weight": np.ones(64),
              "layernorm.bias": np.zeros(64), "rnn.weight_ih": rngp.uniform(-0.125, 0.125, (192, 64)),
              "rnn.weight_hh": rngp.uniform(-0.125, 0.125, (192, 64)), "rnn.bias_ih": rngp.uniform(-0.125, 0.125, 192),
              "rnn.bias_hh": rngp.uniform(-0.125, 0.125, 192), "fc2.weight": rngp.normal(0, 0.1, (4, 64)), "fc2.bias": rngp.uniform(-0.125, 0.125, 4)}
        pol = DevicePolicy(sd, device=dev, std=1.0, seed=11 + rank)
        # the critic of train_process's value / next_value (model.py:217, :225-226): the reference's MLPCritic, random init
        pol.load_critic({"fc1.weight": rngp.normal(0, 0.05, (64, 745)), "fc1.bias": rngp.uniform(-0.04, 0.04, 64), "layernorm.weight": np.ones(64),
                         "layernorm.bias": np.zeros(64), "fc2.weight": rngp.uniform(-0.125, 0.125, (64, 64)), "fc2.bias": rngp.uniform(-0.125, 0.125, 64),
                         "fc3.weight": rngp.uniform(-0.125, 0.125, (1, 64)), "fc3.bias": rngp.uniform(-0.125, 0.125, 1)})
        rollout = {}
        for label, rec, vf in (("acting", 0, None), ("recording", E, None), ("critic", E, "native")):
            buf = DeviceReplayBuffer(2 * E, TRANSITION_FIELDS, device=dev) if rec else None
            ro = DeviceRollout(env, pol, replay=buf, record_envs=rec, value_fn=vf)
            ro.reset()
            for k in range(3):
                ro.step()
            Kr = 30
            evr = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Kr)]
            l0 = env.launch_count() + pol.launch_count()
            barrier()
            for k in range(Kr):
                if not args.no_flush:
                    flush.zero_()
                evr[k][0].record(stream); ro.step(); evr[k][1].record(stream)
            barrier()
            rollout[label] = (E * Kr, sum(a.elapsed_time(b) for a, b in evr), (env.launch_count() + pol.launch_count() - l0) / Kr)
            if buf is not None:
                buf.close()
        pol.close()

    # ---- strong scaling of BASELINE config 5: 2^20 envs IN TOTAL, split over the ranks (every N)
    strong = None
    if not args.no_strong:
        Es = (1 << 20) // world
        envs = BatchedFlexProvisionEnv({"kernel_variant": args.variant}, n_envs=Es, device=dev, profiles=prof, seed=5,
                                       env_offset=rank * Es)
        envs.reset(return_obs=False)
        acts_s = torch.rand(2, Es, 5, 4, device=dev, dtype=torch.float32, generator=g)
        Ks = 20
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Ks)]
        for k in range(3):
            flush.zero_(); envs.step(acts_s[k % 2], want_info=True)
        barrier()
        for k in range(Ks):
            flush.zero_()
            evs[k][0].record(stream); envs.step(acts_s[k % 2], want_info=True); evs[k][1].record(stream)
        barrier()
        strong = (Es, Ks, sum(a.elapsed_time(b) for a, b in evs))
        envs.close(); del acts_s

    # ---- BASELINE config 2 (4096 independent power-flow-only solves, utils/pf.py:115-192), both variants, N = 1 only
    config2 = None
    if world == 1 and not args.no_config2:
        n2 = 4096
        rng2 = np.random.default_rng(0)
        p2 = torch.from_numpy(network.base_p[None, 1:] * rng2.uniform(0.7, 1.3, (n2, 32))).to(dev)      # data_generation.py:27-36
        q2 = torch.from_numpy(network.base_q[None, 1:] * rng2.uniform(0.7, 1.3, (n2, 32))).to(dev)
        config2 = {"workload": "power_flow_only_4096_solves (BASELINE config 2: run_pf.py-style batched solve, V out)",
                   "unit": "solves/s", "bytes_per_solve": 776, "variants": {}}
        for var in ("thread", "warp"):
            e2 = env if var == args.variant else BatchedFlexProvisionEnv({"kernel_variant": var}, n_envs=32, device=dev,
                                                                         profiles=synthetic_profiles(network, 5, T=2000, seed=0), seed=5)
            for k in range(5):
                e2.power_flow(p2, q2, want_flows=False)
            ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(40)]
            for k in range(40):
                flush.zero_()
                ev2[k][0].record(stream); out2 = e2.power_flow(p2, q2, want_flows=False); ev2[k][1].record(stream)
            torch.cuda.synchronize()
            ms2 = statistics.median(a.elapsed_time(b) for a, b in ev2)
            config2["variants"][var] = {"value": n2 / (ms2 * 1e-3), "kernel_ms_median": ms2,
                                        "roofline_frac": 776 * n2 / (ms2 * 1e-3) / 1e9 / peaks()[0],
                                        "passes_max": int(out2["iters"].max()), "failed": int(out2["failed"].sum())}
            if e2 is not env:
                e2.close()
        best = max(config2["variants"], key=lambda v: config2["variants"][v]["value"])
        config2["value"] = config2["variants"][best]["value"]; config2["best_variant"] = best
        config2["note"] = "4096 solves are 128 tiles of 32 on 148 SMs: one launch latency, not a bandwidth measurement"

    # ---- BASELINE config 3 (65 536 envs on one B200), same method, N = 1 only
    config3 = None
    if world == 1 and E != 65536 and not args.no_config3:
        E3 = 65536
        env3 = BatchedFlexProvisionEnv({"kernel_variant": args.variant}, n_envs=E3, device=dev, profiles=prof, seed=5)
        env3.reset(return_obs=False)
        acts3 = torch.rand(4, E3, 5, 4, device=dev, dtype=torch.float32, generator=g)
        K3 = 60
        ev3 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K3)]
        for k in range(5):
            flush.zero_(); env3.step(acts3[k % 4], want_info=True)
        for k in range(K3):
            flush.zero_()
            ev3[k][0].record(stream); env3.step(acts3[k % 4], want_info=True); ev3[k][1].record(stream)
        torch.cuda.synchronize()
        ms3 = [a.elapsed_time(b) for a, b in ev3]
        config3 = {"workload": "fused_env_step_65536_envs (BASELINE config 3)", "value": E3 * K3 / (sum(ms3) * 1e-3),
                   "unit": UNIT, "steps": K3, "kernel_ms_median": statistics.median(ms3),
                   "roofline_frac": B_ALG * E3 / (statistics.median(ms3) * 1e-3) / 1e9 / peaks()[0]}
        env3.close()

    # ---- BASELINE config 4 (voltage predictor + safety penalty -> replay ring, 262 144 envs), N = 1 only
    config4 = None
    if world == 1 and not args.no_config4:
        import numpy as np
        from flexgpu import Network, create_network, DEFAULT_ENV_ARGS
        from flexgpu.predictor import DeviceReplayBuffer, VoltagePredictor
        E4 = 262144
        gp = np.load(os.path.join(ROOT, "tests", "golden", "predictor_golden.npz"))
        pred = VoltagePredictor.from_linear_model(env, gp["coef"], gp["intercept"], gp["x_scale"], gp["x_min"], gp["y_scale"], gp["y_min"])
        net4 = Network(create_network(DEFAULT_ENV_ARGS))
        base4 = torch.from_numpy(np.stack([net4.base_p, net4.base_q], axis=1).reshape(-1)).to(dev)
        # X = interleaved [p_n, q_n] of load scenarios: base loads x U(0.7, 1.3) (data_generation.py:27-36)
        X4 = (base4[None, :] * (0.7 + 0.6 * torch.rand(E4, 66, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(4)))).float().contiguous()
        ring = DeviceReplayBuffer(2 * E4, {"v_pred": 33, "safety_penalty": 1}, device=dev)
        K4 = 40
        ev4 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K4)]
        for k in range(5):
            pred.predict(X4, want_vhat=False, want_penalty=False, sink=ring)
        for k in range(K4):
            flush.zero_()
            ev4[k][0].record(stream); pred.predict(X4, want_vhat=False, want_penalty=False, sink=ring); ev4[k][1].record(stream)
        torch.cuda.synchronize()
        ms4 = statistics.median(a.elapsed_time(b) for a, b in ev4)
        b4 = 66 * 4 + 33 * 4 + 4                                  # X row in, Vhat row + penalty into the ring
        config4 = {"workload": "predictor_penalty_to_replay_ring_262144_envs (BASELINE config 4)", "value": E4 / (ms4 * 1e-3),
                   "unit": "envs/s", "kernel": "k_predict (tcgen05 kind::tf32, 3xTF32, A operand in TMEM)", "kernel_ms_median": ms4,
                   "bytes_per_env": b4, "roofline_frac": b4 * E4 / (ms4 * 1e-3) / 1e9 / peaks()[0], "steps": K4}
        ring.close()

    t = torch.tensor([dev_ms, e2e_s, kern_ms, obs_extra[1] if obs_extra else 0.0, strong[2] if strong else 0.0,
                      rollout["acting"][1] if rollout else 0.0, rollout["recording"][1] if rollout else 0.0,
                      obs_extra[2] if obs_extra else 0.0, rollout["critic"][1] if rollout else 0.0],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s, kern_ms, obs_ms, strong_ms, roll_ms, rollrec_ms, obs_ring_ms, rollcrit_ms = (float(x) for x in t)
    stats = env.episode_stats(reduce=True)                     # the one NCCL collective (16 doubles)
    total_envs = E * world
    value = total_envs * K / (dev_ms * 1e-3)
    e2e = total_envs * Ke / e2e_s

    if rank == 0:
        peak, peak_src = peaks()
        achieved = B_ALG * E / (kern_ms * 1e-3) / 1e9
        cap = ncu_capture(E) if args.variant == "thread" else None
        cfg = make_config(args, world, state["timed_resets"] > 0)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "method": {"kernel_variant": args.variant, "actions": "resident in HBM (8 arrays cycled)",
                       "l2": "flushed before every timed step (256 MiB memset, untimed)" if not args.no_flush else "NOT flushed",
                       "timing": "CUDA events per step on the launching stream, summed; max over ranks",
                       "auto_resets_in_timed_region": state["timed_resets"], "wall_s_incl_flush": t_wall},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": E * 20 * 4, "d2h_bytes_per_step": E * 9,
                    "steps": Ke, "api": "BatchedFlexProvisionEnv.step_host -> fp_step_host (pinned host buffers)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": float(cap["dram_bytes_per_launch"]) if cap else None,
                         "kernel": {"thread": "k_env_t<STEP>", "warp": "k_env<STEP>"}[args.variant], "bytes_per_env_step": B_ALG,
                         "kernel_ms_median": kern_ms, "peak_source": peak_src,
                         "note": "latency-bound per warp, not HBM- or pipe-bound: see roofline_fp64 and DESIGN.md section 3"},
            "stats": {k: float(v) for k, v in stats.items()},
        }
        if cap is not None and clocks and clocks.get("sm_mhz"):
            # the same kernel against the fp64 pipe: lane-operations (DFMA/DADD/DMUL, one each) per launch from the ncu capture
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            pk = FP64_PEAK_LANE_OPS_PER_CLK_SM * sms * clocks["sm_mhz"] * 1e6
            ach = cap["fp64_lane_ops_per_launch"] / (kern_ms * 1e-3)
            line["roofline_fp64"] = {"bound": "fp64 pipe", "achieved_lane_ops": ach, "peak": pk, "unit": "lane-ops/s", "frac": ach / pk,
                                     "lane_ops_per_env_step": cap["fp64_lane_ops_per_env_step"],
                                     "fp32_lane_ops_per_env_step": cap["fp32_lane_ops_per_env_step"],
                                     "peak_source": f"{FP64_PEAK_LANE_OPS_PER_CLK_SM} lane-ops/clk/SM measured (profiles/r1_ubench_fp64_b200.txt) x {sms} SMs x sampled SM clock",
                                     "counts_source": "profiles/r2_step_kernel_traffic.json (ncu --set full)"}
        if obs_extra is not None:
            line["step_plus_get_obs_env_steps_per_s"] = obs_extra[0] * world / (obs_ms * 1e-3)
            line["step_plus_get_obs"] = {"api": "step(..., return_obs='ring') -> fp_step_ring (one launch)", "steps": 40,
                                         "ms_per_step": obs_ms / 40, "l2": "flushed before every step",
                                         "ring_only": {"api": "set_obs_history(False): the fp64 history ring is not pushed (device rollouts)",
                                                       "env_steps_per_s": obs_extra[0] * world / (obs_ring_ms * 1e-3),
                                                       "ms_per_step": obs_ring_ms / 40}}
        if rollout is not None:
            line["rollout_env_steps_per_s"] = rollout["acting"][0] * world / (roll_ms * 1e-3)
            line["rollout"] = {"loop": "k_policy (RNNAgent fc1-LayerNorm-ReLU-GRUCell-fc2 + tanh-Normal sampling, tcgen05) -> fp_step_ring "
                                       "(translate_action + step + get_obs push): model.py:213-254 with zero PCIe bytes per step",
                               "ms_per_step": roll_ms / 30, "launches_per_step": rollout["acting"][2], "steps": 30,
                               "with_transition_writes": {"env_steps_per_s": rollout["recording"][0] * world / (rollrec_ms * 1e-3),
                                                          "ms_per_step": rollrec_ms / 30, "launches_per_step": rollout["recording"][2],
                                                          "bytes_per_transition": 4 * sum(TRANSITION_FIELDS.values()),
                                                          "recorded_envs_per_step": E},
                               "with_critic": {"loop": "the whole train_process body (model.py:213-254): + value = critic(state, action) and next_value = "
                                                       "critic(next_state, a second sampled action) through k_critic (MLPCritic on tcgen05), every transition written",
                                               "env_steps_per_s": rollout["critic"][0] * world / (rollcrit_ms * 1e-3), "ms_per_step": rollcrit_ms / 30,
                                               "launches_per_step": rollout["critic"][2]},
                               "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "l2": "flushed before every step"}
        if strong is not None:
            line["config5_strong"] = {"workload": "fused_env_step_2^20_envs_total (BASELINE config 5, strong scaling: split over the run's GPUs)",
                                      "value": strong[0] * world * strong[1] / (strong_ms * 1e-3), "unit": UNIT, "scaling": "strong",
                                      "envs_per_gpu": strong[0], "steps": strong[1], "ms_per_step": strong_ms / strong[1],
                                      "roofline_frac_per_gpu": B_ALG * strong[0] * strong[1] / (strong_ms * 1e-3) / 1e9 / peak}
        if config2 is not None:
            line["config2"] = config2
        if config3 is not None:
            line["config3"] = config3
        if config4 is not None:
            line["config4"] = config4
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample = cpu_port_rate(prof, E, budget_s=12.0)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "reference_solver_probe": probe_reference_solver()}
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
