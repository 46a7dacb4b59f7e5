#!/usr/bin/env python
"""Benchmark of the gym_dockauv step hot path on B200 (BASELINE.json metric: env-steps/s, ObstaclesDocking3d,
BlueROV2, 64-ray radar, 5 capsules + 3 spheres).

    python bench.py [--gpus N] [--steps K] [--warmup W]                  # our arm (CUDA, through the C ABI)
    python bench.py --impl reference [--gpus N] --steps K --warmup W     # CPU arm: the oracle port on all host cores
    python bench.py --config C2|C3|C4 --scaling weak|strong ...          # the other BASELINE configs / sharding modes
    python bench.py ... --dump-outputs DIR                               # + the last timed step's outputs as DIR/*.npy

Default = config C4 with 1,048,576 envs PER GPU (weak scaling; at 8 GPUs this is config C5: 8M envs, auto-reset, one
NCCL all-reduce of the episode statistics per rollout).  `--scaling strong` shards 1,048,576 envs TOTAL over the ranks
(config C4 as BASELINE.json words it); a run with more than one rank also measures that strong-scaling point in a second
pass and reports it as `strong` next to the weak-scaling `value`.

One "step" = one batched env.step() over every env of the rank (three launches -- dynamics + cull + finish, rays +
finish, episode end -- for each half of the batch, the halves on two streams).  Rank 0 prints ONE JSON line.
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.  The per-step
working set (~0.9 GB at 1M envs) is far larger than L2 (126 MB), so no explicit L2 flush is needed at the default size
(stated in config.l2; smaller configs rotate through a pool of action tensors and say so).  Actions are synthetic
i.i.d. U(-1,1) float32, pre-generated on the device for `value`; the `e2e` number goes through env.step_host() with
pinned HOST actions in and HOST obs/reward/done out every step.
"""
import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HBM_FALLBACK_GBS = 6650.0     # /opt/skills/guides/B200_PROFILING.md fallback
FP64_NOMINAL_TFLOPS = 37.2    # 148 SMs x 64 FP64 FMA / clk x 2 x 1.965 GHz (SURVEY.md 8d)
N_SYNTH_SPHERES = 3

# BASELINE.json configs with the ALGORITHMIC figures of SURVEY.md 8(d), per env-step and split over the launches of the
# pipeline (DESIGN.md 5): dynamics = the 6-DOF integration + navigation errors + obs[0:16] + radar-free reward terms;
# cull_finish = body-collision tests + reward / done / counters; rays_* = n_rays x (rotate 25 + K_c x 33 + K_s x 10 +
# pool / OA 8) -- the contract's brute-force figure, PER ENV THE RAY LAUNCH VISITS: the culls are exact, an env with
# nothing in view needs no ray test, so the launch's algorithmic work is that figure times the listed fraction (read live
# from the library's work-list counter).  Bytes: every persistent item read once and written once, attributed to the
# launch that moves it (state / command / action / goal / obs[0:16] -> dynamics; obstacles, counters, reward, flags ->
# cull_finish; pooled ray cells -> rays_finish); their sum is the config's contract figure.
CONFIGS = {
    "C2": dict(scenario="SimpleDocking3d", vehicle="BlueROV2", envs=65536, radar64=False, n_synth=0, h=0.1,
               bytes=538, flops=2900, launch_flops=dict(dynamics=2900, episode_end=0),
               launch_bytes=dict(dynamics=538, episode_end=0),
               workload="C2: SimpleDocking3d, BlueROV2, 65,536 envs, dynamics + reward only (no obstacles: every ray "
                        "reads max_dist), random actions U(-1,1) f32, auto-reset"),
    "C3": dict(scenario="CapsuleCurrentDocking3d", vehicle="LAUV", envs=262144, radar64=False, n_synth=0, h=0.02,
               bytes=534, flops=7250, launch_flops=dict(dynamics=3050, cull_finish=35, rays_finish=4165, episode_end=0),
               launch_bytes=dict(dynamics=336, cull_finish=118, rays_finish=80, episode_end=0),
               workload="C3: CapsuleCurrentDocking3d, LAUV with ocean current, 262,144 envs, docking-capsule collision "
                        "checks, t_step_size 0.02 (the reference's integrator diverges at its stock 0.1 for this "
                        "vehicle, SURVEY.md 8c), random actions U(-1,1) f32, auto-reset"),
    "C4": dict(scenario="ObstaclesDocking3d", vehicle="BlueROV2", envs=1 << 20, radar64=True, n_synth=N_SYNTH_SPHERES, h=0.1,
               bytes=898, flops=17700, launch_flops=dict(dynamics=2900, cull_finish=205, rays_finish=14592, episode_end=0),
               launch_bytes=dict(dynamics=400, cull_finish=434, rays_finish=64, episode_end=0),
               workload="C4: ObstaclesDocking3d, BlueROV2, 64-ray radar, 5 capsules + 3 spheres, random actions "
                        "U(-1,1) f32, auto-reset of finished envs"),
}
def launch_names(c, n_launches):
    """Names of the launches of one step, from how many the library timed: obstacle-free scenarios are finished by the
    dynamics launch; with obstacles the cull + finish code normally runs inside the dynamics launch (three launches), as a
    launch of its own otherwise (four)."""
    if c["scenario"] == "SimpleDocking3d":
        return ("dynamics", "episode_end")
    if n_launches == 3:
        return ("dynamics_cull_finish", "rays_finish", "episode_end")
    return ("dynamics", "cull_finish", "rays_finish", "episode_end")


def launch_figure(c, key, name):
    """Algorithmic flops / bytes per env of one launch (the fused launch carries the sum of its two parts)."""
    d = c[key]
    if name == "dynamics_cull_finish":
        return d["dynamics"] + d["cull_finish"]
    return d[name]


def workload_config(c):
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = dict(BASE_CONFIG)
    cfg["vehicle"] = c["vehicle"]
    cfg["t_step_size"] = c["h"]
    if c["radar64"]:
        cfg["radar"] = dict(RADAR_64)
    return cfg


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def kernel_source_hash():
    """sha256 over the CUDA sources: the committed ncu figures are only quoted while the kernels they came from are
    the ones being run."""
    h = hashlib.sha256()
    for f in sorted(glob.glob(os.path.join(ROOT, "gym_dockauv_b200", "csrc", "*"))):
        with open(f, "rb") as fh:
            h.update(os.path.basename(f).encode())
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_figures(config_name):
    """Per-launch DRAM traffic and FP64-pipe utilisation from the committed `ncu --set full` capture (written by
    profiles/tools/ncu_launch_json.py); None when the capture belongs to other kernel sources."""
    path = os.path.join(ROOT, "profiles", "r02", f"ncu_per_launch_{config_name}.json")
    try:
        with open(path) as f:
            d = json.load(f)
    except Exception:
        return None, "no committed capture for this config"
    if d.get("kernel_source_hash") != kernel_source_hash():
        return None, f"{os.path.relpath(path, ROOT)} was captured from other kernel sources (stale) -- not quoted"
    return d, os.path.relpath(path, ROOT)


def recorded_numpy_baseline(config_name):
    try:
        with open(os.path.join(ROOT, "profiles", "r02", "reference_numpy_cpu.json")) as f:
            d = json.load(f)
    except Exception:
        return None
    case = d["cases"].get("C4" if config_name == "C4" else "C1")
    if case is None:
        return None
    return {"kind": d["kind"], "unit": d["unit"], "value": case["all_cores"]["value"], "cores": case["all_cores"]["cores"],
            "value_one_core": case["one_process"]["value"], "workload": case["workload"], "cpu": d["cpu"], "date": d["date"],
            "how": "unmodified /root/reference (numpy) timed in the build container by profiles/tools/time_reference_numpy.py; "
                   "/root/reference does not exist on the GPU box, so this figure is recorded, not live"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.rows = index, None, []

    def mark(self):
        """Index of the next sample: brackets the timed region."""
        return len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self, first=0, last=None):
        """Summary of the samples [first, last) (default: all); the timed region of a short run can fall between two
        20 ms samples, so the caller passes the window from the start of the timed region to the end of the measurement
        passes that follow it under the same load."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[first:last]:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for k, nme in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """Host threads this process may use.  torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm runs on rank 0
    alone while the other ranks exit, so it takes every core of its affinity mask and passes the count explicitly."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def bind_to_gpu_numa_node(local_rank):
    """Pins the process to the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned host memory is allocated,
    so that first-touch places the step_host staging buffers on the GPU's NUMA node.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = os.sched_getaffinity(0)
        pick = sorted(cpus & allowed)
        if pick:
            os.sched_setaffinity(0, pick)
            return {"cpus": f"{pick[0]}-{pick[-1]} ({len(pick)})", "source": "nvmlDeviceGetCpuAffinity"}
        return {"cpus": None, "source": "NVML affinity outside the allowed cpuset; left unchanged"}
    except Exception as ex:  # noqa: BLE001
        return {"cpus": None, "source": f"unavailable ({type(ex).__name__})"}


def cpu_port_rate(c, n_envs, seconds, n_threads, steps_cap=10 ** 9, warmup=1):
    """Times the oracle port (oracle/dockauv_oracle.c, OpenMP over envs) on this host's cores."""
    from oracle import oracle as orc
    cfg = workload_config(c)
    bo = orc.BatchOracle(cfg, c["scenario"], n_envs, seed=0, n_extra_spheres=c["n_synth"], n_threads=n_threads)
    n_u = bo.P.n_u
    rng = np.random.default_rng(1)
    pool = [rng.uniform(-1, 1, (n_envs, n_u)).astype(np.float32) for _ in range(4)]
    for i in range(warmup):
        bo.step(pool[i % 4])
    t0 = time.perf_counter()
    k = 0
    while k < steps_cap and (time.perf_counter() - t0 < seconds or k < 2):
        bo.step(pool[k % 4])
        k += 1
    dt = time.perf_counter() - t0
    return n_envs * k / dt, k, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import oracle as orc
    c = CONFIGS[args.config]
    n = args.ref_envs
    threads = host_threads()
    cfg = workload_config(c)
    bo = orc.BatchOracle(cfg, c["scenario"], n, seed=0, n_extra_spheres=c["n_synth"], n_threads=threads)
    n_u = bo.P.n_u
    rng = np.random.default_rng(1)
    pool = [rng.uniform(-1, 1, (n, n_u)).astype(np.float32) for _ in range(4)]
    for i in range(args.warmup):
        bo.step(pool[i % 4])
    t0 = time.perf_counter()
    for k in range(args.steps):
        bo.step(pool[k % 4])
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    line = {
        "impl": "reference", "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": c["workload"],
                   "envs_per_step": n, "sample": f"{n} envs per step (bounded sample of the {c['envs']:,}-env workload)"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{n} envs x {args.steps} steps, oracle/dockauv_oracle.c with OpenMP on {threads} threads "
                                   f"(num_threads passed explicitly; rank 0 only, the other ranks exit)"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    nb = recorded_numpy_baseline(args.config)
    if nb:
        line["cpu_baseline_numpy"] = nb
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 << 20


def last_step_outputs(out, n):
    """Host copies of what env.step returned in the last timed step (obs, reward, done and the info arrays) for a fixed,
    seeded sample of envs sized so that every file together stays within DUMP_BYTES (all envs when they fit); integer
    and flag arrays become float64 / float32.  terminal_observation, episode_return and episode_length are only defined
    for envs whose episode ended in that step, so their other rows are zeroed: what a layout leaves there is not an output."""
    import torch
    obs, reward, done, info = out
    cols = {"obs": obs, "reward": reward, "done": done, **info}
    per_env = 8 + sum(t[0].numel() * 8 for t in cols.values())      # bound: every value as float64, plus env_index
    k = min(n, DUMP_BYTES // per_env)
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    rows = torch.as_tensor(idx, device=obs.device)
    arrays = {"env_index": idx.astype(np.float64)}
    ended = done[rows].bool()
    for name, t in cols.items():
        t = t[rows]
        if name in ("terminal_observation", "episode_return", "episode_length"):
            t = t * ended.view(-1, *([1] * (t.dim() - 1))).to(t.dtype)
        if not t.is_floating_point():
            t = t.to(torch.float32 if name in ("done", "cond_bits") else torch.float64)
        arrays[name] = t.cpu().numpy()
    return arrays


def timed_steps(env, pool, steps, dev):
    """K steps bracketed by CUDA events on the launching stream; returns (total ms, per-step ms array)."""
    import torch
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for k in range(steps):
        env.step(pool[k % len(pool)])
        evs[k + 1].record()
    torch.cuda.synchronize(dev)
    return evs[0].elapsed_time(evs[-1]), np.array([evs[k].elapsed_time(evs[k + 1]) for k in range(steps)])


def run_ours(args, rank, world, local_rank):
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {"cpus": None, "source": "disabled"}
    import torch
    import torch.distributed as dist
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.params import N_STATS, STAT_NAMES

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL writes its version banner (and any debug output) to STDOUT by default; stdout carries only the one
        # JSON line, so NCCL's log goes to stderr
        # (NCCL honours NCCL_DEBUG_FILE only above the VERSION level, the image's default)
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", ""):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    c = CONFIGS[args.config]
    cfg = workload_config(c)
    if args.envs_per_gpu > 0:
        N = args.envs_per_gpu
    elif args.scaling == "strong":
        N = c["envs"] // world
    else:
        N = c["envs"]
    esz = 8 if args.precision == "f64" else 4

    def make_env(n, id0):
        e = envs.SCENARIOS[c["scenario"]](cfg, num_envs=n, device=dev, precision=args.precision, seed=args.seed,
                                          env_id0=id0, n_synthetic_spheres=c["n_synth"], layout=args.layout)
        e.reset()
        return e

    env = make_env(N, rank * N)
    # a pool of action tensors: the timed loop never reads the same actions twice in a row; with pool_bytes >> L2 the
    # inputs of small configs do not stay L2-resident either
    n_pool = args.action_pool if N * env.n_actions * 4 * args.action_pool <= (2 << 30) else max(4, (2 << 30) // (N * env.n_actions * 4))
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = [torch.rand(N, env.n_actions, device=dev, generator=gen) * 2 - 1 for _ in range(n_pool)]
    pool_mb = N * env.n_actions * 4 * n_pool / 1e6

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()       # running well before the timed region (nvidia-smi needs ~0.1 s to deliver its first sample)
    # burn-in: brings the batch from "every env just reset" to a mixed episode-age distribution (episodes last
    # ~100 steps under random actions), so the timed steps see the steady-state mix of ray hits and resets
    for k in range(args.burn_in):
        env.step(pool[k % len(pool)])
    for k in range(args.warmup):
        env.step(pool[k % len(pool)])
    side = torch.cuda.Stream(dev)
    if world > 1:
        # warm-up of the collective too (the first all-reduce of a communicator pays its lazy set-up: ~1.4 ms at 4 GPUs), on
        # the stream the timed ones use
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                dist.all_reduce(env.stats_tensor().clone())
        torch.cuda.current_stream(dev).wait_stream(side)
    env.clear_stats()
    barrier()
    clk_first = sampler.mark()
    launches0 = env.launch_count()
    # ---- the timed region: K steps; one statistics all-reduce per rollout on a side stream (SURVEY.md 8e), at least one
    rollout = max(1, min(args.rollout, args.steps))
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    reduced, n_reduces = None, 0
    evs[0].record()
    for k in range(args.steps):
        out = env.step(pool[k % len(pool)])
        evs[k + 1].record()
        if world > 1 and (k + 1) % rollout == 0:
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                local = env.stats_tensor().clone()      # folds the per-CTA replicas on the side stream first
                reduced = local.clone()
                dist.all_reduce(reduced)
            n_reduces += 1
    torch.cuda.current_stream(dev).wait_stream(side)
    ev_end = torch.cuda.Event(enable_timing=True)      # after the join with the side stream: the last all-reduce is inside the span
    ev_end.record()
    barrier()
    clk_timed_end = sampler.mark()
    if args.dump_outputs and rank == 0:
        # the step outputs are views of buffers the passes below overwrite: copied here, written at the end
        dumped = last_step_outputs(out, N)
    total_ms = evs[0].elapsed_time(ev_end)
    step_ms = np.array([evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps)])
    launches = env.launch_count() - launches0
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    stats = env.get_stats()
    # the reduced vector of the last all-reduce must be the sum of the rank-local vectors it was made from
    allreduce_check = None
    if world > 1 and reduced is not None:
        gathered = [torch.zeros(N_STATS, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(gathered, local)
        total = torch.stack(gathered).sum(0)
        ok = bool(torch.allclose(total, reduced, rtol=1e-12, atol=0.0))
        allreduce_check = {"equals_sum_of_rank_vectors": ok,
                           "reduced": {k: float(reduced[i]) for i, k in enumerate(STAT_NAMES)},
                           "rank0_local_env_steps": float(gathered[0][STAT_NAMES.index("env_steps")])}

    # ---- per-launch durations (CUDA events recorded by the library between the launches of a step, on the launching
    # stream), in a separate short pass so that the marks do not sit inside the timed region above
    env.enable_timing(True)
    per_launch = []
    for k in range(min(32, args.steps)):
        env.step(pool[k % len(pool)])
        per_launch.append(env.last_step_ms()[1])
    env.enable_timing(False)
    launch_ms = np.array(per_launch).mean(axis=0) if per_launch and per_launch[0] else np.zeros(0)
    n_listed, n_ended = env.last_list_counts()      # work-list lengths of the last step
    clocks = None
    if rank == 0:
        time.sleep(0.05)
        clocks = sampler.stop(clk_first, None)
        clocks["samples_inside_timed_region"] = max(0, clk_timed_end - clk_first)
        clocks["window"] = "timed region + the per-launch timing pass that follows it (same kernels, same load)"

    # ---- end to end through the public API with host buffers (rank-local, then max over ranks)
    e2e_steps = max(3, min(args.e2e_steps, args.steps))
    host_pool = [torch.empty(N, env.n_actions, dtype=torch.float32).pin_memory() for _ in range(2)]
    for hp, dp in zip(host_pool, pool):
        hp.copy_(dp)
    host_np = [hp.numpy() for hp in host_pool]
    env.step_host(host_np[0])
    env.step_host(host_np[1])
    barrier()
    t0 = time.perf_counter()
    sink = 0.0
    for k in range(e2e_steps):
        o, r, d, _ = env.step_host(host_np[k % 2])
        sink += float(r[0]) + float(o[0, 0]) + float(d[0])      # results really are in host memory
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s_max = float(t.item())
    h2d = N * env.n_actions * 4
    d2h = N * (env.n_observations * 4 + esz + 1 + 1)
    # ---- the copy ceiling of that path: the same bytes as plain pinned cudaMemcpyAsync, H2D and D2H on two streams,
    # every rank at the same time (what the PCIe links and host memory of this box give with no kernel at all)
    hb_in = torch.empty(h2d, dtype=torch.uint8).pin_memory()
    hb_out = torch.empty(d2h, dtype=torch.uint8).pin_memory()
    db_in = torch.empty(h2d, dtype=torch.uint8, device=dev)
    db_out = torch.empty(d2h, dtype=torch.uint8, device=dev)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def copy_round():
        with torch.cuda.stream(s_in):
            db_in.copy_(hb_in, non_blocking=True)
        with torch.cuda.stream(s_out):
            hb_out.copy_(db_out, non_blocking=True)
    copy_round()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        copy_round()
    torch.cuda.synchronize(dev)
    copy_s = time.perf_counter() - t0
    t = torch.tensor([copy_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    copy_s_max = float(t.item())
    env.close()
    del pool, env

    # ---- strong-scaling point of the same run (config as BASELINE.json words it: the config's envs TOTAL, sharded)
    strong = None
    if world > 1 and args.scaling == "weak" and args.envs_per_gpu <= 0 and not args.no_strong_pass:
        Ns = c["envs"] // world
        env_s = make_env(Ns, rank * Ns)
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        pool_s = [torch.rand(Ns, env_s.n_actions, device=dev, generator=gen) * 2 - 1 for _ in range(args.action_pool)]
        for k in range(args.burn_in + args.warmup):
            env_s.step(pool_s[k % len(pool_s)])
        barrier()
        ms_s, _ = timed_steps(env_s, pool_s, args.steps, dev)
        t = torch.tensor([ms_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        strong = {"scaling": "strong", "envs_total": Ns * world, "envs_per_gpu": Ns, "steps": args.steps,
                  "ms_per_step": float(t.item()) / args.steps, "value": Ns * world * args.steps / (float(t.item()) * 1e-3),
                  "unit": "env-steps/s", "note": "second pass of the same run: the config's envs TOTAL sharded over the "
                                                 "ranks (BASELINE.json configs[3]); the headline `value` is weak scaling"}
        env_s.close()

    if rank == 0:
        value = world * N * args.steps / (total_ms_max * 1e-3)
        kern_ms = float(step_ms.mean())
        per_gpu_rate = N / (kern_ms * 1e-3)
        hbm_peak, hbm_src = measured_hbm_peak()
        fp64_peak = fp32_peak = None
        try:
            import ctypes as C
            from gym_dockauv_b200 import _capi
            a, b = C.c_double(), C.c_double()
            _capi.check(_capi.load().dockauv_measure_peaks(local_rank, C.byref(a), C.byref(b), None))
            fp64_peak, fp32_peak = a.value, b.value
        except Exception as ex:  # noqa: BLE001
            print(f"peak measurement failed: {ex}", file=sys.stderr)
        pipe_name = "fp64" if args.precision == "f64" else "fp32"
        pipe_peak = fp64_peak if args.precision == "f64" else fp32_peak
        names = launch_names(c, len(launch_ms))[:len(launch_ms)]
        launches_ms = {n: float(v) for n, v in zip(names, launch_ms)}
        dominant = names[int(np.argmax(launch_ms))] if len(launch_ms) else None
        ncu, ncu_src = ncu_figures(args.config)
        ncu_ok = ncu is not None and args.precision == ncu.get("precision", "f64") and dominant in ncu.get("launches", {})
        pipe_peak_source = ("dockauv_measure_peaks: 8-chain FMA micro-kernel on this GPU, live (MEASURED_PEAKS.json "
                            f"carries no FP64 figure; nominal {FP64_NOMINAL_TFLOPS} TFLOP/s at 1.965 GHz)")
        roofline = {}
        listed_frac = n_listed / N
        roofline["work_lists"] = {"listed_frac": listed_frac, "ended_frac": n_ended / N,
                                  "note": "envs with an obstacle in view (visited by the ray launch) / envs whose episode "
                                          "ended, in the last step"}
        if dominant is not None and pipe_peak:
            dms = launches_ms[dominant]
            units = N * (listed_frac if dominant.startswith("rays") else 1.0)      # envs the launch has algorithmic work for
            l_flops, l_bytes = launch_figure(c, "launch_flops", dominant), launch_figure(c, "launch_bytes", dominant)
            ach = l_flops * units / (dms * 1e-3) / 1e12
            ach_gbs = l_bytes * N / (dms * 1e-3) / 1e9
            # the binding ceiling of the dominant launch: its algorithmic intensity against the machine balance of the two
            # measured peaks (the fused dynamics + cull launch: 3,105 flop per 834 B = 3.7 flop/B against 5.2 -> HBM; the
            # dynamics launch alone, 7.3 flop/B, and the ray launch -> the FP64 pipe)
            intensity = l_flops * units / (l_bytes * N) if l_bytes else float("inf")
            balance = pipe_peak * 1e12 / (hbm_peak * 1e9)
            fp = {"algorithmic_flops_per_env": l_flops, "envs_with_work_per_launch": units, "achieved": ach, "peak": pipe_peak,
                  "unit": "TFLOP/s", "frac": ach / pipe_peak,
                  "frac_of_nominal": ach / FP64_NOMINAL_TFLOPS if pipe_name == "fp64" else None,
                  "executed_pipe_frac": (ncu["launches"][dominant].get("fp64_pipe_pct", 0.0) / 100.0) if ncu_ok else None,
                  "peak_source": pipe_peak_source}
            hbm = {"algorithmic_bytes_per_env": l_bytes, "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s",
                   "frac": ach_gbs / hbm_peak, "peak_source": hbm_src}
            binding = hbm if intensity < balance else fp
            roofline.update({
                "bound": "hbm" if intensity < balance else pipe_name,
                "achieved": binding["achieved"], "peak": binding["peak"], "unit": binding["unit"], "frac": binding["frac"],
                "peak_source": binding["peak_source"],
                "kernel": dominant, "kernel_ms": dms,
                "intensity_flop_per_byte": intensity, "machine_balance_flop_per_byte": balance,
                "traffic": (ncu["launches"][dominant]["dram_bytes_per_env"] * N) if ncu_ok else None,
                "traffic_source": ncu_src,
                pipe_name: fp, "hbm": hbm,
                "how": "achieved = algorithmic bytes (flops) of the launch x envs per launch / its CUDA-event duration, measured "
                       "live between the launches of a step on the launching stream; the whole batch in one stream for "
                       "this pass (the timed region steps it as two halves on two streams); bound = whichever ceiling the "
                       "launch's algorithmic intensity puts first"})
        step_tf = per_gpu_rate * c["flops"] / 1e12
        step_gbs = per_gpu_rate * c["bytes"] / 1e9
        roofline["step"] = {"ms": kern_ms, "launches_ms": launches_ms,
                            "flops_per_env_step": c["flops"], "bytes_per_env_step": c["bytes"],
                            "fp_achieved_tflops": step_tf, "fp_frac": (step_tf / pipe_peak) if pipe_peak else None,
                            "hbm_achieved_gbs": step_gbs, "hbm_frac": step_gbs / hbm_peak,
                            "traffic": (ncu["step_dram_bytes_per_env"] * N) if ncu_ok else None,
                            "executed_pipe_frac_time_weighted": ncu.get("fp64_pipe_frac_time_weighted") if ncu_ok else None,
                            "note": "algorithmic figures of SURVEY.md 8(d) over the whole step; fp_frac counts the contract's "
                                    "brute-force 64 x 8 ray tests, most of which the culls skip, so it can exceed what the "
                                    "pipe executes -- executed_pipe_frac is the hardware figure"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)        # the CPU baseline takes every host core, not just the GPU's NUMA node
            threads = host_threads()
            rate, k_cpu, dt_cpu = cpu_port_rate(c, args.ref_envs, args.cpu_seconds, threads)
            cpu = {"value": rate, "unit": "env-steps/s", "cores": threads, "kind": "port",
                   "sample": f"{args.ref_envs} envs x {k_cpu} steps ({dt_cpu:.1f} s) of the same workload, "
                             f"oracle/dockauv_oracle.c with OpenMP on {threads} threads"}
        e2e_value = world * N * e2e_steps / e2e_s_max
        copy_value = world * N * e2e_steps / copy_s_max
        line = {
            "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": c["workload"], "name": args.config,
                       "envs_per_gpu": N, "envs_total": world * N, "layout": args.layout, "burn_in_steps": args.burn_in,
                       "rollout_steps": rollout, "stats_allreduces": n_reduces,
                       "l2": (f"working set per step ~{N * (c['bytes'] + 350) / 1e9:.2f} GB per GPU vs 126 MB L2; actions rotate "
                              f"through a pool of {n_pool} tensors ({pool_mb:.0f} MB); no explicit flush"),
                       "host_affinity": numa},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "api": "env.step_host (dockauv_step_host)",
                    "copy_ceiling": {"value": copy_value, "unit": "env-steps/s",
                                     "gbs_per_gpu": (h2d + d2h) * e2e_steps / copy_s_max / 1e9,
                                     "how": "the same H2D + D2H bytes per step as plain pinned cudaMemcpyAsync on two "
                                            "streams, all ranks at once, no kernel"},
                    "frac_of_copy_ceiling": e2e_value / copy_value},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "episode_stats": {k: stats[k] for k in ("episodes", "sum_return", "sum_length", "done_collision",
                                                    "done_out_att", "env_steps")},
        }
        if allreduce_check is not None:
            line["stats_allreduce"] = allreduce_check
        if strong is not None:
            line["strong"] = strong
        if cpu is not None:
            line["cpu_baseline"] = cpu
        nb = recorded_numpy_baseline(args.config)
        if nb:
            line["cpu_baseline_numpy"] = nb
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C4", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="override the config's batch size")
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--layout", default="auto", choices=["auto", "thread_per_env", "warp_rays", "pipeline"])
    ap.add_argument("--burn-in", type=int, default=128)
    ap.add_argument("--rollout", type=int, default=128)
    ap.add_argument("--action-pool", type=int, default=64)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--ref-envs", type=int, default=16384)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong-pass", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (obs, reward, done, info arrays; rank 0's envs, a fixed "
                         "sample of at most 64 MB) as DIR/<name>.npy, to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
