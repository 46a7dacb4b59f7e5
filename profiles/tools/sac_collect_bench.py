#!/usr/bin/env python
"""Collection throughput of SAC with the actor in the loop, three ways, on C2 (65,536 envs) and C4 (16,384, 131,072 and
1,048,576 envs), f64 handles, a 16-slot replay ring, T = 32 steps (a multiple of the slots), auto-reset:

  (a) ``DeviceReplayBuffer.collect(actor.act)``: one Python iteration per step, the example's PyTorch actor (SB3's SAC
      default: n_obs -> 256 -> 256 with ReLU, one Linear(256, 2 n_u) head, tanh-squashed Gaussian) between the steps;
  (b) ``DeviceReplayBuffer.collect_fused``: the same weights evaluated by the library's tensor-core actor kernel
      (bf16 operands, f32 accumulation) between the steps of one captured launch chain (dockauv_replay_collect);
  (c) ``env.rollout`` with actions known up front (dockauv_rollout), the open-loop ceiling.

    python profiles/tools/sac_collect_bench.py --out profiles/r02/sac_collect_b200.json

Each collection is timed with CUDA events around the call after one warm-up call of every path (the warm-up captures
the graphs); the three paths alternate in each round and the JSON keeps the median and every round.  The actor's time
per step is (b) minus (c) per step: both are graph replays without launch gaps, so the difference is the device time of
the actor launch of each step.  Achieved TFLOP/s = 2 (n_obs H + H^2 + 2 n_u H) per env x N / that time.  A fifth case,
C4 at 2,368 envs (148 CTAs of one warp, one 16-env tile each), bounds the per-launch cost of staging the weights
(every CTA reads and converts the ~313 KB of f32 weights once per launch).  The card's name and power limit are read in
the same run.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "examples"))
import torch  # noqa: E402

from gym_dockauv_b200 import envs  # noqa: E402
from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64  # noqa: E402
from gym_dockauv_b200.policy import FusedSquashedActor  # noqa: E402
from gym_dockauv_b200.replay import DeviceReplayBuffer  # noqa: E402
from sac_device_replay import Actor  # noqa: E402

CASES = (("C2", 65536), ("C4", 2368), ("C4", 16384), ("C4", 131072), ("C4", 1 << 20))
H, SLOTS = 256, 16


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                        f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, check=True)
    name, power = [x.strip() for x in r.stdout.strip().split(",")]
    return name, power


def make_env(config, N):
    if config == "C2":
        return envs.SimpleDocking3d(dict(BASE_CONFIG), num_envs=N, seed=0)
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    return envs.ObstaclesDocking3d(cfg, num_envs=N, seed=0, n_synthetic_spheres=3)


def actor_flops(n_obs, n_u):
    return 2 * (n_obs * H + H * H + 2 * n_u * H)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if args.steps % SLOTS:
        raise SystemExit(f"--steps must be a multiple of the {SLOTS} ring slots (one graph per call)")
    name, power = gpu_info()
    T, rows = args.steps, []
    for config, N in CASES:
        env = make_env(config, N)
        buf = DeviceReplayBuffer(env, SLOTS)
        buf.reset_env(seed=0)
        torch.manual_seed(0)
        n_obs, n_u = env.n_observations, env.n_actions
        actor = Actor(n_obs, n_u).to(env.device)
        w, b = actor.net[4].weight, actor.net[4].bias
        fused = FusedSquashedActor([actor.net[0], actor.net[2]], w[:n_u], b[:n_u], w[n_u:], b[n_u:])
        acts = torch.rand(T, N, n_u, device=env.device) * 2 - 1
        obs = torch.empty(T, N, n_obs, device=env.device)
        rew = torch.empty(T, N, dtype=env.dtype, device=env.device)
        done = torch.empty(T, N, dtype=torch.uint8, device=env.device)
        paths = {"a_collect": lambda: buf.collect(actor.act, T), "b_collect_fused": lambda: buf.collect_fused(fused, T),
                 "c_open_loop": lambda: env.rollout(acts, obs, rew, done)}
        for fn in paths.values():
            fn()
        ms = {k: [] for k in paths}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):
            for k, fn in paths.items():
                torch.cuda.synchronize()
                e0.record()
                fn()
                e1.record()
                e1.synchronize()
                ms[k].append(e0.elapsed_time(e1))
        med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
        actor_ms = (med["b_collect_fused"] - med["c_open_loop"]) / T
        flops = actor_flops(n_obs, n_u)
        row = dict(config=config, envs=N, n_obs=n_obs, n_u=n_u, hidden=H, slots=SLOTS,
                   env_steps_per_s={k: N * T / (v * 1e-3) for k, v in med.items()},
                   ms_per_collection=med, ms_per_collection_rounds=ms,
                   speedup_fused_over_collect=med["a_collect"] / med["b_collect_fused"],
                   fused_share_of_open_loop=med["c_open_loop"] / med["b_collect_fused"],
                   actor_ms_per_step=actor_ms, actor_flop_per_env=flops,
                   actor_tflops=flops * N / (actor_ms * 1e-3) / 1e12 if actor_ms > 0 else None,
                   graph_captures=buf.collect_captures())
        rows.append(row)
        print(json.dumps(row), flush=True)
        env.close()
        del buf, env, obs, rew, done, acts
        torch.cuda.empty_cache()
    res = dict(tool="profiles/tools/sac_collect_bench.py", gpu=name, power_limit=power, precision="f64", steps=T,
               timing="CUDA events around one collection of T steps per path, after a warm-up call of each; median of "
                      "rounds that alternate the three paths; actor_ms_per_step = (fused - open loop) / T",
               results=rows)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
