#!/usr/bin/env python
"""Collection throughput of PPO rollouts with the policy in the loop, three ways, on C2 (65,536 envs) and C4 (16,384,
131,072 and 1,048,576 envs), f64 handles, T = 64 steps, auto-reset:

  (a) ``DeviceRolloutBuffer.collect(net.act)``: one Python iteration per step, a PyTorch actor-critic between the steps;
  (b) ``DeviceRolloutBuffer.collect_fused``: the same networks evaluated by the library's policy kernel between the
      steps of one captured rollout (dockauv_rollout_policy), plus the bootstrap value;
  (c) ``DeviceRolloutBuffer.collect_open_loop``: random actions known up front (dockauv_rollout), the ceiling.

    python profiles/tools/policy_rollout_bench.py --out profiles/r02/policy_rollout_b200.json

The policy is the example's ActorCritic (SB3's MlpPolicy shape: separate 64-wide pi and vf nets, Tanh).  Each rollout
is timed with CUDA events around the call after one warm-up rollout of every path (the warm-up captures the graphs);
the three paths alternate in each of the rounds and the JSON keeps the median and every round.  The policy launches'
time per step is (b) minus (c) per step: the graph replays of both leave no launch gaps, so the difference is the
device time of the policy launch of each step (the bootstrap launch is spread over the T steps).  It is set against the
FP32 FMA bound of the policy's arithmetic, 2 x FMAs per env x N / the FP32 rate the library measures in the same run
(dockauv_measure_peaks).  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "examples"))
import torch  # noqa: E402

from gym_dockauv_b200 import _capi, envs  # noqa: E402
from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64  # noqa: E402
from gym_dockauv_b200.policy import FusedActorCritic  # noqa: E402
from gym_dockauv_b200.rollout import DeviceRolloutBuffer  # noqa: E402
from ppo_device_rollout import ActorCritic  # noqa: E402

CASES = (("C2", 65536), ("C4", 16384), ("C4", 131072), ("C4", 1 << 20))


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


def policy_fmas(n_obs, H, n_u):
    return n_obs * H + H * H + H * n_u + n_obs * H + H * H + H


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.cuda.current_device()
    fp32 = C.c_double()
    _capi.check(_capi.load().dockauv_measure_peaks(dev, None, C.byref(fp32), None))
    name, power = gpu_info()
    T, rows = args.steps, []
    for config, N in CASES:
        env = make_env(config, N)
        buf = DeviceRolloutBuffer(env, T)
        buf.reset_env(seed=0)
        torch.manual_seed(0)
        net = ActorCritic(env.n_observations, env.n_actions).to(env.device)
        fused = FusedActorCritic([net.pi[0], net.pi[2], net.pi[4]], [net.v[0], net.v[2], net.v[4]], net.log_std)
        paths = {"a_collect": lambda: buf.collect(net.act), "b_collect_fused": lambda: buf.collect_fused(fused),
                 "c_collect_open_loop": lambda: buf.collect_open_loop()}
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
        policy_ms = (med["b_collect_fused"] - med["c_collect_open_loop"]) / T
        fmas = policy_fmas(env.n_observations, 64, env.n_actions)
        bound_ms = 2.0 * fmas * N / (fp32.value * 1e12) * 1e3
        row = dict(config=config, envs=N, n_obs=env.n_observations, n_u=env.n_actions, hidden=64,
                   env_steps_per_s={k: N * T / (v * 1e-3) for k, v in med.items()},
                   ms_per_rollout=med, ms_per_rollout_rounds=ms,
                   speedup_fused_over_collect=med["a_collect"] / med["b_collect_fused"],
                   fused_share_of_open_loop=med["c_collect_open_loop"] / med["b_collect_fused"],
                   policy_ms_per_step=policy_ms, policy_fma_per_env=fmas, policy_fp32_bound_ms=bound_ms,
                   policy_share_of_fp32_bound=bound_ms / policy_ms if policy_ms > 0 else None,
                   graph_captures=env.rollout_policy_captures())
        rows.append(row)
        print(json.dumps(row), flush=True)
        env.close()
        del buf, env
        torch.cuda.empty_cache()
    res = dict(tool="profiles/tools/policy_rollout_bench.py", gpu=name, power_limit=power, precision="f64", steps=T,
               fp32_tflops_measured=fp32.value,
               timing="CUDA events around one rollout of T steps per path, after a warm-up rollout of each; median of "
                      "rounds that alternate the three paths; policy_ms_per_step = (fused - open loop) / T",
               results=rows)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
