#!/usr/bin/env python
"""Cost of the scenario bank on the flagship workload: C4 (ObstaclesDocking3d, 64-ray radar, 5 capsules + 3 spheres,
1,048,576 envs, f64, auto-reset).

    python profiles/tools/scenario_bank_bench.py [--envs 1048576] [--steps 200] [--rounds 3] [--out FILE]

Cases: no bank, then uniform and weighted banks of 2^16 and 2^20 rows (drawn from the built-in distributions with
``ScenarioBank.from_builtin``; the weights are U(0.5, 1.5)).  Per case and round: the time per graph-replayed step (CUDA
events around `steps` steps of one action tensor, after a warm-up that reaches the steady episode-end rate), and the
launch times of a few timed steps (plain launches, whole batch on one stream: ``last_step_ms``), of which the last is the
episode-end launch.  The cases alternate within each round; the medians over the rounds are reported with the card's
name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        q = f"unknown ({e})"
    return q


def main():
    import numpy as np
    import torch
    from gym_dockauv_b200 import envs
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    from gym_dockauv_b200.scenario_bank import ScenarioBank
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--timed", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    cfg = dict(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    N = args.envs
    env = envs.ObstaclesDocking3d(cfg, num_envs=N, seed=0, n_synthetic_spheres=3)
    banks = {}
    for log2k in (16, 20):
        K = 1 << log2k
        banks[K] = (ScenarioBank.from_builtin(env, K, seed=log2k),
                    torch.rand(K, dtype=torch.float64, device=env.device, generator=torch.Generator(env.device).manual_seed(1)) + 0.5)
    cases = [("none", None, None)]
    for K, (b, w) in banks.items():
        cases += [(f"uniform_2^{K.bit_length() - 1}", b, None), (f"weighted_2^{K.bit_length() - 1}", b, w)]
    act = torch.empty(N, env.n_actions, device=env.device)
    gen = torch.Generator(device=env.device).manual_seed(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {name: dict(step_ms=[], episode_end_ms=[], launch_ms=[], ended_per_step=[]) for name, _, _ in cases}
    for rnd in range(args.rounds):
        for name, bank, w in cases:
            if bank is None:
                env.clear_scenario_bank()
            else:
                env.set_scenario_bank(bank, weights=w)
            env.reset(seed=rnd)
            for _ in range(args.warmup):      # from the synchronous start to the steady rate of episode ends
                env.step(act.uniform_(-1, 1, generator=gen))
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                env.step(act)
            e1.record()
            torch.cuda.synchronize()
            res[name]["step_ms"].append(e0.elapsed_time(e1) / args.steps)
            env.enable_timing(True)
            per, ended = [], []
            for _ in range(args.timed):
                env.step(act.uniform_(-1, 1, generator=gen))
                per.append(env.last_step_ms()[1])
                ended.append(env.last_list_counts()[1])
            env.enable_timing(False)
            per = np.array(per)
            res[name]["launch_ms"].append(per.mean(0).tolist())
            res[name]["episode_end_ms"].append(float(per[:, -1].mean()))
            res[name]["ended_per_step"].append(float(np.mean(ended)))
            print(json.dumps(dict(round=rnd, case=name, step_ms=res[name]["step_ms"][-1],
                                  episode_end_ms=res[name]["episode_end_ms"][-1],
                                  ended_per_step=res[name]["ended_per_step"][-1])), flush=True)
    summary = dict(card=card(), envs=N, config="C4 f64", steps=args.steps, rounds=args.rounds,
                   cases={name: dict(step_ms_median=float(np.median(r["step_ms"])),
                                     episode_end_ms_median=float(np.median(r["episode_end_ms"])),
                                     ended_per_step_median=float(np.median(r["ended_per_step"])), **r)
                          for name, r in res.items()})
    print(json.dumps({k: (v if k != "cases" else {c: {m: x[m] for m in ("step_ms_median", "episode_end_ms_median",
                                                                           "ended_per_step_median")} for c, x in v.items()})
                      for k, v in summary.items()}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    env.close()


if __name__ == "__main__":
    main()
