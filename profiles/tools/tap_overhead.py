"""Device time per graph-replayed step with episode taps off / 64 / 1,024 (dockauv_set_taps), alternated in one run:

    python profiles/tools/tap_overhead.py [--steps 208] [--rounds 3] [--out taps.json]

C2: SimpleDocking3d, 65,536 envs, through ``step`` (cached step graph).
C4: ObstaclesDocking3d, 64 rays, 3 synthetic spheres, 1,048,576 envs, through ``step`` and through
    ``rollout(use_graph=True)`` (16 steps per call).
Each (case, taps) cell: 20 warm-up steps, then CUDA events around `--steps` steps; the median over the rounds is
reported.  Prints one JSON document with the card name and power limit next to the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch  # noqa: E402

from gym_dockauv_b200 import envs  # noqa: E402
from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64  # noqa: E402

TAPS = (0, 64, 1024)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def set_taps(env, k):
    if k == 0:
        env.clear_taps()
    else:
        ids = torch.randperm(env.num_envs, generator=torch.Generator().manual_seed(k))[:k].tolist()
        env.set_taps(ids, 256)


def time_steps(env, how, steps, a, out):
    """ms of device time per step; `how` is "step" or "rollout" (graph replays in both)."""
    T = a.shape[0] if how == "rollout" else 1
    calls = max(1, steps // T)

    def call():
        if how == "rollout":
            env.rollout(a, *out, use_graph=True)
        else:
            env.step(a)

    for _ in range(max(1, 20 // T)):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (calls * T)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=208)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    cfg64 = dict(BASE_CONFIG)
    cfg64["radar"] = dict(RADAR_64)
    gen = torch.Generator(device="cuda").manual_seed(0)
    cases = []
    c2 = envs.SimpleDocking3d(BASE_CONFIG, num_envs=65536, seed=0)
    c2.reset()
    cases.append(("C2 step", c2, "step", torch.rand(65536, c2.n_actions, device="cuda", generator=gen) * 2 - 1, None))
    N, T = 1 << 20, 16
    c4 = envs.ObstaclesDocking3d(cfg64, num_envs=N, seed=0, n_synthetic_spheres=3)
    c4.reset()
    cases.append(("C4 step", c4, "step", torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1, None))
    out = (torch.zeros(T, N, c4.n_observations, device="cuda"), torch.zeros(T, N, dtype=torch.float64, device="cuda"),
           torch.zeros(T, N, dtype=torch.uint8, device="cuda"))
    cases.append(("C4 rollout", c4, "rollout", torch.rand(T, N, 6, device="cuda", generator=gen) * 2 - 1, out))
    ms = {name: {k: [] for k in TAPS} for name, *_ in cases}
    for _ in range(args.rounds):
        for name, env, how, a, o in cases:
            for k in TAPS:
                set_taps(env, k)
                ms[name][k].append(time_steps(env, how, args.steps, a, o))
    for _, env, *_ in cases:
        env.clear_taps()
    name, power = card()
    res = {"gpu": name, "power_limit": power, "steps_per_cell": args.steps, "rounds": args.rounds, "precision": "f64",
           "results": {}}
    for case in ms:
        med = {k: statistics.median(v) for k, v in ms[case].items()}
        res["results"][case] = {
            "ms_per_step": {str(k): round(med[k], 5) for k in TAPS},
            "overhead_us_per_step": {str(k): round(1e3 * (med[k] - med[0]), 2) for k in TAPS if k},
            "all_ms": {str(k): [round(x, 5) for x in v] for k, v in ms[case].items()}}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
