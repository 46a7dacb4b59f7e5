"""One line per library variant: device-timed step of the C4 workload at 1M envs (40 steps after a burn-in), its
per-launch CUDA-event times, the C2 workload at 65,536 envs and SimpleDocking3d at 1M envs; then, with their per-launch
times too, ObstaclesDocking3d at 1M envs with the most float obstacle records a handle can have (8 capsules + 8 spheres)
and with coordinates too large for float records (max_dist_from_goal = 2500: exact culls).

    DOCKAUV_LIB=.../libdockauv_<tag>.so python profiles/tools/ab_step.py [tag]
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
import torch
from gym_dockauv_b200 import envs
from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64

tag = sys.argv[1] if len(sys.argv) > 1 else os.path.basename(os.environ.get("DOCKAUV_LIB", "default"))
quick = "--quick" in sys.argv


def timed(env, pool, steps, burn):
    for k in range(burn):
        env.step(pool[k % len(pool)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        env.step(pool[k % len(pool)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


cfg = dict(BASE_CONFIG)
cfg["radar"] = dict(RADAR_64)
N = 1 << 20
gen = torch.Generator(device="cuda").manual_seed(1)
pool = [torch.rand(N, 6, device="cuda", generator=gen) * 2 - 1 for _ in range(8)]


def step_and_launches(env):
    """best of two 40-step windows after a burn-in, and the mean per-launch times of 16 timed steps"""
    env.reset()
    ms = min(timed(env, pool, 40, 140), timed(env, pool, 40, 0))
    env.enable_timing(True)
    per = []
    for k in range(16):
        env.step(pool[k % 8])
        per.append(env.last_step_ms()[1])
    env.enable_timing(False)
    env.close()
    return ms, " ".join(f"{x * 1e3:.0f}" for x in np.array(per).mean(axis=0))


ms_c4, per = step_and_launches(envs.ObstaclesDocking3d(cfg, num_envs=N, seed=0, n_synthetic_spheres=3))
out = f"{tag:14s} C4 1M {ms_c4:.4f} ms ({N / ms_c4 * 1e3:.3e}/s) launches {per} us"
if not quick:
    env = envs.SimpleDocking3d(dict(BASE_CONFIG), num_envs=N, seed=0)
    env.reset()
    ms_s = timed(env, pool, 40, 60)
    env.close()
    n2 = 65536
    pool2 = [p[:n2].contiguous() for p in pool]
    env = envs.SimpleDocking3d(dict(BASE_CONFIG), num_envs=n2, seed=0)
    env.reset()
    ms_c2 = timed(env, pool2, 400, 100)
    env.close()
    out += f" | Simple 1M {ms_s:.4f} ms | C2 65536 {ms_c2 * 1e3:.1f} us ({n2 / ms_c2 * 1e3:.3e}/s)"
    ms_88, per = step_and_launches(envs.ObstaclesDocking3d(cfg, num_envs=N, seed=0, n_synthetic_spheres=8, n_capsules=8))
    out += f" | 8+8 1M {ms_88:.4f} ms launches {per} us"
    cfg_far = dict(cfg, max_dist_from_goal=2500.0)
    ms_far, per = step_and_launches(envs.ObstaclesDocking3d(cfg_far, num_envs=N, seed=0, n_synthetic_spheres=3))
    out += f" | 2.5km 1M {ms_far:.4f} ms launches {per} us"
print(out, flush=True)
