#!/usr/bin/env python
"""Times the fused replay sampler (dockauv_replay_sample, one kernel) against the same minibatch sampling written as
plain torch indexing (randint, index arithmetic, gathers of obs / actions / reward / done, torch.where for the next
observation, casts), on a C4-shaped ring: n_obs 32, n_u 6, f64 rewards, N = 65,536 envs, S = 64 slots.  Each
observation array of the ring is 0.54 GB, far above the 126 MB L2, so the gathered rows come from HBM.

    python profiles/tools/replay_sample_bench.py --out profiles/r02/replay_sample_b200.json

Both paths are timed with CUDA events around many calls after a warm-up, in rounds that alternate the two paths; the
JSON holds per batch size the µs per call of both (median of the rounds and every round), kernel launches per call
(counted with torch.profiler in a separate pass), algorithmic bytes per call (from the shapes), the fused kernel's
share of HBM bandwidth (7.7 TB/s, data sheet of the HGX B200, one GPU), and the card's name and power limit.  Before
timing, the fused rows are checked bit for bit against the torch gathers at the same indices.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch  # noqa: E402

from gym_dockauv_b200 import _capi  # noqa: E402
from gym_dockauv_b200.params import F64, DockauvReplayRing, DockauvReplaySample  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
BATCHES = (256, 4096, 65536, 1 << 20)
CALLS = {256: 4000, 4096: 4000, 65536: 1000, 1 << 20: 100}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                        f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, check=True)
    name, power = [x.strip() for x in r.stdout.strip().split(",")]
    return name, power


def bytes_per_row(n_obs, n_u, reward_bytes):
    """Reads: obs row, next-observation row (obs or terminal_obs), action row, reward, done flag.  Writes: obs and next
    observation rows, action row, reward and done as float32."""
    return 2 * 4 * n_obs + 4 * n_u + reward_bytes + 1 + 2 * 4 * n_obs + 4 * n_u + 4 + 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--slots", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lib = _capi.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    S, N, n_obs, n_u = args.slots, args.envs, 32, 6
    T = 10 * S + 5                       # steps since the ring was reset: full ring, wrapped
    n_valid = S - 1
    t_first = T - n_valid
    g = torch.Generator(device=dev).manual_seed(0)
    obs = torch.randn(S, N, n_obs, device=dev, generator=g)
    terminal_obs = torch.randn(S, N, n_obs, device=dev, generator=g)
    actions = torch.rand(S, N, n_u, device=dev, generator=g) * 2 - 1
    rewards = torch.randn(S, N, dtype=torch.float64, device=dev, generator=g)
    dones = (torch.rand(S, N, device=dev, generator=g) < 0.01).to(torch.uint8)
    ring = DockauvReplayRing(*[C.c_void_p(t.data_ptr()) for t in (obs, terminal_obs, actions, rewards, dones)])
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def fused(B, out, draw):
        _capi.check(lib.dockauv_replay_sample(C.byref(ring), F64, S, N, n_obs, n_u, t_first, n_valid, B, 0, draw,
                                              C.byref(out), stream))

    def torch_gather(j):
        k = j // N
        e = j - k * N
        slot = (t_first + k) % S
        nxt = (slot + 1) % S
        d = dones[slot, e]
        nx = torch.where(d.bool().unsqueeze(1), terminal_obs[slot, e], obs[nxt, e])
        return obs[slot, e], actions[slot, e], nx, d.float().unsqueeze(1), rewards[slot, e].float().unsqueeze(1)

    def torch_path(B):
        return torch_gather(torch.randint(0, n_valid * N, (B,), device=dev))

    def outputs(B, with_index=False):
        t = dict(obs=torch.empty(B, n_obs, device=dev), actions=torch.empty(B, n_u, device=dev),
                 next_obs=torch.empty(B, n_obs, device=dev), done=torch.empty(B, 1, device=dev),
                 reward=torch.empty(B, 1, device=dev))
        t["index"] = torch.empty(B, dtype=torch.int64, device=dev) if with_index else None
        ptrs = [None if t[k] is None else C.c_void_p(t[k].data_ptr())
                for k in ("obs", "actions", "next_obs", "done", "reward", "index")]
        return t, DockauvReplaySample(*ptrs)

    def launches(fn):
        fn()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)

    def time_us(fn, calls):
        for _ in range(max(3, calls // 10)):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) * 1e3 / calls

    # the fused rows equal the torch gathers at the same indices, bit for bit
    tv, out_chk = outputs(65536, with_index=True)
    fused(65536, out_chk, 12345)
    j = tv["index"] // N - (t_first % S)
    j = (j % S) * N + tv["index"] % N                # ring index -> draw j of the torch path
    ref = torch_gather(j)
    equal = all(torch.equal(tv[k], r) for k, r in zip(("obs", "actions", "next_obs", "done", "reward"), ref))
    if not equal:
        raise SystemExit("fused sampler differs from the torch gathers")
    del tv, out_chk, ref, j

    name, power = gpu_info()
    rows = []
    bpr = bytes_per_row(n_obs, n_u, 8)
    for B in BATCHES:
        _, out = outputs(B)
        draw = [0]

        def fused_call():
            draw[0] += 1
            fused(B, out, draw[0])

        calls = CALLS[B]
        n_fused, n_torch = launches(fused_call), launches(lambda: torch_path(B))
        f_us, t_us = [], []
        for _ in range(args.rounds):
            f_us.append(time_us(fused_call, calls))
            t_us.append(time_us(lambda: torch_path(B), calls))
        f_med, t_med = sorted(f_us)[len(f_us) // 2], sorted(t_us)[len(t_us) // 2]
        row = dict(batch=B, calls_per_round=calls, fused_us=f_med, torch_us=t_med, fused_us_rounds=f_us,
                   torch_us_rounds=t_us, speedup=t_med / f_med, fused_launches_per_call=n_fused,
                   torch_launches_per_call=n_torch, algorithmic_bytes_per_call=bpr * B,
                   fused_hbm_share=bpr * B / (f_med * 1e-6) / HBM_BYTES_PER_S)
        rows.append(row)
        print(json.dumps(row), flush=True)
    res = dict(tool="profiles/tools/replay_sample_bench.py", gpu=name, power_limit=power, envs=N, slots=S, n_obs=n_obs,
               n_u=n_u, reward_dtype="float64", n_valid=n_valid, ring_obs_array_bytes=obs.numel() * 4,
               bytes_per_row=bpr, hbm_bytes_per_s_datasheet=HBM_BYTES_PER_S, outputs_equal=equal,
               timing="CUDA events around calls_per_round back-to-back calls after warm-up, median of rounds that "
                      "alternate fused and torch; the fused call includes its ctypes argument marshalling",
               results=rows)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
