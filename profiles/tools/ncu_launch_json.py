#!/usr/bin/env python
"""`ncu -i X.ncu-rep --page raw --csv` of one steady-state step  ->  profiles/r02/ncu_per_launch_<config>.json, the file
bench.py quotes for `roofline.traffic` / `executed_pipe_frac` (with the hash of the kernel sources it was captured from,
so that a stale capture is never quoted).

    ncu -i profile_out/prof_pipe_cur.ncu-rep --page raw --csv > profiles/r02/<tag>_pipeline_ncu_raw.csv
    python profiles/tools/ncu_launch_json.py profiles/r02/<tag>_pipeline_ncu_raw.csv C4 524288 [f64]

The third argument is the number of envs each captured launch covered (a 1M-env step runs as two halves).
"""
import collections
import csv
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from bench import kernel_source_hash  # noqa: E402

SCALE = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}
NAMES = (("dynamics_kernel", "dynamics_cull_finish"), ("rays_finish_kernel", "rays_finish"), ("rays_thread_kernel", "rays_finish"),
         ("episode_end_kernel", "episode_end"))


def main():
    path, config, envs_per_launch = sys.argv[1], sys.argv[2], int(sys.argv[3])
    precision = sys.argv[4] if len(sys.argv) > 4 else "f64"
    rows = list(csv.reader(open(path)))
    hdr, units, data = rows[0], rows[1], rows[2:]
    col = {h: i for i, h in enumerate(hdr)}

    def val(r, name):
        i = col[name]
        return float(r[i].replace(",", "")) * SCALE.get(units[i], 1.0)

    per = collections.defaultdict(list)
    for r in data:
        kname = r[col["Kernel Name"]]
        short = next((s for k, s in NAMES if k in kname), None)
        if short is None:
            continue
        per[short].append({
            "us": val(r, "gpu__time_duration.sum"),
            "dram_bytes": val(r, "dram__bytes_read.sum") + val(r, "dram__bytes_write.sum"),
            "dram_read_bytes": val(r, "dram__bytes_read.sum"),
            "fp64_pipe_pct": val(r, "sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active"),
            "issue_active_pct": val(r, "smsp__issue_active.avg.pct_of_peak_sustained_active"),
            "warps_active_pct": val(r, "sm__warps_active.avg.pct_of_peak_sustained_active"),
            "registers": val(r, "launch__registers_per_thread"),
        })
    out = {"config": config, "precision": precision, "envs_per_captured_launch": envs_per_launch,
           "kernel_source_hash": kernel_source_hash(), "source_csv": os.path.relpath(path, ROOT), "launches": {}}
    t_tot = pipe_w = bytes_env = 0.0
    for name, ls in per.items():
        n = len(ls)
        avg = {k: sum(x[k] for x in ls) / n for k in ls[0]}
        avg["captured_launches"] = n
        avg["dram_bytes_per_env"] = avg["dram_bytes"] / envs_per_launch
        out["launches"][name] = avg
        t_tot += avg["us"]
        pipe_w += avg["us"] * avg["fp64_pipe_pct"] / 100.0
        bytes_env += avg["dram_bytes_per_env"]
    out["fp64_pipe_frac_time_weighted"] = pipe_w / t_tot if t_tot else None
    out["step_dram_bytes_per_env"] = bytes_env
    dst = os.path.join(ROOT, "profiles", "r02", f"ncu_per_launch_{config}.json")
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
