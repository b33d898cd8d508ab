"""GPU probe (not a test): fixed cost per LP vs cost per pivot of the tier-1 kernel on the bench batch.

Solves bench.py's batch (4096 dense LPs 64 x 128, seed 1234, inputs resident in HBM, gm_simplex_batch_device)
with the pivot cap at 1, 2, 5, 10, 25, 50 and uncapped. A capped LP still runs the whole cold path up to its cap
(input checks, W fill, initial inversion, Phase-I entry, results), so a straight line through the capped points,
kernel_ms = fixed + slope * pivots, splits the kernel time into a per-LP fixed part and a per-pivot part. The
uncapped point minus that line is what only complete solves pay: the polishes and the Phase-II entry.

  python tests/tier1_cost_probe.py [--launches 20] [--out FILE]

Prints one JSON line per cap and a last line with the fit; every line carries the GPU name, power limit and SM clock
read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CAPS = (1, 2, 5, 10, 25, 50, 0)  # 0: the default cap, i.e. solved to the end


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_mhz": float(out[2]), "sm_max_mhz": float(out[3])}
    except Exception as e:
        return {"gpu_info_error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=20, help="timed launches per cap (after 3 warm-up launches)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import torch
    import gomilp_b200 as gm
    import bench

    if not torch.cuda.is_available() or gm.device_count() < 1:
        raise RuntimeError("tier1_cost_probe.py needs a CUDA device")
    gm.init(0)
    dev = torch.device("cuda", 0)
    c, A, b = bench.make_batch(0)
    B, M, N = bench.BATCH, bench.M, bench.N
    dc, dA, db = (torch.from_numpy(v).to(dev) for v in (c, A, b))
    d_status = torch.zeros(B, dtype=torch.int32, device=dev)
    d_optF = torch.zeros(B, dtype=torch.float64, device=dev)
    d_x = torch.zeros(B, N, dtype=torch.float64, device=dev)
    d_basis = torch.zeros(B, M, dtype=torch.int64, device=dev)
    d_stats = torch.zeros(B, 8, dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)

    def launch():
        gm.simplex_batch_device(B, dc.data_ptr(), dA.data_ptr(), db.data_ptr(), M, N, 0.0, d_status.data_ptr(),
                                d_optF.data_ptr(), d_x.data_ptr(), d_basis.data_ptr(), d_stats.data_ptr(),
                                stream.cuda_stream)

    lines, fit_pts = [], []
    try:
        for cap in CAPS:
            gm.set_options(max_pivots=cap)
            for _ in range(3):
                launch()
            stream.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.launches + 1)]
            with torch.cuda.stream(stream):
                ev[0].record(stream)
                for k in range(args.launches):
                    launch()
                    ev[k + 1].record(stream)
            stream.synchronize()
            ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.launches)]
            stats = d_stats.cpu().numpy()
            tm = gm.last_timing()
            pivots = float((stats[:, 0] + stats[:, 1]).sum()) / B
            status = d_status.cpu().numpy()
            row = {"probe": "tier1_cost", "cap": cap, "kernel_ms_median": float(np.median(ms)),
                   "kernel_ms_min": float(np.min(ms)), "kernel_ms_max": float(np.max(ms)), "launches": args.launches,
                   "pivots_per_lp": pivots, "inversions_per_lp": float(stats[:, 3].sum()) / B,
                   "status_counts": {str(int(s)): int((status == s).sum()) for s in np.unique(status)},
                   "tier": tm["tier"], "grid": tm["grid"], **gpu_info()}
            lines.append(row)
            if cap > 0:
                fit_pts.append((pivots, row["kernel_ms_median"]))
            print(json.dumps(row), flush=True)
    finally:
        gm.set_options()
    x = np.array([p[0] for p in fit_pts])
    y = np.array([p[1] for p in fit_pts])
    slope, fixed = np.polyfit(x, y, 1)
    full = lines[-1]
    rest = full["kernel_ms_median"] - (fixed + slope * full["pivots_per_lp"])
    ctas = full["grid"]
    lp_per_cta = B / ctas
    summary = {"probe": "tier1_cost_fit", "fixed_ms": float(fixed), "ms_per_pivot_per_lp": float(slope),
               "uncapped_ms": full["kernel_ms_median"], "uncapped_pivots_per_lp": full["pivots_per_lp"],
               "uncapped_minus_fit_ms": float(rest),
               "fixed_us_per_lp_per_cta": 1e3 * float(fixed) / lp_per_cta,
               "us_per_pivot_per_cta": 1e3 * float(slope) / lp_per_cta,
               "fixed_in_pivots": float(fixed / slope) if slope > 0 else None,
               "fit_caps": [c for c in CAPS if c > 0], **gpu_info()}
    print(json.dumps(summary), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for r in lines + [summary]:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
