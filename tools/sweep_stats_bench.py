#!/usr/bin/env python
"""Monitor summaries of a whole sweep: one DeviceMonitor per (configuration, monitor) against one grouped call.

Scene: the 4f telescope over a 16 x 16 (F1, F2) grid (K = 256 configurations, M = 2 monitors), N = 7, 1e3 and 1e5 rays,
traced once with `trace_sweep`. Arms, alternated rep by rep (medians with min / max), each ending in a device
synchronise:
  a       the K x M loop of `res.monitor(k, m).stats()`
  b       one `res.stats()` (cache cleared before every rep): one optb_monitor_stats_grouped call + one copy back
  kernel  the grouped call alone (all its kernels, CUDA events, workspace and outputs allocated beforehand)
Achieved bandwidth = row-column bytes the grouped call reads per row (group keys: hit_root + hit_monitor, 8 B; first
pass: sorted index + 9 fp64 columns, 76 B; second pass: sorted index + 6 fp64 columns, 52 B; 136 B in all, the radix
sort's own traffic not counted) x rows / kernel time. Writes JSON lines to --out and stdout."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.analytics import _frame
from optable_b200.backend import Engine, lib
from optable_b200.bundle import RayBundle
from optable_b200.sweep import trace_sweep
from optable_b200.workloads import telescope_4f_grid

READ_BYTES_PER_ROW = 8 + (4 + 9 * 8) + (4 + 6 * 8)


def wall(f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    f()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def stats(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "reps": len(v)}


def grouped_kernel_ms(engine, res, K, M, reps):
    """CUDA-event time of optb_monitor_stats_grouped over the sweep's rows, per call (median over `reps`)."""
    hits, n, G = res.hits, int(res.hits["hit_px"].numel()), K * M
    r = A.Result()
    for k, v in hits.items():
        setattr(r, k, v.data_ptr())
    frames = (A.MonitorFrame * G)(*[_frame(res.tables[k].monitors[m]) for k in range(K) for m in range(M)])
    dev = f"cuda:{engine.device}"
    frames_dev = torch.frombuffer(bytearray(frames), dtype=torch.uint8).to(dev)
    out = torch.empty((G, A.MS_STRIDE), dtype=torch.float64, device=dev)
    per_row = torch.empty((5, max(n, 1)), dtype=torch.float64, device=dev)
    ws = torch.empty(int(lib().optb_monitor_stats_grouped_workspace_bytes(n, G)), dtype=torch.uint8, device=dev)
    p = lambda i: C.c_void_p(per_row[i].data_ptr())

    def call():
        st = torch.cuda.current_stream().cuda_stream
        engine._check(lib().optb_monitor_stats_grouped(engine._ctx, C.byref(r), 0, n, res.n, K, M, C.c_void_p(frames_dev.data_ptr()),
                                                       C.c_void_p(out.data_ptr()), p(0), p(1), p(2), p(3), p(4),
                                                       C.c_void_p(ws.data_ptr()), int(ws.numel()), C.c_void_p(st)))
    call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t = []
    for _ in range(reps):
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        t.append(e0.elapsed_time(e1))
    return t


def run_case(engine, tables, n, reps, out):
    K, M = len(tables), len(tables[0].monitors)
    res = trace_sweep(tables, RayBundle.collimated_disc(n, radius=2.5), engine=engine)
    rows = int(res.hits["hit_px"].numel())

    def a():
        return [[res.monitor(k, m).stats() for m in range(M)] for k in range(K)]

    def b():
        res._grouped = None
        return res.stats()

    # the two arms agree: counts and histograms exactly, the sums to rounding
    sa, sb = a(), b()
    worst = 0.0
    for k in range(K):
        for m in range(M):
            assert sa[k][m]["count"] == sb["count"][k, m] and np.array_equal(sa[k][m]["hist_y"], sb["hist_y"][k, m])
            for q in ("sum_intensity", "mean_y", "std_y", "mean_waist_distance"):
                x, y = sa[k][m][q], sb[q][k, m]
                worst = max(worst, abs(x - y) / max(abs(x), 1e-300)) if x != y else worst
    times = {"a": [], "b": []}
    for _ in range(reps):
        times["a"].append(wall(a))
        times["b"].append(wall(b))
    kern = grouped_kernel_ms(engine, res, K, M, 20)
    km = float(np.median(kern))
    rec = {"case": f"4f_grid_16x16_N{n}", "K": K, "M": M, "N": n, "rows": rows,
           "rows_x_read_bytes_MB": rows * READ_BYTES_PER_ROW / 1e6, "a_loop": stats(times["a"]), "b_grouped": stats(times["b"]),
           "kernel": stats(kern), "speedup_a_over_b": float(np.median(times["a"]) / np.median(times["b"])),
           "read_bytes_per_row": READ_BYTES_PER_ROW, "achieved_read_GBps": rows * READ_BYTES_PER_ROW / (km * 1e-3) / 1e9,
           "max_rel_diff_a_vs_b": worst}
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as fh:
            fh.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n", default="7,1000,100000", help="comma-separated bundle sizes")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    head = json.dumps({"gpu": q, "torch": torch.__version__})
    print(head, flush=True)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(head + "\n")
    engine = Engine.get(0)
    F = 43.17 + np.linspace(-1.5, 1.5, 16)
    tables = [telescope_4f_grid(ob, f1, f2) for f1 in F for f2 in F]
    for n in (int(v) for v in args.n.split(",")):
        run_case(engine, tables, n, args.reps if n < 100_000 else max(3, args.reps // 2), args.out)


if __name__ == "__main__":
    main()
