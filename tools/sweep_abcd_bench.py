#!/usr/bin/env python
"""ABCD matrices of a whole 4f scan: K calls of the table method against two sweep traces.

Scene: the 4f telescope over a 16 x 16 (F1, F2) grid (K = 256 configurations, `workloads.telescope_4f_grid`), with
N = 7 rays (`tests.scenes.abcd_rays`, the calibration's bundle) and N = 1000 rays (a disc inside mon0, distinct ids).
Arms, alternated rep by rep (medians with min / max), each ending in a device synchronise:
  a   K x `OpticalTable.calculate_abcd_matrix` on tables built beforehand: what `calibrate_symmetric_4f` does per cost
      evaluation, once per configuration
  b   one `sweep_abcd_matrix` over the same K tables (flatten once, two sweeps, two small device calls)
  c   one `SweepScene.abcd_matrix` that moves lens 2 and monitor 1 (`configure(k)` K times, the table flattened once)
`max_abs_diff_ab` / `max_abs_diff_bc` compare the matrices of the arms at the timed sizes. Writes JSON lines to --out
and stdout; the first line names the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import optable_b200 as ob
from optable_b200.backend import Engine
from optable_b200.sweep import SweepScene, sweep_abcd_matrix
from optable_b200.workloads import telescope_4f_grid
from tests import scenes

F0 = 43.17


def wall(f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = f()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), out


def stats(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "reps": len(v)}


def table(F1, F2):
    sc = telescope_4f_grid(ob, F1, F2)
    t = ob.OpticalTable()
    t.add_components(list(sc.components))
    t.add_monitors(list(sc.monitors))
    return t


def rays(n):
    if n == 7:
        return scenes.abcd_rays(ob)
    rng = np.random.default_rng(20261022)
    rr, th = 2.0 * np.sqrt(rng.uniform(size=n)), rng.uniform(0, 2 * np.pi, n)
    return [ob.Ray([-10, r * np.cos(a), r * np.sin(a)], [1, 0, 0], wavelength=780e-7, w0=61e-4, id=i)
            for i, (r, a) in enumerate(zip(rr, th))]


def run_case(engine, F, n, reps, out):
    K = len(F)
    bundle = rays(n)
    tables = [table(*f) for f in F]
    base = table(F0, F0)
    lens, mon1 = base.components[1], base.monitors[1]
    saved = []

    def walk(o):   # the poses of lens 2 (and its surfaces) and monitor 1: TX is relative, configure(k) is absolute
        saved.append((o, o.origin.copy(), np.array(o.transform_matrix, dtype=np.float64), o._bbox))
        for c in getattr(o, "components", []):
            walk(c)

    walk(lens)
    walk(mon1)
    sw = SweepScene(base, [lens, mon1])

    def configure(k):
        for o, org, T, box in saved:
            o.origin, o.transform_matrix, o._bbox = org.copy(), T.copy(), box
        lens.TX(F[k][0] + F[k][1] - 2 * F0)
        mon1.TX(F[k][0] + 2 * F[k][1] - 3 * F0)

    arms = {
        "a": lambda: np.stack([t.calculate_abcd_matrix(t.monitors[0], t.monitors[1], bundle) for t in tables]),
        "b": lambda: sweep_abcd_matrix(tables, 0, 1, bundle, engine=engine).M,
        "c": lambda: sw.abcd_matrix(0, 1, bundle, configure, K, engine=engine).M,
    }
    got = {k: f() for k, f in arms.items()}      # warm-up of every shape, and the matrices compared below
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, f in arms.items():
            times[k].append(wall(f)[0])
    rec = {"case": f"4f_grid_K{K}_N{n}", "K": K, "N": n, **{f"arm_{k}": stats(v) for k, v in times.items()},
           "speedup_a_over_b": float(np.median(times["a"]) / np.median(times["b"])),
           "speedup_a_over_c": float(np.median(times["a"]) / np.median(times["c"])),
           "max_abs_diff_ab": float(np.nanmax(np.abs(got["a"] - got["b"]))),
           "max_abs_diff_bc": float(np.nanmax(np.abs(got["b"] - got["c"])))}
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as fh:
            fh.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n", default="7,1000", help="comma-separated bundle sizes (7: the calibration's bundle)")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    head = json.dumps({"gpu": q, "torch": torch.__version__})
    print(head, flush=True)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(head + "\n")
    engine = Engine.get(0)
    Fs = F0 + np.linspace(-1.5, 1.5, 16)
    F = [(f1, f2) for f1 in Fs for f2 in Fs]
    for n in (int(v) for v in args.n.split(",")):
        run_case(engine, F, n, args.reps if n <= 7 else max(3, args.reps // 2), args.out)


if __name__ == "__main__":
    main()
