#!/usr/bin/env python
"""Sweeps whose interact caps bind: K `trace_table` calls against one family-serial `trace_sweep`.

Scenes:
  prism_K{64,256}     `tests.scenes.caps_binding` (a TriangularPrism whose faces 2 and 3 stop after 3 hits per ray id,
                      4 ids x 6 wavelengths = 24 rays) over a grid of tilts and face-1 reflectivities: K * F = 4 K
                      families, so the serial kernel runs 4 K threads
  prism_ids{F}_K256   the same prism with F distinct ids, 2 wavelengths each: K * F = 2.6e5 threads at F = 1024
Arms, alternated rep by rep (medians with min / max), each ending in a device synchronise:
  a   K x `trace_table` (what `OpticalTable.ray_tracing` runs) on tables built beforehand, with the components'
      interact counts and the monitors reset before each table
  b   one `trace_sweep` of the same Ray list through the K tables
`rows_equal` checks that the monitor rows of the two arms agree (row count and summed hit coordinates per
configuration). Writes JSON lines to --out and stdout; the first line names the card and its power limit."""
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
from optable_b200.flatten import FlatScene
from optable_b200.sweep import trace_sweep
from optable_b200.table import trace_table

LIMIT = {"max_trace_num": 80}


def wall(f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = f()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), out


def stats(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "reps": len(v)}


def table(refl, tilt):
    ps = ob.TriangularPrism(origin=[0, 0, 0], width=6, height=6, n1=1, n2=ob.Glass_NBK7(), alpha=np.pi / 4,
                            beta=np.pi / 2, reflectivity_1=refl, reflectivity_2=0.5, reflectivity_3=0.4,
                            max_interact_count_2=3, max_interact_count_3=3).RotZ(tilt)
    t = ob.OpticalTable()
    t.add_components([ps])
    t.add_monitors([ob.Monitor([-3, 0, 0], width=12, height=12)])
    return t


def rays(n_ids, n_wl):
    ys = np.linspace(-2.5, 2.5, n_ids)
    r0 = [ob.Ray([3, y + 3, 0.1 * y], [-1, 0.02 * y, 0], wavelength=780e-7, w0=61e-4, id=10 + i) for i, y in enumerate(ys)]
    return ob.multiplex_rays_in_wavelength(r0, list(np.linspace(450e-7, 900e-7, n_wl)))


def reset(tables):
    for t in tables:
        for comp in FlatScene(t.components, t.monitors).capslots:
            comp._interact_count = {}
        for m in t.monitors:
            m.clear()


def run_case(engine, name, K, n_ids, n_wl, reps, out):
    g = int(np.ceil(np.sqrt(K)))
    grid = [(0.2 + 0.25 * (i // g) / g, -0.05 + 0.1 * (i % g) / g) for i in range(K)]
    tables = [table(r, t) for r, t in grid]
    bundle = rays(n_ids, n_wl)

    def arm_a():
        reset(tables)
        for t in tables:
            trace_table(t, bundle, LIMIT, engine=engine)
        return [(t.monitors[0].ndata, float(np.sum(t.monitors[0].get_PList(sort="ID")))) for t in tables]

    def arm_b():
        reset(tables)
        res = trace_sweep(tables, bundle, LIMIT, engine=engine)
        px = [res.rows(k) for k in range(K)]
        return [(len(r["hit_px"]), float((r["hit_px"] + r["hit_py"] + r["hit_pz"]).sum())) for r in px], res

    arms = {"a": arm_a, "b": arm_b}
    got_a, (got_b, res) = arm_a(), arm_b()       # warm-up of every shape, and the rows compared below
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, f in arms.items():
            times[k].append(wall(f)[0])
    rows_equal = all(a[0] == b[0] and abs(a[1] - b[1]) <= 1e-9 * max(1.0, abs(a[1])) for a, b in zip(got_a, got_b))
    rec = {"case": name, "K": K, "rays": len(bundle), "families": n_ids, "serial_threads": K * n_ids,
           **{f"arm_{k}": stats(v) for k, v in times.items()},
           "speedup_a_over_b": float(np.median(times["a"]) / np.median(times["b"])), "rows_equal": bool(rows_equal),
           "max_interact_count_reached": int(res.interact_counts.max())}
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as fh:
            fh.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="prism_K64,prism_K256,prism_ids1024_K256")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    head = json.dumps({"gpu": q, "torch": torch.__version__})
    print(head, flush=True)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(head + "\n")
    engine = Engine.get(0)
    cases = {"prism_K64": (64, 4, 6), "prism_K256": (256, 4, 6), "prism_ids1024_K256": (256, 1024, 2)}
    for name in args.cases.split(","):
        K, n_ids, n_wl = cases[name]
        run_case(engine, name, K, n_ids, n_wl, args.reps if n_ids <= 4 else max(2, args.reps // 2), args.out)


if __name__ == "__main__":
    main()
