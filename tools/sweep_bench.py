#!/usr/bin/env python
"""One sweep (`trace_sweep`: K configurations of a scene in one device call) against K separate calls, on the GPU.

Arms, alternated rep by rep (medians with min / max):
  a_e2e   K x (flatten + upload + trace) with `trace_bundle`, as the GUI's scan / optimize loops do
  a_dev   the same with the K FlatScenes built beforehand (upload + trace per configuration)
  b       pose-only sweeps: K x (FlatScene.refresh + optb_scene_update_nodes + trace) on one uploaded scene (the f3
          path of the GUI slider loop). update_nodes carries no monitor rows: on the 4f grid this arm moves lens 2 only.
  c_e2e   one trace_sweep, including the K flattens
  c_dev   one sweep on FlatScenes built beforehand (sweep upload + trace + row sort)
  c_trace the trace of an uploaded sweep scene alone (CUDA events)
  d       one SweepScene.trace: configure + FlatScene.refresh x K on a table flattened once, the varied rows uploaded
          and the K configuration blobs built on the device (optb_scene_upload_sweep_rows), trace, row sort
  d_build the blob-building kernel alone (torch.profiler kernel time, in a pass of its own after the timed reps), with
          its write bandwidth: K x blob bytes over kernel time
Scenes: the 4f telescope over a 16 x 16 (F1, F2) grid (lens 2 and monitor 1 move; arm b moves lens 2 only) with N = 7,
1e3, 1e5; a splitting glass slab between two partially transmitting mirrors (tilt, index and reflectivity of the slab
vary; roots reach the 300-pop cap), K = 64; ripa with one mirror of its first group moved, K = 8 and 64, N = 1e4.
The _dev arms and b get a fixed live-ray budget and row capacity per root so that no attempt is repeated; the
_e2e arms use the public entry points as they are (which grow it on overflow). Writes JSON lines to --out and stdout."""
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
from optable_b200 import _abi as A
from optable_b200.backend import Engine
from optable_b200.bundle import DeviceTrace, RayBundle, trace_bundle
from optable_b200.flatten import FlatScene, batch_wavelengths_m
from optable_b200.sweep import SweepScene, trace_sweep
from optable_b200.workloads import WORKLOADS, Scene, ripa, telescope_4f_grid


def wall(f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    f()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def stats(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "reps": len(v)}


def checked(dt):
    cnt = dt.counters()
    if int(cnt[A.C_STATUS]):
        raise RuntimeError(f"status {int(cnt[A.C_STATUS])}: raise the live-ray budget or the row capacity")
    return cnt


def blob_bytes(f):
    """Bytes of one configuration blob (liboptb's blob_layout): 16-byte aligned sections."""
    al = lambda b: (b + 15) // 16 * 16
    return (al(max(f.n_nodes, 1) * 64) + al(f.n_nodes * A.NF_STRIDE * 8) + al(f.n_nodes * A.NI_STRIDE * 4)
            + al(f.n_materials * 4) + al(f.n_materials * A.MF_STRIDE * 8) + al(max(f.n_monitors, 1) * (A.MON_STRIDE + 4) * 8)
            + al(max(f.aux.size, 1) * 8))


def build_kernel_ms(engine, rows, reps):
    """Device time of the blob-building kernel per optb_scene_upload_sweep_rows call (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            engine.upload_sweep(rows).close()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if "sweep_build_kernel" in e.name and e.device_type.name == "CUDA"]
    if len(ev) != reps:
        raise RuntimeError(f"expected {reps} sweep_build_kernel launches in the profile, found {len(ev)}")
    return [e.device_time_total / 1e3 for e in ev]


def run_case(engine, name, tables, bundle, limit, reps, moved=None, out=None, live_per_root=None, rows_per_root=4,
             sweep=None):
    """moved: (builder of the base table, function(table, k) that applies configuration k's pose change, component
    getter) for the b arm, or None. sweep: (table, varied objects, configure(k)) for the d arms, or None."""
    K, n = len(tables), bundle.n
    lim = None if limit is None else {"max_trace_num": limit}
    wls = batch_wavelengths_m(bundle.columns["wavelength"], 1e-2)
    flats = [FlatScene(t.components, t.monitors, wavelengths_m=wls) for t in tables]
    rays_t = bundle.to_torch(device=f"cuda:{engine.device}")
    cap = n * rows_per_root
    max_trace = 2000 if limit is None else limit
    live = None if live_per_root is None else live_per_root * n
    live_k = None if live is None else live * K

    def a_e2e():
        for t in tables:
            trace_bundle(t, bundle, lim, engine=engine)

    def a_dev():
        for f in flats:
            dt = DeviceTrace(engine, f, n, cap, max_trace_num=max_trace)
            dt.run(rays_t, live)
            checked(dt)
            dt.scene.close()

    def c_e2e():
        trace_sweep(tables, bundle, lim, engine=engine)

    def c_dev():
        dt = DeviceTrace(engine, flats[0], n, cap * K, max_trace_num=max_trace, configs=flats)
        dt.run(rays_t, live_k)
        nh = int(checked(dt)[A.C_HITS])
        engine._sort_rows_on_device(dt.res, 0, nh, max_trace, flats[0].n_monitors)
        dt.scene.close()

    arms = {"a_e2e": a_e2e, "a_dev": a_dev, "c_e2e": c_e2e, "c_dev": c_dev}
    if moved is not None:
        base_table, pose, comp = moved
        bflat = FlatScene(base_table.components, base_table.monitors, wavelengths_m=wls)
        bdt = DeviceTrace(engine, bflat, n, cap, max_trace_num=max_trace)

        def b():
            for k in range(K):
                pose(base_table, k)
                bdt.scene.update_nodes(bflat.refresh(comp(base_table)))
                bdt.run(rays_t, live)
                checked(bdt)
        arms["b"] = b
    # the sweep trace alone: one uploaded sweep scene, CUDA events around the trace
    sdt = DeviceTrace(engine, flats[0], n, cap * K, max_trace_num=max_trace, configs=flats)
    sdt.run(rays_t, live_k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def c_trace():
        e0.record()
        sdt.run(rays_t, live_k)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    cnt = checked(sdt)
    if sweep is not None:
        sw = SweepScene(sweep[0], sweep[1])
        arms["d"] = lambda: sw.trace(bundle, sweep[2], K, lim, engine=engine)
    for f in arms.values():   # warm-up of every arm
        f()
    c_trace()
    times = {k: [] for k in list(arms) + ["c_trace"]}
    for _ in range(reps):
        for k, f in arms.items():
            times[k].append(wall(f))
        times["c_trace"].append(c_trace())
    flat_ms = [wall(lambda: [FlatScene(t.components, t.monitors, wavelengths_m=wls) for t in tables]) for _ in range(2)]
    sdt.scene.close()
    rec = {"case": name, "K": K, "N": n, "roots": K * n, "leaves": flats[0].n_leaves,
           "interactions": int(cnt[A.C_INTERACTIONS]), "dropped": int(cnt[A.C_DROPPED]),
           "flatten_K_tables_ms": float(np.median(flat_ms)), **{k: stats(v) for k, v in times.items()}}
    rec["c_trace_per_config_ms"] = rec["c_trace"]["median_ms"] / K
    if sweep is not None:
        captured = []

        def grab(rows, *a, **kw):   # the SweepRows of one trace call, without tracing
            captured.append(rows)
            raise StopIteration

        try:
            sw.trace(bundle, sweep[2], K, lim, engine=engine, tracer=grab)
        except StopIteration:
            pass
        rows = captured[0]
        build = build_kernel_ms(engine, rows, reps)
        nbytes = K * blob_bytes(rows.flat)
        rec["d_build"] = stats(build)
        rec["d_build_bytes_written"] = nbytes
        rec["d_build_write_TBps"] = nbytes / (rec["d_build"]["median_ms"] * 1e-3) / 1e12
        rec["d_varied_node_rows"], rec["d_varied_monitors"] = int(rows.nodes.size), int(rows.monitors.size)
        rec["speedup_d_over_c_e2e"] = rec["c_e2e"]["median_ms"] / rec["d"]["median_ms"]
        if "b" in rec:
            rec["speedup_d_over_b"] = rec["b"]["median_ms"] / rec["d"]["median_ms"]
    rec["speedup_dev_a_over_c"] = rec["a_dev"]["median_ms"] / rec["c_dev"]["median_ms"]
    rec["speedup_e2e_a_over_c"] = rec["a_e2e"]["median_ms"] / rec["c_e2e"]["median_ms"]
    if "b" in rec:
        rec["speedup_b_over_c_dev"] = rec["b"]["median_ms"] / rec["c_dev"]["median_ms"]
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as fh:
            fh.write(line + "\n")


def slab(n2, refl, tilt):
    """A glass slab with reflecting faces between two partially transmitting mirrors: roots reach the pop cap."""
    return Scene([ob.Mirror([-2, 0, 0], radius=3, reflectivity=0.9, transmission=0.1),
                  ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=1, n2=n2, reflectivity=refl).RotZ(tilt),
                  ob.Mirror([2, 0, 0], radius=3, reflectivity=0.9, transmission=0.1).RotZ(np.pi)],
                 [], [ob.Monitor([3, 0, 0], 6, 6), ob.Monitor([-3, 0, 0], 6, 6)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default=None, help="comma-separated case prefixes (4f, slab, ripa)")
    ap.add_argument("--n4f", default="7,1000,100000", help="bundle sizes of the 4f cases")
    ap.add_argument("--kripa", default="8,64", help="configuration counts of the ripa cases")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    head = json.dumps({"gpu": q, "torch": torch.__version__})
    print(head, flush=True)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(head + "\n")
    engine = Engine.get(0)
    want = lambda c: args.only is None or any(c.startswith(p) for p in args.only.split(","))
    if want("4f"):
        F = 43.17 + np.linspace(-1.5, 1.5, 16)
        tables = [telescope_4f_grid(ob, f1, f2) for f1 in F for f2 in F]
        base = telescope_4f_grid(ob, F[0], F[0])

        def pose(t, k):   # lens 2 to configuration k's place (the monitor cannot move on this path)
            f1, f2 = F[k // 16], F[k % 16]
            t.components[1].TX(43.17 + f1 + f2 - t.components[1].origin[0])

        dbase = telescope_4f_grid(ob, F[0], F[0])

        def configure(k):   # lens 2 and monitor 1 to configuration k's places
            f1, f2 = F[k // 16], F[k % 16]
            pose(dbase, k)
            dbase.monitors[1].TX(43.17 + f1 + 2 * f2 - dbase.monitors[1].origin[0])

        for n in [int(v) for v in args.n4f.split(",")]:
            reps = args.reps if n < 100_000 else max(3, args.reps // 2)
            run_case(engine, f"4f_grid_16x16_N{n}", tables, RayBundle.collimated_disc(n, radius=2.5), None, reps,
                     (base, pose, lambda t: t.components[1]), args.out,
                     sweep=(dbase, [dbase.components[1], dbase.monitors[1]], configure))
    if want("slab"):
        rng = np.random.default_rng(7)
        tables = [slab(1.45 + 0.1 * rng.uniform(), 0.1 + 0.2 * rng.uniform(), 0.1 * rng.uniform(-1, 1)) for _ in range(64)]
        bundle = RayBundle.collimated_disc(1000, x0=-3, radius=0.6, direction=(1.0, 0.01, 0.0))
        run_case(engine, "slab_cavity_split_K64_N1000", tables, bundle, 300, args.reps, None, args.out, live_per_root=600,
                 rows_per_root=160)
    for K in ([int(v) for v in args.kripa.split(",")] if want("ripa") else []):
        tables = []
        for k in range(K):
            sc = ripa(ob, n_rays=0)
            sc.components[0].components[1].TX(1e-4 * k)
            tables.append(sc)
        base, dbase = ripa(ob, n_rays=0), ripa(ob, n_rays=0)
        dx = {id(base): 0, id(dbase): 0}

        def pose(t, k):
            t.components[0].components[1].TX(1e-4 * (k - dx[id(t)]))
            dx[id(t)] = k

        w = WORKLOADS["c5_ripa_64"]
        run_case(engine, f"ripa_K{K}_N10000", tables, w.bundle(10_000, 0), w.max_trace_num, max(3, args.reps // 2),
                 (base, pose, lambda t: t.components[0].components[1]), args.out, live_per_root=64,
                 rows_per_root=int(w.rows_per_ray * 2),
                 sweep=(dbase, [dbase.components[0].components[1]], lambda k: pose(dbase, k)))


if __name__ == "__main__":
    main()
