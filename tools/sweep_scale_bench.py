#!/usr/bin/env python
"""Sweeps sharded over GPUs by configuration against the one-GPU sweep. Run under torchrun, one rank per GPU:

    python -m torch.distributed.run --nproc-per-node 8 tools/sweep_scale_bench.py --out sweep_scale.jsonl

Arms, alternated rep by rep (medians with min / max over the reps):
  one    rank 0 runs the sweep alone (group=None) while the other ranks wait at a barrier
  world  every rank runs its shard (group=True, gather=False)
Both arms end with `stats()`, which the sharded call computes eagerly, so both do the same work.
  e2e    host clock around the whole call, after a barrier, up to a device synchronise: flattens (trace_sweep) or
         configure + refresh of every configuration (SweepScene; its base flatten is cached by the warm-up), trace,
         row sort, statistics and, for `world`, the exchange; the slowest rank
  dev    CUDA events around the sweep tracer (sweep upload + trace + row sort) on each rank; the slowest rank
Cases: the 4f telescope over a 16 x 16 (F1, F2) grid, K = 256, N = 1e3 and 1e5 (trace_sweep); ripa with one mirror of
its first group moved, K = 64, N = 1e4 (SweepScene). Shards are contiguous and equal in configuration count.
The first line is the card, its power limit and max SM clock; every line goes to stdout and, on rank 0, to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import optable_b200 as ob
from optable_b200.backend import Engine
from optable_b200.bundle import RayBundle
from optable_b200.sweep import SweepScene, _device_sweep, trace_sweep
from optable_b200.workloads import WORKLOADS, ripa, telescope_4f_grid


class EventTracer:
    """The CUDA sweep with CUDA events around it: `ms()` is the device time of the last call (0 when it ran none)."""

    def __init__(self):
        self.ev = None

    def __call__(self, *a, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = _device_sweep(*a, **kw)
        e.record()
        self.ev = (s, e)
        return out

    def ms(self):
        if self.ev is None:
            return 0.0
        self.ev[1].synchronize()
        v, self.ev = self.ev[0].elapsed_time(self.ev[1]), None
        return v


def slowest(v):
    t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def spread(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "reps": len(v)}


def run_case(name, call, reps, emit):
    """call(group, tracer) -> SweepResult; alternates the arms, warm-up first."""
    rank, world = dist.get_rank(), dist.get_world_size()
    tr = EventTracer()
    times = {"one": ([], []), "world": ([], [])}
    for rep in range(reps + 1):
        for arm in ("one", "world") if rep % 2 == 0 else ("world", "one"):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if arm == "world" or rank == 0:
                res = call(True if arm == "world" else None, tr)
                res.stats()
                torch.cuda.synchronize()
            e2e = 1e3 * (time.perf_counter() - t0)
            e2e, dev = slowest(e2e if arm == "world" or rank == 0 else 0.0), slowest(tr.ms())
            if rep:
                times[arm][0].append(e2e)
                times[arm][1].append(dev)
    line = {"case": name, "world": world}
    for arm, (e, d) in times.items():
        line[f"{arm}_e2e"], line[f"{arm}_dev"] = spread(e), spread(d)
    line["speedup_e2e"] = line["one_e2e"]["median_ms"] / line["world_e2e"]["median_ms"]
    line["speedup_dev"] = line["one_dev"]["median_ms"] / line["world_dev"]["median_ms"]
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default=None, help="comma-separated case prefixes (4f, ripa)")
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    rank = dist.get_rank()
    engine = Engine.get(local)

    def emit(obj):
        if rank == 0:
            s = json.dumps(obj)
            print(s, flush=True)
            if args.out:
                with open(args.out, "a") as fh:
                    fh.write(s + "\n")

    if rank == 0:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip().splitlines()
        emit({"gpu": q[local] if q else "", "gpus": dist.get_world_size(), "torch": torch.__version__})
    want = lambda c: args.only is None or any(c.startswith(p) for p in args.only.split(","))
    if want("4f"):
        F = 43.17 + np.linspace(-1.5, 1.5, 16)
        tables = [telescope_4f_grid(ob, f1, f2) for f1 in F for f2 in F]
        for n in (1000, 100_000):
            bundle = RayBundle.collimated_disc(n, radius=2.5)
            run_case(f"4f_grid_16x16_K256_N{n}",
                     lambda group, tr: trace_sweep(tables, bundle, engine=engine, tracer=tr, group=group),
                     args.reps if n < 100_000 else max(3, args.reps // 2), emit)
    if want("ripa"):
        w = WORKLOADS["c5_ripa_64"]
        sc = ripa(ob, n_rays=0)
        mirror = sc.components[0].components[1]
        saved = (mirror.origin.copy(), np.array(mirror.transform_matrix, dtype=np.float64), mirror._bbox)

        def configure(k):   # absolute: back to the first pose, then k steps
            mirror.origin, mirror.transform_matrix, mirror._bbox = saved[0].copy(), saved[1].copy(), saved[2]
            mirror.TX(1e-4 * k)

        sweep, bundle = SweepScene(sc, [mirror]), w.bundle(10_000, 0)
        run_case("ripa_SweepScene_K64_N10000",
                 lambda group, tr: sweep.trace(bundle, configure, 64, {"max_trace_num": w.max_trace_num}, engine=engine,
                                               tracer=tr, group=group),
                 max(3, args.reps // 2), emit)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
