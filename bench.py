#!/usr/bin/env python
"""Benchmark of the optable ray_tracing hot path on B200 (contract: see the repo brief / DESIGN.md section 6).

  python bench.py --gpus N --steps K --warmup W          # CUDA arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference --steps K --warmup W  # CPU arm: the reference's path on all host cores

Headline workload (BASELINE.json configs[1], SURVEY 8(d) C2): two LENS-9 parametric aspheres as a 4f relay, monitors
at x = 0 and x = 2F1 + 2F2, 1e7 synthetic collimated Gaussian rays per GPU (disc radius 3, splitmix64 positions).
A step = one trace of the whole batch incl. monitor row capture. Metric = ray-surface interactions per second
(an interaction = one popped ray that hit a surface = one output segment of finite length).

The same line carries, under "workloads", the other BASELINE configs measured the same way in the same run:
c3 (Sellmeier doublets x 16 wavelengths, 1e7 rays/GPU), c4 (4-mirror cavity, 1e6 rays x 4000 bounces) and c5 (the
7,689-leaf ripa MMA scene, 12.5e6 rays per GPU = the north-star 100M-ray batch at 8 GPUs), each with its own device
value, end-to-end value, roofline and CPU baseline (`--workload X` makes X the headline instead; `--only` skips the rest).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ray-surface interactions/sec (fp64)"
UNIT = "interactions/s"
WORKLOAD = "c2_4f_telescope"
RAY_RECORD_BYTES = 104  # SURVEY 8: 12 fp64 + root + flags per ray
# SURVEY 8(d) algorithmic fp64 flops: 55 per planar leaf test, 200 per curved leaf test (local box + 10-sample sign
# scan + root), 25 per lab-box test, 180 per applied interaction (to-local, physics incl. 2 Sellmeier, Snell, complex
# division, to-lab); FMA = 2. The test counts are the device's own counters of the measured run (OPTB_C_TESTS,
# OPTB_C_TESTS_CURVED, OPTB_C_BOX_TESTS), so nothing here is pasted from a profile.
FLOPS_PLANAR, FLOPS_CURVED, FLOPS_BOX, FLOPS_INTERACT = 55, 200, 25, 180
# default monitor row of the end-to-end leg = what Monitor._data_raw holds (monitor.py:15-20): P_local, intensity, t
# + the packed (root, monitor, pop) key = 48 B; direction and q of the segment are opt-in columns
# (--e2e-columns all: 92 B with the key as three columns)
E2E_COLUMNS = ("hit_key", "hit_px", "hit_py", "hit_pz", "hit_intensity", "hit_t")


def workloads():
    from optable_b200.workloads import WORKLOADS

    return WORKLOADS


def build_scene(workload=WORKLOAD):
    return workloads()[workload].flat()


def make_bundle(n, start, workload=WORKLOAD):
    return workloads()[workload].bundle(n, start)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def _nvml_loop(self):
        """NVML in-process: a sample every 10 ms (the nvidia-smi binary needs ~0.3 s per query, i.e. one sample
        for a 0.3 s timed region)."""
        import pynvml as N

        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(self.index)
        reasons_fn = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = (0x8, 0x40, 0x20, 0x4)  # HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap
        mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        while not self._halt.is_set():
            sm, mask = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM), int(reasons_fn(h))
            self.rows.append([str(sm), str(mx)] + ["Active" if mask & b else "Not Active" for b in bits])
            self._halt.wait(0.01)

    def run(self):
        try:
            self._nvml_loop()
            return
        except Exception:
            pass
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows for k in range(4) if len(r) >= 6 and r[2 + k].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ---- CPU arms ----------------------------------------------------------------------------------------------------
def cpu_arm(flat, n_sample, threads, repeats=1, workload=WORKLOAD):
    """Oracle port of the reference on the host cores: interactions/s on the first n_sample rays of the workload."""
    from oracle import oracle as O

    w = workloads()[workload]
    arrs = w.bundle(n_sample, 0).materialise()
    best = None
    inter = 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        # same outputs as the CUDA step: every monitor row + histograms (capacity given: no counting pass)
        out = O.trace(flat, arrs, max_trace_num=w.max_trace_num, record_segments=False, record_hits=True, record_hist=True,
                      nthreads=threads, hit_capacity=n_sample * w.rows_per_ray + 1024)
        dt = time.perf_counter() - t0
        inter = int(out["counters"][1])
        best = dt if best is None else min(best, dt)
    cpu_arm.counters = np.asarray(out["counters"]).astype(np.int64)  # the reference loop's own work counts on the sample
    return inter / best, inter, best


def _py_ref_worker(job):
    """One process of the kind="reference" leg: the UNMODIFIED Python reference (baseline/_ref, imported through
    oracle/ref_harness) tracing its share of the sample with its own OpticalTable.ray_tracing."""
    workload, lo, hi = job
    import contextlib
    import io

    from oracle import ref_harness as RH

    ref = RH.load_reference()
    w = workloads()[workload]
    sc = w.scene(ref)
    table = ref.OpticalTable()
    table.add_components(sc.components)
    table.add_monitors(sc.monitors)
    cols = w.bundle(hi - lo, lo).materialise()
    hasq = bool(cols["flags"][0] & 2)
    rays = []
    for k in range(hi - lo):
        r = ref.Ray([cols["ox"][k], cols["oy"][k], cols["oz"][k]], [cols["dx"][k], cols["dy"][k], cols["dz"][k]],
                    wavelength=float(cols["wavelength"][k]), intensity=float(cols["intensity"][k]))
        if hasq:
            r.qo = complex(cols["q_re"][k], cols["q_im"][k])
        rays.append(r)
    limit = {"max_trace_num": w.max_trace_num}
    with contextlib.redirect_stdout(io.StringIO()):  # the reference prints progress lines every second
        t0 = time.perf_counter()
        table.ray_tracing(rays, perfomance_limit=limit)
        dt = time.perf_counter() - t0
    inter = sum(1 for r in table.rays if r.length is not None and not r.alive)
    return inter, dt


def python_reference_arm(workload, n_sample, procs):
    """kind = "reference": the real reference (pure Python, single-threaded by design) run as one process per host
    core on disjoint slices of the first n_sample rays. Returns None when baseline/_ref is absent."""
    from oracle import ref_harness as RH

    if not RH.reference_available():
        return None
    import multiprocessing as mp

    procs = max(1, min(procs, n_sample))
    bounds = [n_sample * k // procs for k in range(procs + 1)]
    jobs = [(workload, bounds[k], bounds[k + 1]) for k in range(procs) if bounds[k + 1] > bounds[k]]
    ctx = mp.get_context("spawn")  # never fork a process that may hold a CUDA context
    t0 = time.perf_counter()
    with ctx.Pool(len(jobs)) as pool:
        res = pool.map(_py_ref_worker, jobs)
    wall = time.perf_counter() - t0
    inter = sum(r[0] for r in res)
    trace_s = max(r[1] for r in res)  # the slowest worker bounds the parallel trace (scene build + imports excluded)
    return {"value": inter / trace_s, "unit": UNIT, "cores": len(jobs), "kind": "reference",
            "per_core": inter / sum(r[1] for r in res),
            "sample": f"first {n_sample} rays of the {workload} batch, unmodified optable package ({os.path.relpath(RH.REFERENCE_ROOT, ROOT)}) "
                      f"OpticalTable.ray_tracing, one process per core ({inter} interactions, slowest worker {trace_s:.2f} s, wall {wall:.1f} s)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = workloads()[args.workload]
    flat = w.flat()
    threads = os.cpu_count() or 1
    n_sample = args.ref_rays or w.cpu_rays
    for _ in range(args.warmup):
        cpu_arm(flat, max(n_sample // 10, 100), threads, workload=args.workload)
    total, dt = 0, 0.0
    for _ in range(args.steps):  # only the trace is timed (cpu_arm builds the synthetic rays outside its timer)
        _, inter, step_s = cpu_arm(flat, n_sample, threads, workload=args.workload)
        total += inter
        dt += step_s
    value = total / dt
    sample = f"first {n_sample} rays of the {args.workload} batch per step, oracle/optb_oracle.c (C port of the reference), {threads} threads"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "rays_per_step": n_sample, "surfaces": int(flat.n_leaves), "monitors": int(flat.n_monitors)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    # beside the port: the real Python reference on a smaller sample of the same batch (it is ~500x slower per core
    # than the C port, so the headline `value` above is the conservative denominator)
    try:
        py = python_reference_arm(args.workload, args.pyref_rays, threads)
    except Exception as e:  # never lose the line over the side leg
        py = {"unavailable": f"{type(e).__name__}: {e}"}
    line["cpu_baseline_reference"] = py if py is not None else {"unavailable": "baseline/_ref not present"}
    print(json.dumps(line))


def bind_to_gpu_numa_node(index):
    """Pin this rank (and the pinned host buffers it allocates next) to the CPUs closest to its GPU, so that the
    host<->device copies of eight ranks do not all cross one socket link. Best effort."""
    try:
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
    except Exception:
        pass


# ---- CUDA arm ----------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self):
        import torch

        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        bind_to_gpu_numa_node(self.local)
        self.dev = f"cuda:{self.local}"
        if self.world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device(self.dev))

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.barrier()

    def max_f(self, x):
        if self.world == 1:
            return float(x)
        import torch
        import torch.distributed as dist

        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_i(self, x):
        if self.world == 1:
            return int(x)
        import torch
        import torch.distributed as dist

        t = torch.tensor([x], device=self.dev, dtype=torch.int64)
        dist.all_reduce(t)
        return int(t.item())


def measure(args, D, engine, name, steps, warmup, e2e_steps, with_cpu, peaks, fp64_peak, dump=False):
    """One workload at D.world GPUs: device-timed value, end-to-end value through optb_trace_host, rooflines, CPU
    baseline. Returns the dict that becomes the JSON line (headline) or an entry of "workloads"."""
    import torch
    import torch.distributed as dist

    from optable_b200 import _abi as A
    from optable_b200.bundle import DeviceTrace

    w = workloads()[name]
    flat = w.flat()
    n = args.rays or w.rays_per_gpu
    bundle = w.bundle(n, D.rank * n)  # weak scaling: every rank traces its own n rays of the endless bundle
    rays_dev = bundle.to_torch(device=D.dev)
    hit_cap = n * w.rows_per_ray + 1024
    cols = E2E_COLUMNS if args.e2e_columns == "raw" else None
    dt = DeviceTrace(engine, flat, n, hit_cap, record_hist=True, max_trace_num=w.max_trace_num, chain_len=args.chain_len,
                     **({"hit_columns": cols} if cols else {}))
    stream = torch.cuda.current_stream()
    live = w.max_live * n or None  # live-ray budget of the wavefront (splitting scenes)

    def merge_monitors():
        # the only cross-GPU exchange of the path: monitor histograms (+ counters); rows stay sharded
        if D.world > 1:
            dist.all_reduce(dt.t["hist_y"])
            dist.all_reduce(dt.t["hist_yz"])

    for _ in range(max(warmup, 3)):
        dt.run(rays_dev, live)
        merge_monitors()
    torch.cuda.synchronize()
    cnt = dt.counters()
    engine._raise_status(cnt)
    inter, hits, launches = int(cnt[A.C_INTERACTIONS]), int(cnt[A.C_HITS]), int(cnt[A.C_LAUNCHES])
    pops = int(cnt[A.C_SEGMENTS])
    tests, curved, boxes = int(cnt[A.C_TESTS]), int(cnt[A.C_TESTS_CURVED]), int(cnt[A.C_BOX_TESTS])
    # ---- timed region: device-resident inputs, CUDA events on the launching stream, max over ranks ----
    step_bytes = bundle_bytes(bundle) + hits * dt.hit_row_bytes()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=D.dev) if step_bytes <= 126e6 else None
    sampler = ClockSampler(D.local)
    sampler.start()
    D.barrier()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    kern = []
    ev[0].record(stream)
    for k in range(steps):
        if flush is not None:
            flush.fill_(k & 0xff)  # the step's own traffic fits the 126 MB L2: write 256 MB between timed steps
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(stream)
        dt.run(rays_dev, live)
        k1.record(stream)
        merge_monitors()
        ev[k + 1].record(stream)
        kern.append((k0, k1))
    torch.cuda.synchronize()
    D.barrier()
    total_ms = D.max_f(ev[0].elapsed_time(ev[-1]))
    trace_ms = float(np.mean([a.elapsed_time(b) for a, b in kern]))
    clocks = sampler.stop()
    dumped = dump_outputs(args.dump_outputs, dt, n, D.world) if args.dump_outputs and dump and D.rank == 0 else None
    inter_all = D.sum_i(inter)
    ms_per_step = total_ms / steps
    value = inter_all / (ms_per_step * 1e-3)

    # ---- end to end through the C ABI with HOST buffers (optb_trace_host): H2D rays + D2H monitor rows ----
    hit_columns, hit_dtypes, row_bytes = dt.hit_columns, {k: dt.t[k].dtype for k in dt.hit_columns}, dt.hit_row_bytes()
    hist_shapes = (tuple(dt.t["hist_y"].shape), tuple(dt.t["hist_yz"].shape))
    for k in list(dt.t):  # the device-resident result buffers are not needed any more: give the memory back
        if k.startswith(("hit_", "seg_")):
            del dt.t[k]
    del rays_dev
    engine._workspace = None
    torch.cuda.empty_cache()
    flushed = flush is not None
    del flush
    e2e, e2e_hist = run_e2e(args, D, engine, dt, bundle, n, hit_cap, hit_columns, hit_dtypes, row_bytes, hist_shapes, inter,
                            hits, inter_all, e2e_steps)
    out = {"value": value, "unit": UNIT, "ms_per_step": ms_per_step, "steps": steps,
           "config": {"workload": name, "what": w.config, "rays_per_gpu": n, "surfaces": int(flat.n_leaves),
                      "monitors": int(flat.n_monitors), "max_trace_num": w.max_trace_num,
                      "interactions_per_step_per_gpu": inter, "pops_per_step_per_gpu": pops,
                      "monitor_rows_per_step_per_gpu": hits,
                      "leaf_tests_per_step_per_gpu": tests, "curved_leaf_tests_per_step_per_gpu": curved,
                      "box_tests_per_step_per_gpu": boxes,
                      "monitor_row_bytes": row_bytes,
                      "l2": "inputs+outputs per step (%.2f GB) exceed the 126 MB L2" % (step_bytes / 1e9) if not flushed else
                            "inputs+outputs per step (%.3f GB) fit the L2: a 256 MB buffer is written between timed steps (inside ms_per_step)" % (step_bytes / 1e9),
                      "parallelism": f"rays sharded over {D.world} GPU(s), scene tables replicated, histograms all-reduced"},
           "clocks": clocks, "gpu_launches": launches * steps, "e2e": e2e}
    if dumped:
        out["outputs_dump"] = dumped
    if e2e_hist:
        out["e2e_histograms_only"] = e2e_hist
    if D.rank == 0:
        out.update(rooflines(name, n, inter, pops, hits, tests, curved, boxes, row_bytes, bundle, trace_ms, peaks, fp64_peak))
        if with_cpu:
            threads = os.cpu_count() or 1
            try:
                os.sched_setaffinity(0, range(threads))  # the CPU baseline gets every host core again
            except Exception:
                pass
            cpu_rays = args.cpu_rays or w.cpu_rays
            cpu_val, cpu_inter, cpu_dt = cpu_arm(flat, cpu_rays, threads, workload=name)
            out["cpu_baseline"] = {"value": cpu_val, "unit": UNIT, "cores": threads, "kind": "port",
                                   "sample": f"first {cpu_rays} rays of the same batch ({cpu_inter} interactions in {cpu_dt:.2f} s), "
                                             f"oracle/optb_oracle.c with {threads} threads"}
            # the same FP64 bound with the work the REFERENCE's loop does per interaction (every child of a hit group box
            # is tested: component_group.py:98-115) instead of the tests this engine executed -- front-to-back dismissal
            # skips tests the formula of SURVEY 8(d) charges for, so the executed-work fraction above is the lower one
            from optable_b200 import _abi as A
            c = cpu_arm.counters
            fp = out["roofline"] if out["roofline"]["bound"] == "fp64" else out.get("roofline_fp64")
            if fp is not None and int(c[A.C_INTERACTIONS]) > 0:
                ref_flops = (FLOPS_PLANAR * (c[A.C_TESTS] - c[A.C_TESTS_CURVED]) + FLOPS_CURVED * c[A.C_TESTS_CURVED]
                             + FLOPS_BOX * c[A.C_BOX_TESTS] + FLOPS_INTERACT * c[A.C_INTERACTIONS]) / float(c[A.C_INTERACTIONS])
                a_ref = ref_flops * inter / (fp["kernel_ms"] * 1e-3) / 1e12
                fp["reference_loop"] = {"flops_per_interaction": float(ref_flops), "achieved": a_ref, "frac": a_ref / fp["peak"],
                                        "counts_from": f"oracle/optb_oracle.c on the first {cpu_rays} rays (the reference's loop, no dismissal)"}
            bind_to_gpu_numa_node(D.local)
    dt.scene.close()
    del dt
    torch.cuda.empty_cache()
    return out


DUMP_SEED = 0
DUMP_MAX_BYTES = 48 << 20  # monitor rows of the output sample; histograms and counts come on top (< 1 MB)


def dump_outputs(out_dir, dt, n_rays, world_size):
    """Write what the last timed step left in the device result buffers as DIR/<name>.npy (float64):
    the monitor histograms, the result counts (pops, interactions, monitor rows) and the monitor rows of a fixed,
    seeded sample of the initial rays, in (root, monitor, pop) order. Rows are appended in device order, so they are
    selected by their root ray and sorted by their packed key: two builds that compute the same rows write the same
    files. The sample has as many rays as keep the rows under DUMP_MAX_BYTES; if the chosen rays still yield more
    rows, the first rows in key order are kept. Only rank 0 writes: with --gpus > 1 the histograms are the
    all-reduced ones of every GPU, but the rows and counts are rank 0's shard (its own rays), and "world_size" in the
    line's "outputs_dump" says how many GPUs shared the batch."""
    import torch

    from optable_b200 import _abi as A

    os.makedirs(out_dir, exist_ok=True)
    cnt = dt.counters()
    rows = int(cnt[A.C_HITS])
    cols = ("hit_px", "hit_py", "hit_pz", "hit_intensity", "hit_t")
    row_bytes = 8 * (len(cols) + 3)  # + root, monitor and pop
    max_rows = DUMP_MAX_BYTES // row_bytes
    per_ray = rows / max(n_rays, 1)
    k = n_rays if per_ray * n_rays <= max_rows else max(1, int(max_rows / per_ray))
    roots = np.sort(np.random.default_rng(DUMP_SEED).choice(n_rays, size=k, replace=False)) if k < n_rays else None
    if "hit_key" in dt.t:
        key = dt.t["hit_key"][:rows]
    else:  # --e2e-columns all: the key is three columns
        u32 = lambda c: dt.t[c][:rows].to(torch.int64) & 0xffffffff  # noqa: E731
        key = (u32("hit_root") << 32) | (u32("hit_monitor") << 24) | u32("hit_pop")
    if roots is not None:
        chosen = torch.zeros(n_rays, dtype=torch.bool, device=key.device)
        chosen[torch.from_numpy(roots).to(key.device)] = True
        sel = torch.nonzero(chosen[key >> 32]).flatten()
    else:
        sel = torch.arange(rows, device=key.device)
    order = sel[torch.argsort(key[sel])][:max_rows]
    key = key[order]
    arrays = {"hit_root": key >> 32, "hit_monitor": (key >> 24) & 0xff, "hit_pop": key & 0xffffff}
    arrays.update({c: dt.t[c][:rows][order] for c in cols})
    arrays["hist_y"], arrays["hist_yz"] = dt.t["hist_y"], dt.t["hist_yz"]
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "counts.npy"), cnt[[A.C_SEGMENTS, A.C_INTERACTIONS, A.C_HITS]].astype(np.float64))
    return {"dir": out_dir, "rows": int(order.numel()), "rows_per_step": rows,
            "sampled_rays": n_rays if roots is None else k, "seed": DUMP_SEED, "world_size": world_size,
            "rows_from": "rank 0 (its own rays)" if world_size > 1 else "the whole batch"}


def bundle_bytes(bundle):
    return sum(np.asarray(c).nbytes for c in bundle.columns.values() if c is not None)


def rooflines(name, n, inter, pops, hits, tests, curved, boxes, row_bytes, bundle, trace_ms, peaks, fp64_peak):
    """Both bounds of SURVEY 8(d) for the dominant kernel (trace_kernel), from this run's own counters:
    fp64: algorithmic flops (formula above) / kernel time against the in-run DFMA peak;
    hbm:  persistent-form algorithmic bytes (every ray record read once and written once = 208 B per RAY, plus the
          monitor rows the step writes) / kernel time against the measured copy bandwidth. The larger fraction binds."""
    sec = trace_ms * 1e-3
    flops = FLOPS_PLANAR * (tests - curved) + FLOPS_CURVED * curved + FLOPS_BOX * boxes + FLOPS_INTERACT * inter
    hbm_peak, peak_src = (peaks.get("hbm_gbs"), "measured (MEASURED_PEAKS.json)") if peaks.get("hbm_gbs") else (6650.0, "fallback (B200_PROFILING.md)")
    alg_bytes = 2 * RAY_RECORD_BYTES * n + hits * row_bytes
    a_hbm = alg_bytes / sec / 1e9
    a_fp = flops / sec / 1e12
    r_hbm = {"bound": "hbm", "achieved": a_hbm, "peak": hbm_peak, "unit": "GB/s", "frac": a_hbm / hbm_peak, "traffic": None,
             "peak_source": peak_src, "kernel": "trace_kernel", "kernel_ms": trace_ms,
             "algorithmic_bytes": int(alg_bytes),
             "convention": "persistent form: 208 B per initial ray (record read + written once) + monitor row bytes; "
                           "SURVEY 8(d)'s wavefront-form figure (208 B per interaction) would be %.1f GB/s" % (208 * inter / sec / 1e9)}
    r_fp = {"bound": "fp64", "achieved": a_fp, "peak": fp64_peak["tflops"], "unit": "TFLOP/s", "frac": a_fp / fp64_peak["tflops"],
            "traffic": None,
            "peak_source": "measured in this run: optb_measure_fp64_peak (8 independent DFMA chains per thread), SM clock %s MHz while it ran" % fp64_peak.get("sm_mhz"),
            "kernel": "trace_kernel", "kernel_ms": trace_ms, "algorithmic_flops": int(flops),
            "flops_per_interaction": flops / max(inter, 1),
            "formula": "55*planar_leaf_tests + 200*curved_leaf_tests + 25*box_tests + 180*interactions (SURVEY 8d), counts from this run's device "
                       "counters = tests EXECUTED (tests skipped by front-to-back dismissal are not credited; reference_loop credits them)"}
    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from one `ncu --set full` capture of this very command
    # (profiles/r2_traffic.json names the capture); only valid for the batch size it was captured at
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            cap = json.load(f).get(name)
        if cap and int(cap["rays_per_gpu"]) == int(n):
            r_hbm["traffic"] = r_fp["traffic"] = int(cap["dram_bytes_per_launch"])
            r_hbm["traffic_source"] = r_fp["traffic_source"] = cap["source"]
    except (OSError, ValueError, KeyError):
        pass
    binding, other = (r_fp, r_hbm) if r_fp["frac"] >= r_hbm["frac"] else (r_hbm, r_fp)
    return {"roofline": binding, "roofline_" + other["bound"]: other}


def run_e2e(args, D, engine, dt, bundle, n, hit_cap, hit_columns, hit_dtypes, row_bytes, hist_shapes, inter_per_step,
            hits_per_step, inter_all, e2e_steps):
    import copy

    import torch

    from optable_b200 import _abi as A
    from optable_b200.flatten import rays_struct

    if e2e_steps <= 0:
        return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "steps": 0}, None
    host = bundle.to_torch(pin=True)
    host_np = {k: v.numpy() for k, v in host.items()}
    host_np["length"] = None
    rs = rays_struct({**{k: None for k in A.RAY_F64}, **host_np})
    rs.n = n
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    hy = torch.zeros(hist_shapes[0], dtype=torch.int64).pin_memory()
    hyz = torch.zeros(hist_shapes[1], dtype=torch.int64).pin_memory()
    hc = torch.zeros(A.C_COUNT, dtype=torch.int64).pin_memory()
    small = hy.numel() * 8 + hyz.numel() * 8 + A.C_COUNT * 8

    def timed(res, prm):
        for _ in range(2):
            engine.trace_host(dt.scene, rs, prm, res)
        torch.cuda.synchronize()
        D.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            engine.trace_host(dt.scene, rs, prm, res)
        torch.cuda.synchronize()
        s = D.max_f(time.perf_counter() - t0)
        assert int(hc[A.C_STATUS]) == 0 and int(hc[A.C_INTERACTIONS]) == inter_per_step, (hc.tolist(), inter_per_step)
        return inter_all * e2e_steps / s

    rows_gb = hits_per_step * row_bytes / 1e9
    e2e = None
    if rows_gb <= args.e2e_max_row_gb:
        prm_rows = copy.copy(dt.prm)
        prm_rows.sorted_rows = 1  # rows arrive in (root, monitor, pop) order: what Monitor._data_raw would hold
        res = A.Result()
        res.seg_capacity, res.hit_capacity = 0, hit_cap
        host_out = {}
        for k in hit_columns:
            host_out[k] = torch.empty(hit_cap, dtype=hit_dtypes[k]).pin_memory()
            setattr(res, k, host_out[k].data_ptr())
        res.hist_y, res.hist_yz, res.counters = hy.data_ptr(), hyz.data_ptr(), hc.data_ptr()
        v = timed(res, prm_rows)
        keys = host_out["hit_key"][:hits_per_step].numpy() if "hit_key" in host_out else None
        if keys is not None:
            ku = keys.view(np.uint64)
            assert bool((ku[1:] >= ku[:-1]).all()), "rows not in reference order"
        e2e = {"value": v, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(hits_per_step * row_bytes + small),
               "steps": e2e_steps, "api": "optb_trace_host (C ABI, pinned host buffers)",
               "result": f"every monitor row ({row_bytes} B: {', '.join(c[4:] for c in hit_columns)}) in (root, monitor, pop) order + histograms + counters",
               "input_encoding": "%d real fp64 columns + %d broadcast (one value for all rays)" % (
                   sum(1 for v in host.values() if v.numel() > 1), sum(1 for v in host.values() if v.numel() == 1))}
        del host_out, res
    # the same call when the caller only wants the monitors' histograms back (no row columns)
    prm2 = copy.copy(dt.prm)
    prm2.record_hits = 0
    res2 = A.Result()
    res2.hist_y, res2.hist_yz, res2.counters = hy.data_ptr(), hyz.data_ptr(), hc.data_ptr()
    vh = timed(res2, prm2)
    e2e_hist = {"value": vh, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(small), "steps": e2e_steps,
                "api": "optb_trace_host (C ABI, pinned host buffers)", "result": "monitor histograms + counters (no row columns)"}
    if e2e is None:  # rows of this workload exceed the host-memory budget of the bench: histogram result is the e2e
        e2e = dict(e2e_hist)
        e2e["note"] = "monitor rows per step (%.1f GB per GPU) exceed --e2e-max-row-gb: the end-to-end result is the histogram set" % rows_gb
        e2e_hist = None
    return e2e, e2e_hist


def run_cuda(args):
    import torch
    import torch.distributed as dist

    from optable_b200.backend import Engine

    D = Dist()
    engine = Engine.get(D.local)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # DFMA peak with its own clock sample (the denominator of roofline_fp64)
    s = ClockSampler(D.local)
    s.start()
    fp64 = engine.fp64_peak_tflops()
    c = s.stop()
    fp64_peak = {"tflops": fp64, "sm_mhz": c.get("sm_mhz"), "reasons": c.get("reasons")}
    head = measure(args, D, engine, args.workload, args.steps, args.warmup, min(args.e2e_steps, args.steps), True, peaks, fp64_peak,
                   dump=True)
    extra = {}
    if not args.only:
        for name in workloads():
            if name == args.workload:
                continue
            extra[name] = measure(args, D, engine, name, max(1, min(args.steps, args.extra_steps)), 3,
                                  min(args.e2e_steps, 3), True, peaks, fp64_peak)
    flagged = None
    if D.rank == 0 and args.flag_rays > 0:
        flagged = flagged_fraction(engine, args.workload, args.flag_rays)
    if D.rank == 0:
        cfg = head.pop("config")
        line = {"metric": METRIC, "value": head.pop("value"), "unit": UNIT, "n_gpus": D.world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": head.pop("ms_per_step"), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg}
        head.pop("unit", None)
        head.pop("steps", None)
        line.update(head)
        line["fp64_peak"] = fp64_peak
        if flagged is not None:
            line["flagged_fraction"] = flagged
        if extra:
            line["workloads"] = extra
        print(json.dumps(line))
    if D.world > 1:
        dist.destroy_process_group()


def flagged_fraction(engine, workload, n):
    """Share of initial rays whose hit index / bounce count hinge on less than the stated epsilon (SURVEY A.9),
    computed on the device (params.flag_ambiguity) for the first n rays of the workload. Outside the timed region."""
    from optable_b200 import _abi as A
    from optable_b200.bundle import DeviceTrace

    try:
        w = workloads()[workload]
        flat = w.flat()
        dt = DeviceTrace(engine, flat, n, 0, record_hist=False, max_trace_num=w.max_trace_num, flag_ambiguity=True)
        dt.run(w.bundle(n, 0).to_torch(device=f"cuda:{engine.device}"), w.max_live * n or None)
        cnt = dt.counters()
        return {"value": int(cnt[A.C_FLAGGED]) / n, "rays": n, "flagged": int(cnt[A.C_FLAGGED]),
                "rule": "SURVEY A.9 (OPTB_AMB_* bits of include/optb.h), evaluated in-kernel at every pop"}
    except Exception as e:
        return {"value": None, "error": f"{type(e).__name__}: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline workload (also caps --e2e-steps)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--rays", type=int, default=0, help="rays per GPU per step (0 = the workload's default)")
    ap.add_argument("--workload", default=WORKLOAD, choices=list(workloads()))
    ap.add_argument("--only", action="store_true", help="measure only --workload (skip the other BASELINE configs)")
    ap.add_argument("--extra-steps", type=int, default=5, help="timed steps of the workloads reported under \"workloads\"")
    ap.add_argument("--cpu-rays", type=int, default=0, help="bounded sample for the in-run CPU baseline (0 = per workload)")
    ap.add_argument("--ref-rays", type=int, default=0, help="rays per step of the reference arm (0 = per workload)")
    ap.add_argument("--pyref-rays", type=int, default=2000, help="sample of the kind=reference (pure Python) leg of --impl reference")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-columns", default="raw", choices=["raw", "all"],
                    help="monitor row of the end-to-end leg: raw = Monitor._data_raw fields + key (52 B); all = + direction and q (92 B)")
    ap.add_argument("--e2e-max-row-gb", type=float, default=6.0,
                    help="largest per-GPU row set the end-to-end leg copies to pinned host memory; above it e2e returns histograms")
    ap.add_argument("--flag-rays", type=int, default=1_000_000, help="rays of the ambiguity-flag pass (0 = skip)")
    ap.add_argument("--chain-len", type=int, default=0, help="max in-register pops per launch (0 = unlimited); scheduling only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline workload's results of the last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "cuda":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
