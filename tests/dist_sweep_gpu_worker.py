"""Worker of tests/test_gpu_dist_sweep.py: run under `python -m torch.distributed.run --nproc-per-node N` (one rank per
GPU, NCCL). Sweeps sharded over the ranks by configuration (`trace_sweep` / `SweepScene.trace` with `group=True`)
against the one-GPU sweep of the same configurations, bit for bit: every hit column, the histograms, every key of
stats() and every counter but the launch and generation counts. Also the recipe of a C host: per-rank sweeps of its
own configurations, root keys shifted by k0 * N, histograms merged with optb_monitor_merge over [K][M] buffers."""
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import optable_b200 as ob  # noqa: E402
from optable_b200 import _abi as A  # noqa: E402
from optable_b200 import backend  # noqa: E402
from optable_b200.bundle import RayBundle  # noqa: E402
from optable_b200.dist import shard_bounds  # noqa: E402
from optable_b200.flatten import FlatScene  # noqa: E402
from optable_b200.sweep import SweepScene, trace_sweep  # noqa: E402
from optable_b200.workloads import WORKLOADS, ripa, telescope_4f_grid  # noqa: E402
from tests import scenes  # noqa: E402

HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64
SAME_COUNTERS = [c for c in range(A.C_COUNT) if c not in (A.C_LAUNCHES, A.C_GENERATIONS)]


def host(v):
    return np.ascontiguousarray(v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v))


def same_rows(got, want, what):
    assert len(got["hit_root"]) == len(want["hit_root"]), f"{what}: {len(got['hit_root'])} != {len(want['hit_root'])} rows"
    for c in HIT_COLS:
        assert np.array_equal(host(got[c]).view(np.uint8), host(want[c]).view(np.uint8)), f"{what}: column {c}"


def same_result(got, want, what):
    """Every hit column (after gather), histograms, every stats() key (NaN-aware), counters but launches/generations."""
    same_rows(got.hits, want.hits, what)
    assert torch.equal(got.hist_y, want.hist_y) and torch.equal(got.hist_yz, want.hist_yz), f"{what}: histograms"
    a, b = got.stats(), want.stats()
    assert a.keys() == b.keys()
    for q in a:
        assert np.array_equal(a[q], b[q], equal_nan=True), f"{what}: stats {q}"
    assert np.array_equal(np.asarray(got.counters)[SAME_COUNTERS], np.asarray(want.counters)[SAME_COUNTERS]), \
        f"{what}: counters {got.counters} != {want.counters}"


def plan_bits(engine, flats, n, limit, chain_len):
    """The trace_kernel variant (OPTB_PLAN_* bits; where the histograms accumulate is not a variant) of a sweep."""
    scene = engine.upload_sweep(flats)
    try:
        arrs = {"ox": np.zeros(n), "family": np.arange(n, dtype=np.int32)}
        plan = engine.trace_plan(scene, arrs, max_trace_num=limit, record_segments=False, record_hist=True,
                                 chain_len=chain_len)
    finally:
        scene.close()
    return plan["bits"] & ~A.PLAN_HIST_SMEM


def moving(obj, step):
    """configure(k): `obj` (and everything below it) back to its first pose, then moved by k * step along x. Absolute,
    as SweepScene.trace requires: a rank configures only its own k."""
    saved = []

    def walk(o):
        saved.append((o, o.origin.copy(), np.array(o.transform_matrix, dtype=np.float64), o._bbox))
        for c in getattr(o, "components", []):
            walk(c)

    walk(obj)

    def configure(k):
        for o, org, T, box in saved:
            o.origin, o.transform_matrix, o._bbox = org.copy(), T.copy(), box
        obj.TX(step * k)

    return configure


def grid_tables(K):
    F = 43.17 + np.linspace(-1.5, 1.5, 16)
    return [telescope_4f_grid(ob, F[k // 16 % 16], F[k % 16]) for k in range(K)]


def slab_tables(K):
    """The splitting slab whose faces reflect nothing in configuration 0."""
    def one(k):
        slab = ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=1, n2=1.5, reflectivity=0.05 * k)
        slab.RotZ(0.02 * (k - 1))
        return scenes.Scene([ob.Mirror([-2, 0, 0], radius=3, reflectivity=0.9, transmission=0.0), slab,
                             ob.Mirror([2, 0, 0], radius=3, reflectivity=0.9, transmission=0.0).RotZ(np.pi)],
                            [], [ob.Monitor([1, 0, 0], 6, 6), ob.Monitor([-3, 0, 0], 6, 6)])
    return [one(k) for k in range(K)]


def case_4f_grid(engine, rank, world):
    """4f grid, trace_sweep, K = 256, N = 1000: gathered, and each rank's own rows(k) without gather. Returns the
    one-GPU sweep and the case for the C-host recipe."""
    K, n = 256, 1000
    tables, bundle = grid_tables(K), RayBundle.collimated_disc(n, radius=2.5)
    one = trace_sweep(tables, bundle, record_hist=True, engine=engine)
    res = trace_sweep(tables, bundle, record_hist=True, engine=engine, group=True, gather=True)
    k0, k1 = shard_bounds(K, rank, world)
    assert res.shard == (k0, k1) and res.n_configs == K and res.chain_len == 0
    same_result(res, one, "4f grid, gather=True")
    mine = trace_sweep(tables, bundle, record_hist=True, engine=engine, group=True)
    same_rows(mine.hits, {c: v[one._bounds[k0]:one._bounds[k1]] for c, v in one.hits.items()}, "4f grid, own rows")
    for k in range(k0, k1):
        same_rows(mine.rows(k), one.rows(k), f"4f grid, rows({k}) on rank {rank}")
    assert torch.equal(mine.hist_y, one.hist_y) and torch.equal(mine.hist_yz, one.hist_yz), "4f grid, gather=False"
    for q, v in mine.stats().items():
        assert np.array_equal(v, one.stats()[q], equal_nan=True), f"4f grid, gather=False: stats {q}"
    if rank == 0:
        print(f"SWEEP_CASE_OK 4f_grid: K={K} N={n} on {world} GPUs, {len(one.hits['hit_root'])} rows bit-identical", flush=True)
    return one, tables, bundle


def c_host_recipe(engine, rank, world, one, tables, bundle):
    """What a C host does: a sweep of its own configurations, root keys + k0 N, optb_monitor_merge over [K][M] buffers
    that are zero outside its slice."""
    K, n = len(tables), bundle.n
    k0, k1 = shard_bounds(K, rank, world)
    L = backend.lib()
    L.optb_comm_unique_id.argtypes = [C.c_void_p, C.c_void_p]
    L.optb_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.optb_monitor_merge.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.optb_comm_destroy.argtypes = [C.c_void_p]
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        buf = (C.c_char * 128)()
        engine._check(L.optb_comm_unique_id(engine._ctx, buf))
        uid = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
    uid = uid.cuda()
    dist.broadcast(uid, 0)
    engine._check(L.optb_comm_init(engine._ctx, bytes(uid.cpu().numpy().tobytes()), rank, world))
    part = trace_sweep(tables[k0:k1], bundle, record_hist=True, engine=engine) if k1 > k0 else None
    M = len(tables[0].monitors)
    hy = torch.zeros((K, M, A.HIST_BINS), dtype=torch.int64, device="cuda")
    hyz = torch.zeros((K, M, A.HIST_BINS, A.HIST_BINS), dtype=torch.int64, device="cuda")
    cnt = torch.zeros(A.C_COUNT, dtype=torch.int64, device="cuda")
    if part is not None:
        hy[k0:k1], hyz[k0:k1] = part.hist_y, part.hist_yz
        cnt.copy_(torch.from_numpy(np.asarray(part.counters, dtype=np.int64)))
        root = (part.hits["hit_root"].long() & 0xFFFFFFFF) + k0 * n
        assert torch.equal(root, one.hits["hit_root"][one._bounds[k0]:one._bounds[k1]].long() & 0xFFFFFFFF)
    engine._check(L.optb_monitor_merge(engine._ctx, hy.data_ptr(), hyz.data_ptr(), K * M, cnt.data_ptr(),
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    engine._check(L.optb_comm_destroy(engine._ctx))
    assert torch.equal(hy, one.hist_y) and torch.equal(hyz, one.hist_yz), "C-host recipe: merged histograms"
    assert np.array_equal(host(cnt)[SAME_COUNTERS], np.asarray(one.counters)[SAME_COUNTERS]), "C-host recipe: counters"
    if rank == 0:
        print("SWEEP_CABI_OK optb_monitor_merge over [K][M] slices", flush=True)


def case_ripa(engine, rank, world):
    """ripa SweepScene, one mirror of the first group moving, K = 8, N = 1e4, max_trace_num 40."""
    K, limit = 8, {"max_trace_num": 40}
    w = WORKLOADS["c5_ripa_64"]
    rbundle = w.bundle(10_000, 0)
    results = []
    for group in (None, True):
        sc = ripa(ob, n_rays=0)
        mirror = sc.components[0].components[1]
        configure = moving(mirror, 2e-4)

        results.append((SweepScene(sc, [mirror]).trace(rbundle, configure, K, limit, record_hist=True, engine=engine,
                                                      group=group, gather=True), mirror))
    (one_r, m1), (res_r, m2) = results
    same_result(res_r, one_r, "ripa SweepScene, gather=True")
    assert np.array_equal(m1.origin, m2.origin), "the table stands in configuration K - 1"
    if rank == 0:
        print(f"SWEEP_CASE_OK ripa: K={K} N=10000 on {world} GPUs, {len(one_r.hits['hit_root'])} rows bit-identical", flush=True)


def case_slab(engine, rank, world):
    """The splitting slab, reflectivity 0 in configuration 0, which rank 0 traces alone: every rank runs the variant
    of the one-GPU sweep."""
    K, lim = world + 1, 40
    tables = slab_tables(K)
    sbundle = RayBundle.collimated_disc(2000, x0=-1.5, radius=0.6, direction=(1.0, 0.01, 0.0))
    one_s = trace_sweep(tables, sbundle, {"max_trace_num": lim}, record_hist=True, engine=engine)
    res_s = trace_sweep(tables, sbundle, {"max_trace_num": lim}, record_hist=True, engine=engine, group=True, gather=True)
    same_result(res_s, one_s, "splitting slab, gather=True")
    k0, k1 = res_s.shard
    flats = [FlatScene(t.components, t.monitors) for t in tables]
    want_bits = plan_bits(engine, flats, sbundle.n, lim, 0)
    assert want_bits & A.PLAN_SPLIT
    got_bits = plan_bits(engine, flats[k0:k1], sbundle.n, lim, res_s.chain_len)
    assert got_bits == want_bits, f"rank {rank}: variant {got_bits:#x} != one-GPU {want_bits:#x}"
    if rank == 0:
        alone = plan_bits(engine, flats[k0:k1], sbundle.n, lim, 0)
        assert res_s.chain_len == lim + 1 and not alone & A.PLAN_SPLIT, (res_s.chain_len, alone)
        print(f"SWEEP_CASE_OK slab: variant {want_bits:#x} on every rank (rank 0 alone would run {alone:#x})", flush=True)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    engine = backend.Engine.get(local)
    one, tables, bundle = case_4f_grid(engine, rank, world)
    c_host_recipe(engine, rank, world, one, tables, bundle)
    case_ripa(engine, rank, world)
    case_slab(engine, rank, world)
    if rank == 0:
        print("SWEEP_DIST_OK", flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
