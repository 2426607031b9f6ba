"""GPU: optb_trace_host (host buffers in, host buffers out) against the device entry points the suite already trusts:
`trace_arrays` (optb_trace + a sort), `trace_sweep` and a device-resident DeviceTrace. One chunk and the chunked path
above 3 Mi rays, with sorted rows, segments, interact caps, sweeps, the live-ray grow loop and the rerun as one chunk
when a chunk outgrows its share of the result capacity."""
import copy
import re

import numpy as np
import pytest

import optable_b200 as ob
from optable_b200 import _abi as A
from tests import scenes

pytestmark = pytest.mark.gpu

SEG_COLS = A.SEG_F64 + A.SEG_U32 + A.SEG_I32
HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64
# counter slots that do not depend on the live-ray budget (a larger wavefront capacity runs fewer, larger generations)
WORK = [c for c in range(A.C_COUNT) if c not in (A.C_LAUNCHES, A.C_GENERATIONS)]


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _pinned(shape, dtype, fill=None):
    import torch

    t = torch.empty(shape, dtype=dtype, pin_memory=True)
    if fill is not None:
        t.fill_(fill)
    return t.numpy()


def _host_buffers(rays, seg_cap, hit_cap, n_hist=1, cap_counts=None):
    """Pinned copies of the ray columns (dict of numpy arrays; length 1 = broadcast) and pinned result buffers of every
    row column; returns (optb_rays, optb_result, dict of the result arrays)."""
    import torch

    from optable_b200.flatten import rays_struct

    staged = {}
    for k in A.RAY_F64 + ("flags", "family"):
        a = rays.get(k)
        if a is not None:
            staged[k] = torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    rs = rays_struct(staged)
    res = A.Result()
    res.seg_capacity, res.hit_capacity = seg_cap, hit_cap
    out = {}
    for cols, cap in ((SEG_COLS, seg_cap), (HIT_COLS, hit_cap)):
        for k in cols:
            out[k] = _pinned(cap, torch.float64 if k in A.SEG_F64 + A.HIT_F64 else torch.int32)
    out["hist_y"] = _pinned((n_hist, A.HIST_BINS), torch.int64, -1)
    out["hist_yz"] = _pinned((n_hist, A.HIST_BINS, A.HIST_BINS), torch.int64, -1)
    out["counters"] = _pinned(A.C_COUNT, torch.int64, -1)
    if cap_counts is not None:
        out["cap_counts"] = _pinned(cap_counts.shape, torch.int32)
        out["cap_counts"][:] = cap_counts
    for k, v in out.items():
        setattr(res, k, v.ctypes.data)
    return rs, res, out


def host_trace(engine, scene, rays, prm, seg_cap, hit_cap, **kw):
    """optb_trace_host with pinned host buffers; returns the filled row prefixes (uint32 columns as uint32),
    histograms, counters and cap_counts."""
    rs, res, out = _host_buffers(rays, seg_cap, hit_cap, **kw)
    engine.trace_host(scene, rs, prm, res)
    cnt = out["counters"]
    nseg = int(cnt[A.C_SEGMENTS]) if prm.record_segments else 0
    nhit = int(cnt[A.C_HITS]) if prm.record_hits else 0
    got = {k: v[:nseg] for k, v in out.items() if k in SEG_COLS}
    got.update({k: v[:nhit] for k, v in out.items() if k in HIT_COLS})
    got.update({k: v for k, v in out.items() if k not in SEG_COLS + HIT_COLS})
    for k in A.SEG_U32 + A.HIT_U32:
        got[k] = got[k].view(np.uint32)
    return got


def sorted_params(prm):
    p = copy.copy(prm)
    p.sorted_rows = 1
    return p


def assert_rows_equal(got, want, cols):
    for k in cols:
        assert len(got[k]) == len(want[k]), k
        assert np.array_equal(np.asarray(got[k]).view(np.uint8), np.asarray(want[k]).view(np.uint8)), k


def test_small_batch_sorted_rows_equal_trace_arrays(engine):
    """One chunk of a scene that cannot split: sorted segments and monitor rows equal trace_arrays bit for bit, and
    histograms and all 12 counters equal optb_trace's on the same rays."""
    from optable_b200.bundle import RayBundle

    sc = scenes.telescope_4f(ob, n_rays=0)
    scene = engine.upload(sc.flat())
    n, limit = 3000, 100
    arrs = RayBundle.collimated_disc(n, start=99).materialise()
    want = engine.trace_arrays(scene, arrs, max_trace_num=limit, record_hist=True)
    prm = sorted_params(engine.make_params(limit, record_hist=True, n_families=n))
    m = sc.flat().n_monitors
    got = host_trace(engine, scene, arrs, prm, 6 * n, 6 * n, n_hist=m)
    assert len(got["seg_root"]) == 5 * n and len(got["hit_root"]) > 0
    assert_rows_equal(got, want, SEG_COLS + HIT_COLS)
    np.testing.assert_array_equal(got["hist_y"], want["hist_y"][:m])
    np.testing.assert_array_equal(got["hist_yz"], want["hist_yz"][:m])
    np.testing.assert_array_equal(got["counters"], want["counters"])
    scene.close()


def test_splitting_scene_grows_the_live_budget():
    """A stack of partial mirrors: 64 roots need far more live rays than the grow loop's first budget (1024 on a fresh
    context). Rows and counters equal trace_arrays."""
    from optable_b200.backend import Engine

    fresh = Engine(0)  # its own context: no live-ray hint from earlier calls
    comps = [ob.Mirror([float(x), 0, 0], radius=3, reflectivity=0.6, transmission=0.4).RotZ(0.002 * k)
             for k, x in enumerate(range(0, 16, 2))]
    sc = scenes.Scene(comps, [], [ob.Monitor([20, 0, 0], 8, 8)])
    scene = fresh.upload(sc.flat())
    n, limit = 64, 2000
    arrs = scenes.ray_arrays(n, [-1, 0, 0], [0, 0.5, 0.5], [1, 0, 0], [0, 0, 0])
    prm = fresh.make_params(limit, n_families=n)
    probe, t = fresh.alloc_result(scene, n * limit, n * limit, n)
    fresh.trace_device(scene, fresh.rays_to_device(arrs), prm, probe, max_live=1024)
    assert int(t["counters"][A.C_STATUS]) & A.ST_WORK_OVERFLOW, "the first live budget was meant to be too small"
    want = fresh.trace_arrays(scene, arrs, max_trace_num=limit)
    got = host_trace(fresh, scene, arrs, sorted_params(prm), n * limit, n * limit)
    assert int(got["counters"][A.C_DROPPED]) > 0
    assert_rows_equal(got, want, SEG_COLS + HIT_COLS)
    np.testing.assert_array_equal(got["counters"][WORK], want["counters"][WORK])
    scene.close()


def test_binding_caps_with_family_column(engine):
    """Interact caps that bind, rays sharing ids (the family-serial path): cap_counts in and out and the rows equal
    trace_arrays from the same starting counts."""
    from optable_b200.flatten import pack_rays

    sc = scenes.caps_binding(ob)
    flat = sc.flat()
    scene = engine.upload(flat)
    arrs, fam_ids, unit = pack_rays(sc.rays)
    n, nfam, limit = len(arrs["ox"]), len(fam_ids), 80
    caps0 = np.random.default_rng(5).integers(0, 2, (flat.n_capslots, nfam)).astype(np.int32)
    want = engine.trace_arrays(scene, arrs, max_trace_num=limit, unit=unit, n_families=nfam, cap_counts=caps0)
    prm = sorted_params(engine.make_params(limit, unit, n_families=nfam))
    got = host_trace(engine, scene, arrs, prm, n * limit, n * limit * flat.n_monitors, cap_counts=caps0)
    assert not np.array_equal(got["cap_counts"], caps0)
    np.testing.assert_array_equal(got["cap_counts"], want["cap_counts"])
    assert_rows_equal(got, want, SEG_COLS + HIT_COLS)
    np.testing.assert_array_equal(got["counters"][WORK], want["counters"][WORK])
    scene.close()


def test_sweep_histograms_and_sorted_rows_equal_trace_sweep(engine):
    """A sweep scene (K = 3): histograms come back as [K][M] and equal trace_sweep's, and so do the sorted monitor
    rows (configuration-major)."""
    from optable_b200.bundle import RayBundle
    from optable_b200.flatten import FlatScene, batch_wavelengths_m
    from optable_b200.sweep import trace_sweep
    from optable_b200.workloads import telescope_4f_grid

    tables = [telescope_4f_grid(ob, 43.17 + d, 43.17) for d in (-1.0, 0.0, 0.7)]
    n, K = 500, len(tables)
    bundle = RayBundle.collimated_disc(n, start=3)
    want = trace_sweep(tables, bundle, record_hist=True, engine=engine)
    wls = batch_wavelengths_m(bundle.columns["wavelength"], getattr(tables[0], "unit", 1e-2))
    flats = [FlatScene(t.components, t.monitors, wavelengths_m=wls) for t in tables]
    M = flats[0].n_monitors
    scene = engine.upload_sweep(flats)
    prm = sorted_params(engine.make_params(2000, record_segments=False, record_hist=True, n_families=K * n))
    got = host_trace(engine, scene, dict(bundle.columns), prm, 0, 2 * K * n * M, n_hist=K * M)
    np.testing.assert_array_equal(got["hist_y"].reshape(K, M, A.HIST_BINS), want.hist_y.cpu().numpy())
    np.testing.assert_array_equal(got["hist_yz"].reshape(K, M, A.HIST_BINS, A.HIST_BINS), want.hist_yz.cpu().numpy())
    assert_rows_equal(got, {k: v.cpu().numpy() for k, v in want.hits.items()}, HIT_COLS)
    np.testing.assert_array_equal(got["counters"][WORK], np.asarray(want.counters)[WORK])
    scene.close()


def _big_trace(engine, n, seg_capacity, dx=None):
    """The benchmark scene and bundle at n rays, traced device-resident (DeviceTrace); `dx`: a direction x column.
    Returns the DeviceTrace and the ray columns as numpy arrays."""
    import torch

    import bench
    from optable_b200.bundle import DeviceTrace

    cols = {k: v.numpy() for k, v in bench.make_bundle(n, 777).to_torch().items()}
    if dx is not None:
        cols["dx"] = dx
    dt = DeviceTrace(engine, bench.build_scene(), n, 2 * n, seg_capacity=seg_capacity, record_hist=True)
    dt.run({k: torch.from_numpy(v).cuda() for k, v in cols.items()})
    return dt, cols


def _key_sorted(t, cols, rows, key_cols):
    """Device rows [:rows] of `cols` sorted by their row key (root << 32 | monitor << 24 | pop, or root << 32 | pop)."""
    import torch

    u32 = lambda c: t[c][:rows].to(torch.int64) & 0xFFFFFFFF  # noqa: E731
    key = u32(key_cols[0]) << 32
    if len(key_cols) == 3:
        key |= u32(key_cols[1]) << 24
    key |= u32(key_cols[-1])
    order = torch.argsort(key, stable=True)
    return {k: t[k][:rows][order].cpu().numpy() for k in cols}


def test_chunked_sorted_rows_with_segments_equal_device_trace(engine):
    """3.3 Mi rays (chunked, sorted_rows = 1, segments recorded): segment and monitor rows come back in key order and
    equal the device trace's rows sorted by key."""
    import torch

    n = 3_300_000
    dt, cols = _big_trace(engine, n, 5 * n + 1024)
    cnt = dt.counters()
    nseg, nhit = int(cnt[A.C_SEGMENTS]), int(cnt[A.C_HITS])
    got = host_trace(engine, dt.scene, cols, sorted_params(dt.prm), nseg, 2 * n, n_hist=2)
    hc = got["counters"]
    assert int(hc[A.C_STATUS]) == 0 and int(hc[A.C_LAUNCHES]) > int(cnt[A.C_LAUNCHES]), "meant to run in chunks"
    for c in (A.C_SEGMENTS, A.C_INTERACTIONS, A.C_HITS, A.C_DROPPED):
        assert int(hc[c]) == int(cnt[c]), c
    np.testing.assert_array_equal(got["hist_y"], dt.t["hist_y"].cpu().numpy())
    want = _key_sorted(dt.t, SEG_COLS, nseg, ("seg_root", "seg_pop"))
    assert_rows_equal(got, {k: v.view(np.uint32) if k in A.SEG_U32 else v for k, v in want.items()}, SEG_COLS)
    want = _key_sorted(dt.t, HIT_COLS, nhit, ("hit_root", "hit_monitor", "hit_pop"))
    assert_rows_equal(got, {k: v.view(np.uint32) if k in A.HIT_U32 else v for k, v in want.items()}, HIT_COLS)
    dt.close()
    torch.cuda.empty_cache()


def test_chunk_overflow_reruns_as_one_chunk(engine):
    """3.3 Mi rays of which only the first 1 Mi reach the monitors, hit_capacity = the exact total: chunk 0 outgrows
    its estimated share, so the call reruns as one chunk. Rows, histograms and all 12 counters equal the device
    trace's."""
    import torch

    n = 3_300_000
    dx = np.ones(n)
    dx[1 << 20:] = -1.0  # these rays leave the scene backwards
    dt, cols = _big_trace(engine, n, 0, dx=dx)
    cnt = dt.counters()
    nhit = int(cnt[A.C_HITS])
    assert nhit > 0 and int(dt.t["hit_root"][:nhit].max()) < (1 << 20)
    got = host_trace(engine, dt.scene, cols, sorted_params(dt.prm), 0, nhit, n_hist=2)
    np.testing.assert_array_equal(got["counters"], cnt)
    np.testing.assert_array_equal(got["hist_y"], dt.t["hist_y"].cpu().numpy())
    np.testing.assert_array_equal(got["hist_yz"], dt.t["hist_yz"].cpu().numpy())
    want = _key_sorted(dt.t, HIT_COLS, nhit, ("hit_root", "hit_monitor", "hit_pop"))
    assert_rows_equal(got, {k: v.view(np.uint32) if k in A.HIT_U32 else v for k, v in want.items()}, HIT_COLS)
    dt.close()
    torch.cuda.empty_cache()


def test_rejections_match_optb_trace(engine):
    """Options the library refuses fail through optb_trace_host with optb_trace's code and message, and leave the
    caller's counters alone."""
    from optable_b200.backend import BackendError
    from optable_b200.bundle import RayBundle

    flat = scenes.telescope_4f(ob, n_rays=0).flat()
    n = 64
    arrs = RayBundle.collimated_disc(n, radius=2.5).materialise()
    del arrs["family"]
    single, sweep = engine.upload(flat), engine.upload_sweep([flat, flat, flat])
    for scene, msg in ((single, "flag_ambiguity needs result.root_flags [rays.n]"),
                       (sweep, "sweep: flag_ambiguity and reference_roots are not available on sweep scenes")):
        prm = engine.make_params(80, record_segments=False, record_hits=False, n_families=3 * n, flag_ambiguity=True)
        rs, res, out = _host_buffers(arrs, 0, 0)
        with pytest.raises(BackendError, match=re.escape(f"liboptb error -7: {msg}")):
            engine.trace_host(scene, rs, prm, res)
        assert (out["counters"] == -1).all()
    single.close()
    sweep.close()
