"""GPU: monitor histograms and monitor statistics against numpy, exactly, at the bin edges.

The contract is np.histogram(y, bins=30, range=(-w/2, w/2)) (and np.histogram2d for the (y, z) histogram), both for the
histograms a trace accumulates (record_hist) and for the monitor statistics (optb_monitor_stats_grouped). Comparing one
device histogram with another cannot see a binning error, so every comparison here is with numpy of the rows themselves."""
import ctypes as C
import math

import numpy as np
import pytest

from tests import golden_io
from tests import hist_cases as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


# ---- optb_monitor_stats_grouped on row columns built directly ----------------------------------------------------
def _rows(y, z, seed=1, monitor=None, d=None):
    """Row columns of a monitor whose local hit points are (0, y, z), as CUDA tensors."""
    import torch

    n = len(y)
    rng = np.random.default_rng(seed)
    if d is None:
        d = np.stack([np.ones(n), rng.normal(0, 1e-2, n), rng.normal(0, 1e-2, n)], 1)
        d /= np.linalg.norm(d, axis=1, keepdims=True)
    host = {"hit_px": np.zeros(n), "hit_py": np.asarray(y, np.float64), "hit_pz": np.asarray(z, np.float64),
            "hit_intensity": rng.uniform(0.1, 2.0, n), "hit_t": rng.uniform(1.0, 50.0, n),
            "hit_dx": d[:, 0], "hit_dy": d[:, 1], "hit_dz": d[:, 2], "hit_q_re": rng.uniform(-30.0, 30.0, n)}
    if monitor is not None:
        host["hit_monitor"] = np.asarray(monitor, np.int32)
    cols = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in host.items()}
    return host, cols


def _monitor_stats(engine, cols, first, n, n_monitors, hw, hh, frame=None):
    """One optb_monitor_stats_grouped call over rows [first, first + n), one configuration, monitors 0..n_monitors-1
    all in one frame; returns (stats [n_monitors, OPTB_MS_STRIDE], per-row [y, z, tY, tZ, waist]) on the host."""
    import torch

    from optable_b200 import _abi as A
    from optable_b200.backend import lib

    res = A.Result()
    for k, v in cols.items():
        setattr(res, k, v.data_ptr())
    fr = A.MonitorFrame()
    ty, tz, nrm = frame if frame is not None else ((0.0, 1.0, 0.0), (0.0, 0.0, 1.0), (1.0, 0.0, 0.0))
    fr.tangent_y[:], fr.tangent_z[:], fr.normal[:] = list(ty), list(tz), list(nrm)
    fr.half_width, fr.half_height = float(hw), float(hh)
    frames = torch.frombuffer(bytearray((A.MonitorFrame * n_monitors)(*[fr] * n_monitors)), dtype=torch.uint8).cuda()
    stats = torch.full((n_monitors, A.MS_STRIDE), 7.0, dtype=torch.float64, device="cuda")
    per_row = torch.full((5, max(n, 1)), 7.0, dtype=torch.float64, device="cuda")
    L = lib()
    ws = torch.empty(int(L.optb_monitor_stats_grouped_workspace_bytes(n, n_monitors)), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    ptr = lambda r: C.c_void_p(per_row[r].data_ptr())
    engine._check(L.optb_monitor_stats_grouped(engine._ctx, C.byref(res), int(first), int(n), 0, 1, int(n_monitors),
                                               C.c_void_p(frames.data_ptr()), C.c_void_p(stats.data_ptr()), ptr(0), ptr(1),
                                               ptr(2), ptr(3), ptr(4), C.c_void_p(ws.data_ptr()), int(ws.numel()),
                                               C.c_void_p(st)))
    torch.cuda.synchronize()
    return stats.cpu().numpy(), per_row[:, :n].cpu().numpy()


def _hist(stats):
    from optable_b200 import _abi as A

    return stats[A.MS_HIST:A.MS_HIST + H.BINS].astype(np.int64)


@pytest.mark.parametrize("hw", H.HALF_WIDTHS)
def test_grouped_stats_hist_is_np_histogram_at_the_edges(engine, hw):
    y = H.edge_values(hw)
    _, cols = _rows(y, np.zeros_like(y), monitor=np.zeros(len(y)))
    stats, per_row = _monitor_stats(engine, cols, 0, len(y), 1, hw, 1.0)
    got = _hist(stats[0])
    assert np.array_equal(got, H.numpy_hist(y, hw)), H.explain_hist(y, got, hw)
    np.testing.assert_array_equal(per_row[0], y)   # identity frame: y passes through unchanged (NaN included)


def _numpy_stats(h, sel, frame=None):
    """Reference quantities of the selected rows, float64 numpy."""
    ty, tz, nrm = (np.asarray(v, np.float64) for v in (frame or ((0, 1, 0), (0, 0, 1), (1, 0, 0))))
    P = np.stack([h["hit_px"], h["hit_py"], h["hit_pz"]], 1)[sel]
    D = np.stack([h["hit_dx"], h["hit_dy"], h["hit_dz"]], 1)[sel]
    dist = h["hit_q_re"][sel] + h["hit_t"][sel]
    return {"y": P @ ty, "z": P @ tz, "ty": D @ ty, "tz": D @ tz, "wd": np.where(D @ nrm > 0, -dist, dist),
            "I": h["hit_intensity"][sel], "absP": np.abs(P), "absD": np.abs(D), "frame": (ty, tz)}


def _check_sums(stats, ref):
    from optable_b200 import _abi as A

    for slot, terms in ((A.MS_SUM_I, ref["I"]), (A.MS_SUM_Y, ref["y"]), (A.MS_SUM_Z, ref["z"]), (A.MS_SUM_TY, ref["ty"]),
                        (A.MS_SUM_WD, ref["wd"])):
        want, scale = math.fsum(terms), math.fsum(np.abs(terms))
        assert abs(stats[slot] - want) <= 1e-13 * scale, (slot, stats[slot], want)


def _check_rows(per_row, ref, sel, exact):
    """Per-row outputs of the selected rows equal numpy (exact for an identity frame)."""
    for r, k in enumerate(("y", "z", "ty", "tz", "wd")):
        got = per_row[r]
        if exact or k == "wd":
            np.testing.assert_array_equal(got[sel], ref[k], err_msg=k)
        else:   # a dot product of three terms: within 1e-15 of the sum of the magnitudes of its terms
            t = ref["frame"][0 if k in ("y", "ty") else 1]
            mag = (ref["absP"] if k in ("y", "z") else ref["absD"]) @ np.abs(t)
            assert (np.abs(got[sel] - ref[k]) <= 1e-15 * mag).all(), k


@pytest.mark.parametrize("n,first,select", [
    (0, 10, "all"), (1, 0, "all"), (1000 + 37, 0, "all"), (1000 + 37, 0, "monitor"), (1000 + 37, 0, "key"),
    (5000, 123, "monitor"), (5000, 123, "key"), (1_000_000, 0, "all"), (1_000_000, 17, "monitor")])
def test_grouped_stats_against_numpy(engine, n, first, select):
    """Every group = monitor against numpy of its rows: counts, histogram, extrema exact; sums to 1e-13 of fsum; per-row
    columns exact. Rows have monitors 0..2; "all" has a group for each, "monitor" and "key" (the monitor read from
    hit_key) only for 0 and 1, so monitor 2's rows belong to no group and their per-row columns must be NaN. 1e6 rows
    make a group of many tiles, combined in tile order."""
    import torch

    hw, hh = 2.5, 1.5
    rng = np.random.default_rng(n + first)
    total = first + n
    y = rng.uniform(-1.01 * hw, 1.01 * hw, total)
    grid = H.on_edge_grid(hw)
    y[:min(total, grid.size)] = grid[:total]          # edge values first, so every case holds some
    z = rng.uniform(-1.2 * hh, 1.2 * hh, total)
    mon = rng.integers(0, 3, total)
    h, cols = _rows(y, z, seed=n, monitor=mon)
    M = 3 if select == "all" else 2
    if select == "key":   # root << 32 | monitor << 24 | pop, and no hit_monitor column
        key = (np.arange(total, dtype=np.int64) << 32) | (mon.astype(np.int64) << 24) | 5
        cols["hit_key"] = torch.from_numpy(key).cuda()
        del cols["hit_monitor"]
    stats, per_row = _monitor_stats(engine, cols, first, n, M, hw, hh)
    from optable_b200 import _abi as A

    assert np.isnan(per_row[:, mon[first:] >= M]).all(), "rows of no group must be NaN"
    win = np.zeros(total, bool)
    win[first:] = True
    for g in range(M):
        s = stats[g]
        sel_all = win & (mon == g)
        sel = sel_all[first:]
        ref = _numpy_stats(h, sel_all)
        assert s[A.MS_COUNT] == sel.sum(), g
        got = _hist(s)
        assert np.array_equal(got, H.numpy_hist(ref["y"], hw)), H.explain_hist(ref["y"], got, hw)
        if sel.sum() == 0:
            assert s[A.MS_MIN_Y] == math.inf and s[A.MS_MAX_Y] == -math.inf
            assert s[A.MS_MIN_Z] == math.inf and s[A.MS_MAX_Z] == -math.inf
            assert (s[:A.MS_MIN_Y] == 0).all() and (s[A.MS_SUM_TY:A.MS_HIST + H.BINS] == 0).all()
            continue
        assert s[A.MS_MIN_Y] == ref["y"].min() and s[A.MS_MAX_Y] == ref["y"].max()
        assert s[A.MS_MIN_Z] == ref["z"].min() and s[A.MS_MAX_Z] == ref["z"].max()
        _check_sums(s, ref)
        _check_rows(per_row, ref, sel, exact=True)


def test_grouped_stats_rotated_frame(engine):
    """A rotated frame: per-row columns within 1e-15 of numpy, sums within 1e-13; the histogram is numpy's of the y
    the kernel writes."""
    import torch

    from optable_b200 import _abi as A

    n, hw, hh = 50_000, 3.0, 2.0
    rng = np.random.default_rng(5)
    a, b = 0.3, -0.2
    Rz = np.array([[math.cos(a), -math.sin(a), 0], [math.sin(a), math.cos(a), 0], [0, 0, 1]])
    Ry = np.array([[math.cos(b), 0, math.sin(b)], [0, 1, 0], [-math.sin(b), 0, math.cos(b)]])
    T = Rz @ Ry
    frame = (T[:, 1], T[:, 2], T[:, 0])
    h, cols = _rows(rng.uniform(-3.2, 3.2, n), rng.uniform(-2.2, 2.2, n), seed=6, monitor=np.zeros(n))
    h["hit_px"] = rng.uniform(-0.5, 0.5, n)
    cols["hit_px"].copy_(torch.from_numpy(h["hit_px"]))
    stats, per_row = _monitor_stats(engine, cols, 0, n, 1, hw, hh, frame=frame)
    stats = stats[0]
    sel = np.ones(n, bool)
    ref = _numpy_stats(h, sel, frame=frame)
    assert stats[A.MS_COUNT] == n
    _check_sums(stats, ref)
    _check_rows(per_row, ref, sel, exact=False)
    y = per_row[0]
    assert np.array_equal(_hist(stats), H.numpy_hist(y, hw))   # the kernel bins the y it writes


@pytest.mark.parametrize("ratio", [1.0, 1e3, 1e5])
def test_monitor_stats_std_of_an_off_axis_spot(engine, ratio):
    """std_y / std_z of DeviceMonitor.stats() within 1e-9 of np.std for a small spot far off the monitor's axis."""
    from types import SimpleNamespace

    from optable_b200.analytics import DeviceMonitor

    n = 100_000
    rng = np.random.default_rng(int(ratio))
    y = 2.0 + (2.0 / ratio) * rng.standard_normal(n)
    z = -0.7 + (0.7 / ratio) * rng.standard_normal(n)
    _, cols = _rows(y, z, seed=3, monitor=np.zeros(n))
    mon = SimpleNamespace(tangent_Y=[0.0, 1.0, 0.0], tangent_Z=[0.0, 0.0, 1.0], normal=[1.0, 0.0, 0.0], width=5.0, height=5.0)
    s = DeviceMonitor(mon, cols, 0, engine=engine).stats()
    assert s["count"] == n
    assert s["std_y"] == pytest.approx(np.std(y), rel=1e-9)
    assert s["std_z"] == pytest.approx(np.std(z), rel=1e-9)
    assert s["mean_y"] == pytest.approx(np.mean(y), rel=1e-14)


# ---- histograms a trace accumulates (emit_segment) -----------------------------------------------------------------
MON_HW = (2.5, 3.0, 0.5, 5.0)
MON_HH = (1.0, 5.0, 3.0, 2.5)


def _edge_table(copies=1, rotate=None, shift=0.0, roll=0):
    """Axis-aligned monitors (half-widths MON_HW, half-heights MON_HH, `copies` times along x) and an absorbing block
    behind them. `roll` rotates the size lists (sweep configurations), `rotate` turns monitor 0 about z."""
    import optable_b200 as ob

    hws, hhs = np.roll(MON_HW, roll), np.roll(MON_HH, roll)
    mons = []
    for c in range(copies):
        for i, (hw, hh) in enumerate(zip(hws, hhs)):
            mons.append(ob.Monitor([1.0 + shift + 4 * c + i, 0, 0], width=2 * hw, height=2 * hh))
    if rotate is not None:
        mons[0] = mons[0].RotZ(rotate)
    table = ob.OpticalTable()
    table.add_components([ob.Block([4.0 * copies + 5.0, 0, 0], width=40, height=40)])
    table.add_monitors(mons)
    return table


def _edge_bundle(step=1):
    """Rays along +x from (0, y, z), (y, z) on the grid of the monitors' edge values (every `step`-th y)."""
    from optable_b200.bundle import RayBundle

    ys = np.unique(np.concatenate([H.on_edge_grid(hw) for hw in MON_HW]))[::step]
    zs = np.unique(np.concatenate([np.nextafter(H.edges(hh), t) for hh in MON_HH for t in (-np.inf, 0.0, np.inf)]))
    zs = zs[np.abs(zs) <= max(MON_HH)]   # the edges of every height and +-1 ulp
    Y, Z = np.meshgrid(ys, zs, indexing="ij")
    b = RayBundle.collimated_disc(Y.size, x0=0.0, w0=0)
    b.columns["oy"], b.columns["oz"] = Y.ravel().copy(), Z.ravel().copy()
    return b


def _check_trace_hists(table, rows, hist_y, hist_yz, y0, label, rotated=()):
    """hist_y[m] = np.histogram of monitor m's rows, hist_yz[m] = np.histogram2d; axis-aligned monitors see the ray's y."""
    mon = rows["hit_monitor"].cpu().numpy()
    py, pz = rows["hit_py"].cpu().numpy(), rows["hit_pz"].cpu().numpy()
    root = rows["hit_root"].cpu().numpy().view(np.uint32)
    hy, hyz = hist_y.cpu().numpy(), hist_yz.cpu().numpy()
    assert mon.size > 0
    for m, mo in enumerate(table.monitors):
        hw, hh = float(mo.width) / 2, float(mo.height) / 2
        sel = mon == m
        if m in rotated:
            continue
        y, z = py[sel], pz[sel]
        assert np.array_equal(y, y0[root[sel]]), f"{label}: monitor {m} rows do not carry the ray's y"
        assert sel.sum() > 0 and np.array_equal(hy[m], H.numpy_hist(y, hw)), f"{label} monitor {m}: " + H.explain_hist(y, hy[m], hw)
        want2 = np.histogram2d(y, z, H.BINS, [[-hw, hw], [-hh, hh]])[0].astype(np.int64)
        bad = np.argwhere(hyz[m] != want2)
        assert bad.size == 0, f"{label} monitor {m}: hist_yz differs at (y bin, z bin) {bad[:8].tolist()}"


@pytest.mark.parametrize("copies", [1, 5])
def test_trace_histograms_on_edge_grid(engine, copies):
    """4 monitors (histograms in shared memory) and 20 (K * M * 30 * 31 * 4 B > 64 KiB: global atomics)."""
    from optable_b200 import _abi as A
    from optable_b200.bundle import trace_bundle

    table = _edge_table(copies)
    b = _edge_bundle(step=1 if copies == 1 else 3)
    out = trace_bundle(table, b, record_hist=True, engine=engine)
    assert int(out["counters"][A.C_STATUS]) == 0
    _check_trace_hists(table, out, out["hist_y"], out["hist_yz"], b.columns["oy"], f"{4 * copies} monitors")


@pytest.mark.parametrize("K", [1, 12])
def test_sweep_histograms_on_edge_grid(engine, K):
    """trace_sweep: configuration k's histograms = numpy of its own rows (configurations differ in monitor sizes)."""
    import optable_b200 as ob

    tables = [_edge_table(1, shift=0.1 * k, roll=k) for k in range(K)]
    b = _edge_bundle(step=2)
    sw = ob.trace_sweep(tables, b, record_hist=True, engine=engine)
    for k in range(K):
        r = sw.rows(k)
        _check_trace_hists(tables[k], r, r["hist_y"], r["hist_yz"], b.columns["oy"], f"sweep K={K} config {k}")


def test_trace_histograms_rotated_monitor(engine):
    """A monitor turned about z: y = local point . lab tangent (include/optb.h, the reference's convention). Exact on
    bins no row within 1e-12 of an edge can reach; totals = rows with y (and z) in range."""
    from optable_b200.bundle import RayBundle, trace_bundle

    table = _edge_table(1, rotate=0.3)
    b = RayBundle.collimated_disc(200_000, x0=0.0, radius=4.0, w0=0)
    out = trace_bundle(table, b, record_hist=True, engine=engine)
    mon = out["hit_monitor"].cpu().numpy()
    sel = mon == 0
    P = np.stack([out[k].cpu().numpy()[sel] for k in ("hit_px", "hit_py", "hit_pz")], 1)
    mo = table.monitors[0]
    T = np.asarray(mo.transform_matrix, np.float64)
    y, z = P @ (T @ [0.0, 1.0, 0.0]), P @ (T @ [0.0, 0.0, 1.0])
    hw, hh = float(mo.width) / 2, float(mo.height) / 2
    hy, hyz = out["hist_y"][0].cpu().numpy(), out["hist_yz"][0].cpu().numpy()
    ey, ez = H.edges(hw), H.edges(hh)
    near_y = np.abs(y[:, None] - ey[None, :]).min(1) <= 1e-12
    near_z = np.abs(z[:, None] - ez[None, :]).min(1) <= 1e-12
    in_y, in_z = np.abs(y) <= hw, np.abs(z) <= hh
    assert int(hy.sum()) == int(in_y.sum()) and int(hyz.sum()) == int((in_y & in_z).sum())
    assert sel.sum() > 1000
    # bins that a row within 1e-12 of an edge could fall into on either side are left out of the exact comparison
    def loose(v, e):
        k = np.abs(v[:, None] - e[None, :]).argmin(1)
        return np.isin(np.arange(H.BINS), np.concatenate([k - 1, k]))
    keep_y, keep_z = ~loose(y[near_y], ey), ~loose(z[near_z], ez)
    np.testing.assert_array_equal(hy[keep_y], H.numpy_hist(y, hw)[keep_y])
    want2 = np.histogram2d(y, z, H.BINS, [[-hw, hw], [-hh, hh]])[0].astype(np.int64)
    cells = keep_y[:, None] & keep_z[None, :]
    np.testing.assert_array_equal(hyz[cells], want2[cells])


# ---- device against the C oracle on the golden scenes --------------------------------------------------------------
def _monitor_names():
    return [n for n in golden_io.names() if golden_io.load(n)[0].n_monitors > 0]


@pytest.mark.parametrize("name", _monitor_names())
def test_trace_histograms_match_oracle_golden(engine, name):
    """hist_y and hist_yz of a device trace = the oracle's. A difference is allowed only in bins that a row within
    1e-9 of an edge touches (the two traces may place such a row an ulp apart); such rows are named."""
    from optable_b200 import _abi as A
    from oracle import oracle as O

    flat, rays, params, _ = golden_io.load(name)
    scene = engine.upload(flat)
    dev = engine.trace_arrays(scene, rays, record_segments=False, record_hist=True, **params)
    orc = O.trace(flat, rays, record_segments=False, record_hist=True, **params)
    for m in range(flat.n_monitors):
        mf = flat.mon_f[m]
        hw, hh = mf[A.MON_HW], mf[A.MON_HH]
        if np.array_equal(dev["hist_y"][m], orc["hist_y"][m]) and np.array_equal(dev["hist_yz"][m], orc["hist_yz"][m]):
            continue
        sel = orc["hit_monitor"] == m
        P = np.stack([orc["hit_px"][sel], orc["hit_py"][sel], orc["hit_pz"][sel]], 1)
        y, z = P @ mf[A.MON_TY:A.MON_TY + 3], P @ mf[A.MON_TZ:A.MON_TZ + 3]
        near = (np.abs(y[:, None] - H.edges(hw)).min(1) <= 1e-9) | (np.abs(z[:, None] - H.edges(hh)).min(1) <= 1e-9)
        named = [(int(orc["hit_root"][sel][i]), int(orc["hit_pop"][sel][i]), float(y[i]), float(z[i])) for i in np.flatnonzero(near)]
        diff = int(np.abs(dev["hist_y"][m] - orc["hist_y"][m]).sum())
        assert 0 < len(named) and diff <= 2 * len(named), \
            f"{name} monitor {m}: histograms differ ({diff} counts) with no row near an edge to explain it"
        bins = set(np.flatnonzero(dev["hist_y"][m] != orc["hist_y"][m]).tolist())
        allowed = set()
        for _, _, v, _ in named:
            k = int(np.abs(H.edges(hw) - v).argmin())
            allowed |= {k - 1, k}
        assert bins <= allowed, f"{name} monitor {m}: bins {sorted(bins - allowed)} differ; rows near an edge: {named[:6]}"
        print(f"{name} monitor {m}: histogram difference explained by near-edge rows (root, pop, y, z) {named[:6]}")
