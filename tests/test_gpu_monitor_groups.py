"""GPU: grouped monitor statistics (optb_monitor_stats_grouped, SweepResult.stats, analytics.monitor_stats).

Every (configuration, monitor) group is checked against numpy of its own rows (counts, histograms and extrema exactly,
sums to 1e-13 of math.fsum), bit for bit against a separate DeviceMonitor per group on traced scenes, and for
bit-identical results between calls and streams."""
import ctypes as C
import math
from types import SimpleNamespace

import numpy as np
import pytest

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.bundle import RayBundle, trace_bundle
from optable_b200.sweep import trace_sweep
from optable_b200.workloads import telescope_4f_grid
from tests import hist_cases as H
from tests import scenes
from tests.test_gpu_sweep import _bundle_of, _slab

pytestmark = pytest.mark.gpu

IDENTITY = ((0.0, 1.0, 0.0), (0.0, 0.0, 1.0), (1.0, 0.0, 0.0))


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _rotation(a, b):
    Rz = np.array([[math.cos(a), -math.sin(a), 0], [math.sin(a), math.cos(a), 0], [0, 0, 1]])
    Ry = np.array([[math.cos(b), 0, math.sin(b)], [0, 1, 0], [-math.sin(b), 0, math.cos(b)]])
    T = Rz @ Ry
    return T[:, 1], T[:, 2], T[:, 0]


def _monitor(frame, hw, hh=2.0):
    ty, tz, nrm = frame
    return SimpleNamespace(tangent_Y=list(ty), tangent_Z=list(tz), normal=list(nrm), width=2 * hw, height=2 * hh)


def _frames(monitors):
    from optable_b200.analytics import _frame

    return (A.MonitorFrame * len(monitors))(*[_frame(m) for m in monitors])


def _to_device(host):
    import torch

    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in host.items()}


def _rows(y, z, root, mon, seed, px=None):
    """Row columns whose local hit points are (px, y, z), with hit_root / hit_monitor, on the host."""
    n = len(y)
    rng = np.random.default_rng(seed)
    d = np.stack([np.ones(n), rng.normal(0, 1e-2, n), rng.normal(0, 1e-2, n)], 1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return {"hit_px": np.zeros(n) if px is None else px, "hit_py": np.asarray(y, np.float64), "hit_pz": np.asarray(z, np.float64),
            "hit_intensity": rng.uniform(0.1, 2.0, n), "hit_t": rng.uniform(1.0, 50.0, n),
            "hit_dx": d[:, 0], "hit_dy": d[:, 1], "hit_dz": d[:, 2], "hit_q_re": rng.uniform(-30.0, 30.0, n),
            "hit_root": np.asarray(root, np.uint32).view(np.int32), "hit_monitor": np.asarray(mon, np.int32)}


def _grouped(engine, cols, monitors, K, M, per_config):
    """One grouped call; (stats [G, 48], per-row [5, n]) on the host."""
    import torch

    stats, per_row = engine.monitor_stats_grouped(cols, _frames(monitors), K, M, per_config)
    torch.cuda.synchronize()
    return stats.cpu().numpy(), per_row.cpu().numpy()


def _case(kind, seed=0):
    """(K, M, rays per configuration, host rows, group of every row (-1: none), per-group frames and half-widths).
    Every group's rows hold edge values of its histogram (hist_cases.on_edge_grid of its half-width); the many-groups
    case spreads them over the groups, a few per group. Rows come in random order."""
    rng = np.random.default_rng(seed)
    if kind == "small":
        K, M, N = 3, 4, 50
        sizes = rng.integers(0, 400, K * M)
        sizes[[1, 6]] = 0          # empty groups
        sizes[[2, 9]] = 1          # one-row groups
    elif kind == "one_big":
        K, M, N = 1, 1, 0
        sizes = np.array([1_000_000])
    else:                          # 4096 configurations x 3 monitors, a few rows each
        K, M, N = 4096, 3, 8
        sizes = rng.integers(0, 6, K * M)
    G = K * M
    hws = np.array([H.HALF_WIDTHS[g % len(H.HALF_WIDTHS)] for g in range(G)])
    grids = {hw: H.on_edge_grid(hw) for hw in set(hws.tolist())}
    ys, grp = [], []
    for g in range(G):
        grid = grids[hws[g]]
        s = int(sizes[g])
        if s == 0:
            continue
        if kind == "many":
            y = grid[(g * 3 + np.arange(s)) % grid.size]
        elif s == 1:
            y = grid[:1]
        else:
            y = np.concatenate([grid, rng.uniform(-1.01 * hws[g], 1.01 * hws[g], s)])
        ys.append(y)
        grp.append(np.full(y.size, g))
    y, grp = np.concatenate(ys), np.concatenate(grp)
    # rows of no group: a monitor index past the last, and a root past the last configuration
    n_bad = 7
    y = np.concatenate([y, rng.uniform(-1, 1, n_bad)])
    grp = np.concatenate([grp, np.full(n_bad, -1)])
    perm = rng.permutation(y.size)
    y, grp = y[perm], grp[perm]
    k, m = np.where(grp >= 0, grp // M, 0), np.where(grp >= 0, grp % M, 0)
    bad = np.flatnonzero(grp < 0)
    m[bad[::2]] = M
    k[bad[1::2]] = K if N else 0
    if not N:
        m[bad] = M
    root = k * max(N, 1) + rng.integers(0, max(N, 1), y.size)
    z = rng.uniform(-2.4, 2.4, y.size)
    return K, M, N, y, z, root, m, grp, hws


def _check_groups(h, grp, stats, per_row, frames, hws, exact):
    order = np.argsort(grp, kind="stable")
    G = stats.shape[0]
    bounds = np.searchsorted(grp[order], np.arange(G + 1))
    none = grp < 0
    assert np.isnan(per_row[:, none]).all(), "rows of no group must be NaN"
    assert int(stats[:, A.MS_COUNT].sum()) == int((~none).sum())
    P = np.stack([h["hit_px"], h["hit_py"], h["hit_pz"]], 1)
    D = np.stack([h["hit_dx"], h["hit_dy"], h["hit_dz"]], 1)
    for g in range(G):
        sel = order[bounds[g]:bounds[g + 1]]
        s = stats[g]
        assert s[A.MS_COUNT] == sel.size, g
        if sel.size == 0:
            assert s[A.MS_MIN_Y] == math.inf and s[A.MS_MAX_Y] == -math.inf, g
            assert s[A.MS_MIN_Z] == math.inf and s[A.MS_MAX_Z] == -math.inf, g
            assert (s[:A.MS_MIN_Y] == 0).all() and (s[A.MS_SUM_TY:] == 0).all(), g
            continue
        ty, tz, nrm = (np.asarray(v, np.float64) for v in frames[g])
        ref = {"y": P[sel] @ ty, "z": P[sel] @ tz, "ty": D[sel] @ ty, "tz": D[sel] @ tz}
        dist = h["hit_q_re"][sel] + h["hit_t"][sel]
        ref["wd"] = np.where(D[sel] @ nrm > 0, -dist, dist)
        got = {q: per_row[r, sel] for r, q in enumerate(("y", "z", "ty", "tz", "wd"))}
        for q in ("y", "z", "ty", "tz", "wd"):
            if exact or q == "wd":
                np.testing.assert_array_equal(got[q], ref[q], err_msg=f"group {g} {q}")
            else:
                t = ty if q in ("y", "ty") else tz
                mag = (np.abs(P[sel]) if q in ("y", "z") else np.abs(D[sel])) @ np.abs(t)
                assert (np.abs(got[q] - ref[q]) <= 1e-15 * mag).all(), (g, q)
        y = got["y"]   # the device bins the y it writes (= numpy's for an identity frame)
        hist = s[A.MS_HIST:A.MS_HIST + H.BINS].astype(np.int64)
        assert np.array_equal(hist, H.numpy_hist(y, hws[g])), f"group {g}: " + H.explain_hist(y, hist, hws[g])
        assert s[A.MS_MIN_Y] == y.min() and s[A.MS_MAX_Y] == y.max(), g
        assert s[A.MS_MIN_Z] == got["z"].min() and s[A.MS_MAX_Z] == got["z"].max(), g
        for slot, terms in ((A.MS_SUM_I, h["hit_intensity"][sel]), (A.MS_SUM_Y, ref["y"]), (A.MS_SUM_Z, ref["z"]),
                            (A.MS_SUM_TY, ref["ty"]), (A.MS_SUM_WD, ref["wd"])):
            want, scale = math.fsum(terms), math.fsum(np.abs(terms))
            assert abs(s[slot] - want) <= 1e-13 * scale, (g, slot, s[slot], want)


@pytest.mark.parametrize("kind", ["small", "one_big", "many"])
@pytest.mark.parametrize("rotated", [False, True])
def test_groups_against_numpy(engine, kind, rotated):
    """Counts, histograms and extrema exact; sums within 1e-13 of fsum; per-row columns exact (identity frames) or
    within 1e-15 of their terms (a different rotation per group); rows of no group NaN and counted nowhere.
    `one_big`: 1e6 rows in one group (245 tiles); `many`: 4096 x 3 groups of 0-5 rows."""
    K, M, N, y, z, root, m, grp, hws = _case(kind, seed=len(kind) + rotated)
    G = K * M
    rng = np.random.default_rng(11)
    frames = [_rotation(*rng.uniform(-0.4, 0.4, 2)) if rotated else IDENTITY for _ in range(G)]
    h = _rows(y, z, root, m, seed=5, px=rng.uniform(-0.5, 0.5, y.size) if rotated else None)
    stats, per_row = _grouped(engine, _to_device(h), [_monitor(frames[g], hws[g]) for g in range(G)], K, M, N)
    _check_groups(h, grp, stats, per_row, frames, hws, exact=not rotated)


@pytest.mark.parametrize("ratio", [1.0, 1e3, 1e5])
def test_off_axis_spots_are_centred_per_group(engine, ratio):
    """std_y, std_z and std_tY within 1e-9 of np.std for groups whose spots sit at different means, |mean| / std = ratio:
    each group's second pass is taken about its own means."""
    from optable_b200.analytics import stats_arrays

    K, M, per = 2, 2, 50_000
    rng = np.random.default_rng(int(ratio))
    means = [(2.0, -0.7, 0.3), (-1.5, 0.4, -0.2), (0.8, 1.9, 0.1), (-2.2, -1.1, -0.35)]
    ys, zs, dys, ks, ms = [], [], [], [], []
    for g, (my, mz, mty) in enumerate(means):
        ys.append(my + (abs(my) / ratio) * rng.standard_normal(per))
        zs.append(mz + (abs(mz) / ratio) * rng.standard_normal(per))
        dys.append(mty + (abs(mty) / ratio) * rng.standard_normal(per))
        ks.append(np.full(per, g // M))
        ms.append(np.full(per, g % M))
    y, z, dy, k, m = (np.concatenate(v) for v in (ys, zs, dys, ks, ms))
    perm = rng.permutation(y.size)
    y, z, dy, k, m = y[perm], z[perm], dy[perm], k[perm], m[perm]
    h = _rows(y, z, k * 10 + 3, m, seed=2)
    h["hit_dx"], h["hit_dy"], h["hit_dz"] = np.ones_like(dy), dy, np.zeros_like(dy)   # tY = dy exactly
    stats, _ = _grouped(engine, _to_device(h), [_monitor(IDENTITY, 5.0)] * (K * M), K, M, 10)
    s = stats_arrays(stats.reshape(K, M, -1), np.full((K, M), 10.0))
    for g in range(K * M):
        sel = (k * M + m) == g
        kk, mm = divmod(g, M)
        assert s["count"][kk, mm] == per
        assert s["std_y"][kk, mm] == pytest.approx(np.std(y[sel]), rel=1e-9), g
        assert s["std_z"][kk, mm] == pytest.approx(np.std(z[sel]), rel=1e-9), g
        assert s["std_tY"][kk, mm] == pytest.approx(np.std(dy[sel]), rel=1e-9), g
        assert s["mean_y"][kk, mm] == pytest.approx(np.mean(y[sel]), rel=1e-14), g


@pytest.mark.parametrize("kind", ["one_big", "many"])
def test_bit_identical_between_calls_and_streams(engine, kind):
    import torch

    from optable_b200.analytics import DeviceMonitor

    K, M, N, y, z, root, m, grp, hws = _case(kind, seed=3)
    cols = _to_device(_rows(y, z, root, m, seed=4))
    monitors = [_monitor(IDENTITY, hws[g]) for g in range(K * M)]

    def call():
        """The grouped call's stats and row values, and the stats of a DeviceMonitor of the last monitor as one array."""
        stats, rows = _grouped(engine, cols, monitors, K, M, N)
        d = DeviceMonitor(monitors[M - 1], cols, M - 1, engine=engine).stats()
        return stats, rows, np.hstack(list(d.values())).astype(np.float64)

    a, ra, da = call()
    b, rb, db = call()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c, rc, dc = call()
    assert da[0] > 0   # the DeviceMonitor's count
    for other, rows, dm in ((b, rb, db), (c, rc, dc)):
        assert np.array_equal(a.view(np.int64), other.view(np.int64))
        assert np.array_equal(ra.view(np.int64), rows.view(np.int64))
        assert np.array_equal(da.view(np.int64), dm.view(np.int64))


# ---- traced scenes: the grouped call against one DeviceMonitor per (configuration, monitor) ---------------------------
def _compare(s, rv, k, m, dm, mon, lo=0, hi=None):
    """stats()[q][k, m] against DeviceMonitor dm's stats, and the row values of monitor m among rows [lo, hi) (`mon`: the
    hit_monitor column) against dm's columns, all bit for bit: both reduce the same rows in the same tiles and order."""
    d = dm.stats()
    assert set(d) == set(s)
    for q, v in d.items():
        assert np.array_equal(s[q][k, m], v, equal_nan=True), (k, m, q)
    assert np.array_equal(dm.std_histy, d["std_histy"], equal_nan=True), (k, m)
    sel = (mon[lo:hi] == m).nonzero().squeeze(1)
    for key, acc in (("y", dm.get_yList), ("z", dm.get_zList), ("tY", dm.get_tYList), ("tZ", dm.get_tZList),
                     ("waist_distance", dm.get_waist_distance)):
        got = rv[key][lo:hi][sel].cpu().numpy()
        want = acc(sort=None).cpu().numpy()
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (k, m, key)


def _check_sweep_stats(engine, tables, bundle, limit=None):
    res = trace_sweep(tables, bundle, limit, engine=engine)
    s, rv = res.stats(), res.row_values()
    assert res.stats() is s   # cached
    M = len(tables[0].monitors)
    assert s["count"].shape == (len(tables), M) and s["hist_y"].shape == (len(tables), M, A.HIST_BINS)
    assert int(s["count"].sum()) == int(res.hits["hit_px"].numel()) > 0
    mon = res.hits["hit_monitor"]
    for k in range(len(tables)):
        for m in range(M):
            _compare(s, rv, k, m, res.monitor(k, m), mon, res._bounds[k], res._bounds[k + 1])
    return s


def test_sweep_with_a_monitor_rotated_per_configuration(engine):
    """Configuration k's monitor is turned by its own angle: each group is evaluated in its own frame."""
    angles = (0.0, 0.12, -0.25, 0.4, 0.07)
    tables = []
    for a in angles:
        t = ob.OpticalTable()
        t.add_components([ob.Block([9.0, 0, 0], width=40, height=40)])
        t.add_monitors([ob.Monitor([3.0, 0, 0], width=5.0, height=4.0).RotZ(a), ob.Monitor([6.0, 0.3, 0], width=3.0, height=3.0)])
        tables.append(t)
    s = _check_sweep_stats(engine, tables, RayBundle.collimated_disc(3000, x0=0.0, radius=1.8, start=5))
    assert (s["count"] > 0).all()


def test_sweep_4f_grid(engine):
    grid = [(43.17 + a, 43.17 + b) for a in (-1.0, 0.0, 0.7) for b in (-0.5, 0.0, 1.1)]
    _check_sweep_stats(engine, [telescope_4f_grid(ob, f1, f2) for f1, f2 in grid], RayBundle.collimated_disc(2000, start=7))


def test_sweep_splitting_slab(engine):
    """Several rows per root and monitor; the pop cap is reached."""
    tables = [_slab(n2, refl, tilt) for n2, refl, tilt in ((1.5, 0.2, 0.0), (1.45, 0.3, 0.05), (1.6, 0.1, -0.08))]
    bundle = RayBundle.collimated_disc(45, x0=-3, radius=0.6, direction=(1.0, 0.01, 0.0))
    _check_sweep_stats(engine, tables, bundle, {"max_trace_num": 300})


def test_sweep_pass_through_monitor(engine):
    base = scenes.monitor_as_component(ob)
    tables = []
    for ang in (2.8, 2.75, 2.9):
        lens = ob.Lens([4, 0, 0], focal_length=9.0, radius=2.0)
        screen = ob.Monitor([8, 0.5, 0], 1.2, 1.2).RotZ(0.15)
        mirror = ob.Mirror([12, 0, 0], radius=3.0).RotZ(ang)
        far = ob.Monitor([6, -6, 0], 6, 6).RotZ(-1.2)
        tables.append(scenes.Scene([lens, screen, mirror], [], [screen, far]))
    _check_sweep_stats(engine, tables, _bundle_of(base.rays), base.limit)


@pytest.mark.parametrize("which", ["4f", "pass_through", "edge_monitors"])
def test_bundle_monitor_stats_equal_device_monitors(engine, which):
    """K = 1 on an unsorted trace_bundle result: analytics.monitor_stats = one DeviceMonitor per monitor."""
    from optable_b200.analytics import DeviceMonitor, grouped_stats, monitor_stats

    if which == "4f":
        table, bundle, limit = telescope_4f_grid(ob, 43.17, 43.17), RayBundle.collimated_disc(5000, start=2), None
    elif which == "pass_through":
        base = scenes.monitor_as_component(ob)
        table, bundle, limit = base, _bundle_of(base.rays), base.limit
    else:
        table = ob.OpticalTable()
        table.add_components([ob.Block([12.0, 0, 0], width=40, height=40)])
        table.add_monitors([ob.Monitor([1.0 + i, 0, 0], width=2 * hw, height=4.0) for i, hw in enumerate((2.5, 3.0, 0.5, 5.0))])
        bundle, limit = RayBundle.collimated_disc(20_000, x0=0.0, radius=4.0, start=3), None
    out = trace_bundle(table, bundle, limit, engine=engine)
    s = monitor_stats(table.monitors, out, engine=engine)
    M = len(table.monitors)
    assert s["count"].shape == (M,) and int(s["count"].sum()) == int(out["hit_px"].numel())
    _, rv = grouped_stats(out, [list(table.monitors)], 0, engine)
    rv = dict(zip(("y", "z", "tY", "tZ", "waist_distance"), rv))
    s2 = {q: v[None] for q, v in s.items()}
    for m in range(M):
        _compare(s2, rv, 0, m, DeviceMonitor(table.monitors[m], out, m, engine=engine), out["hit_monitor"])


# ---- errors ---------------------------------------------------------------------------------------------------------
def _raw_call(engine, cols, K, M, per_config, rows=True, ws_bytes=None):
    """optb_monitor_stats_grouped straight through ctypes: (return code, error message)."""
    import torch

    from optable_b200.backend import lib

    res = A.Result()
    for k, v in cols.items():
        setattr(res, k, v.data_ptr())
    n = int(cols["hit_px"].numel())
    frames = torch.zeros((max(K * M, 1), 11), dtype=torch.float64, device="cuda")
    stats = torch.zeros((max(min(K * M, 1 << 20), 1), A.MS_STRIDE), dtype=torch.float64, device="cuda")
    per_row = torch.zeros((5, max(n, 1)), dtype=torch.float64, device="cuda")
    L = lib()
    need = int(L.optb_monitor_stats_grouped_workspace_bytes(n, max(min(K * M, 1 << 20), 1)))
    ws = torch.empty(max(need if ws_bytes is None else ws_bytes, 1), dtype=torch.uint8, device="cuda")
    p = lambda r: C.c_void_p(per_row[r].data_ptr()) if rows else None
    rc = L.optb_monitor_stats_grouped(engine._ctx, C.byref(res), 0, n, per_config, K, M, C.c_void_p(frames.data_ptr()),
                                      C.c_void_p(stats.data_ptr()), p(0), p(1), p(2), p(3), p(4), C.c_void_p(ws.data_ptr()),
                                      int(ws.numel()) if ws_bytes is None else int(ws_bytes), None)
    torch.cuda.synchronize()
    return rc, L.optb_last_error(engine._ctx).decode()


def test_documented_errors(engine):
    from optable_b200.backend import lib

    h = _rows(np.zeros(10), np.zeros(10), np.arange(10), np.zeros(10), seed=1)
    full = _to_device(h)
    assert _raw_call(engine, full, 2, 1, 5)[0] == 0
    drop = lambda *ks: {k: v for k, v in full.items() if k not in ks}
    cases = [
        (drop("hit_t"), 2, 1, 5, True, None, "hit_px/py/pz, hit_intensity and hit_t are required"),
        (drop("hit_monitor"), 2, 1, 5, True, None, "needs hit_monitor or hit_key"),
        (drop("hit_root"), 2, 1, 5, True, None, "needs hit_root or hit_key"),
        (drop("hit_dx"), 2, 1, 5, True, None, "slopes / waist distances need hit_dx, hit_dy, hit_dz"),
        (drop("hit_q_re"), 2, 1, 5, True, None, "waist distances need hit_q_re"),
        (full, 1, 257, 0, True, None, "at most 256 monitors"),
        (full, 4097, 256, 5, True, None, "n_configs * n_monitors must be at most 2^20"),
        (full, 2, 1, 5, True, 64, "workspace too small"),
    ]
    for cols, K, M, per, rows, ws, msg in cases:
        rc, err = _raw_call(engine, cols, K, M, per, rows, ws)
        assert rc == -7 and msg in err and err.startswith("optb_monitor_stats_grouped"), (msg, rc, err)
    # without a root column the configuration is only needed for rays_per_config > 0; without slopes, rows=None is fine
    assert _raw_call(engine, drop("hit_root"), 1, 1, 0)[0] == 0
    assert _raw_call(engine, drop("hit_dx", "hit_q_re"), 2, 1, 5, rows=False)[0] == 0
    L = lib()
    assert L.optb_monitor_stats_grouped_workspace_bytes(10, 0) == -1
    assert L.optb_monitor_stats_grouped_workspace_bytes(10, (1 << 20) + 1) == -1
    assert L.optb_monitor_stats_grouped_workspace_bytes(-1, 1) == -1


def test_rows_outside_every_group_are_reported(engine):
    from optable_b200.analytics import grouped_stats

    h = _rows(np.zeros(20), np.zeros(20), np.arange(20), np.r_[np.zeros(19), 2], seed=1)
    mons = [[_monitor(IDENTITY, 1.0), _monitor(IDENTITY, 1.0)]]
    with pytest.raises(ValueError, match="1 of 20 monitor rows belong to no"):
        grouped_stats(_to_device(h), mons, 0, engine)
    h["hit_monitor"][-1] = 1
    with pytest.raises(ValueError, match="10 of 20 monitor rows belong to no"):   # roots 10..19: configuration 1 of 1
        grouped_stats(_to_device(h), mons, 10, engine)
    s, _ = grouped_stats(_to_device(h), mons, 20, engine)
    assert s["count"].tolist() == [[19, 1]]


def test_sweep_without_hits_raises(engine):
    tables = [telescope_4f_grid(ob, 43.17, 43.17), telescope_4f_grid(ob, 43.0, 43.5)]
    res = trace_sweep(tables, RayBundle.collimated_disc(50), record_hits=False, engine=engine)
    with pytest.raises(ValueError, match="record_hits=False"):
        res.stats()
    with pytest.raises(ValueError, match="record_hits=False"):
        res.row_values()
