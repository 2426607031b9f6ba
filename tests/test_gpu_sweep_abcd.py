"""GPU: ABCD matrices of every configuration of a sweep (sweep_abcd_matrix, SweepScene.abcd_matrix,
optb_sweep_abcd_pivots / optb_sweep_abcd) against OpticalTable.calculate_abcd_matrix on each configuration."""
import copy
import ctypes as C
import os

import numpy as np
import pytest
import torch

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.analytics import _frame
from optable_b200.sweep import SweepScene, sweep_abcd_matrix
from optable_b200.workloads import asphere_lens9, telescope_4f_grid
from tests import golden_io, scenes
from tests.test_gpu_sweep_rows import _poser

pytestmark = pytest.mark.gpu

F0 = 43.17


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _table(F1=F0, F2=F0, extra=()):
    sc = telescope_4f_grid(ob, F1, F2)
    t = ob.OpticalTable()
    t.add_components(list(sc.components) + list(extra))
    t.add_monitors(list(sc.monitors))
    return t


def _grid(K):
    return [(F0 + 0.3 * (k // 4 - 1.5), F0 + 0.3 * (k % 4 - 1.5)) for k in range(K)]


def _table_method(t, rays):
    m0, m1 = t.monitors[:2]
    return t.calculate_abcd_matrix(m0, m1, rays)


def _same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


@pytest.mark.parametrize("K", [16, 1])
def test_every_configuration_equals_the_table_method(engine, K):
    rays = scenes.abcd_rays(ob)
    tables = [_table(*f) for f in _grid(K)]
    res = sweep_abcd_matrix(tables, 0, 1, rays, engine=engine)
    assert res.M.shape == (K, 7, 2, 2) and res.row_counts.shape == (K, 7, 3)
    assert res.valid.all() and res.defined.all() and (res.row_counts == 1).all()
    assert res.ids == sorted(r._id for r in rays)
    assert res.traces[0].n == 14 and res.traces[1].n == 7
    for k, t in enumerate(tables):
        np.testing.assert_allclose(res.M[k], _table_method(t, rays), rtol=0, atol=1e-9, err_msg=f"configuration {k}")


def test_golden_values_of_the_4f_calibration():
    """Tables built as calibrate_symmetric_4f's simulate builds them, the golden (F1, F2) among them."""
    z = np.load(os.path.join(golden_io.GOLDEN_DIR, "abcd_4f.npz"))
    F1g, F2g = (float(v) for v in z["F"])
    lens = asphere_lens9(ob, [F0, 0, 0])

    def simulate(F1, F2):
        first = lens.copy()._Translate(np.array([F1, 0, 0]) - lens.origin)
        second = lens.copy()._Translate(np.array([F1 + 2 * F2, 0, 0]) - lens.origin).RotZ(np.pi)
        t = ob.OpticalTable()
        t.add_components([first, second])
        t.add_monitors([ob.Monitor(origin=[0, 0, 0], width=5, height=5),
                        ob.Monitor(origin=[2 * F1 + 2 * F2, 0, 0], width=5, height=5)])
        return t

    F = [(F1g - 0.2, F2g), (F1g, F2g), (F1g, F2g + 0.3), (F1g + 0.1, F2g - 0.1)]
    tables = [simulate(*f) for f in F]
    res = sweep_abcd_matrix(tables, 0, 1, scenes.abcd_rays(ob))
    assert res.valid.all()
    np.testing.assert_allclose(res.M[1], z["Ms"], rtol=1e-5, atol=2e-4)


def _rows(res_trace, m):
    h = res_trace.hits
    root = h["hit_root"].cpu().numpy().view(np.uint32).astype(np.int64)
    mon = h["hit_monitor"].cpu().numpy()
    v = res_trace.row_values()
    return root, mon == m, v["y"].cpu().numpy(), v["tY"].cpu().numpy()


def _numpy_fd(res, m1, disp=1e-5, rot=1e-5):
    """M from the two traces' own row_values(): numpy's finite differences of the same y and tY."""
    ra, rb = res.traces
    K, N = res.M.shape[:2]
    root_a, sel_a, ya, ta = _rows(ra, m1)
    root_b, sel_b, yb, tb = _rows(rb, m1)
    M = np.full((K, N, 2, 2), np.nan)
    counts = np.zeros((K, N, 3), np.int64)
    for k in range(K):
        for r in range(N):
            j = [np.nonzero(sel_a & (root_a == k * 2 * N + r))[0], np.nonzero(sel_a & (root_a == k * 2 * N + N + r))[0],
                 np.nonzero(sel_b & (root_b == k * N + r))[0]]
            counts[k, r] = [len(x) for x in j]
            if all(len(x) == 1 for x in j):
                y0, y1, y2 = ya[j[0][0]], ya[j[1][0]], yb[j[2][0]]
                t0, t1, t2 = ta[j[0][0]], ta[j[1][0]], tb[j[2][0]]
                M[k, r] = [[(y1 - y0) / disp, (y2 - y0) / rot], [(t1 - t0) / disp, (t2 - t0) / rot]]
    return M, counts


def _undefined_tables():
    """Configuration 0: the relay; 1: mon1 moved sideways; 2: mon1 narrowed (both lose the outer rays); 3: a small
    tilted mirror behind mon1 sends the centre ray back through mon1 once more (and past the lenses, away from mon0).
    Every configuration holds the mirror (one topology): out of the beam where it is not wanted."""
    tables = []
    for k in range(4):
        mirror = ob.Mirror([4 * F0 + 2, 0 if k == 3 else 100, 0], radius=0.3).RotZ(np.radians(10))
        t = _table(extra=[mirror])
        if k == 1:
            t.monitors[1]._Translate([0, 1.5, 0])
        if k == 2:
            t.monitors[1].width = 2.0
        tables.append(t)
    return tables


def test_undefined_rays_are_nan_and_bit_exact_elsewhere(engine):
    rays = scenes.abcd_rays(ob)
    tables = _undefined_tables()
    res = sweep_abcd_matrix(tables, 0, 1, rays, engine=engine)
    M, counts = _numpy_fd(res, 1)
    assert np.array_equal(res.row_counts, counts)
    assert _same(res.M, M)                                  # bit for bit, NaN where undefined
    assert np.array_equal(np.isnan(res.M).any((2, 3)), ~res.defined)
    assert res.defined[0].all()
    assert (~res.defined[1]).sum() == 2 and (res.row_counts[1][~res.defined[1]] == 0).all()
    assert (~res.defined[2]).sum() == 4 and (res.row_counts[2][~res.defined[2]] == 0).all()
    assert (~res.defined[3]).sum() == 1 and (res.row_counts[3][~res.defined[3]] == 2).all()
    for k, t in enumerate(tables):
        try:
            want = _table_method(t, rays)
        except (AssertionError, ValueError):
            assert not res.valid[k], f"configuration {k}"
            continue
        assert res.valid[k], f"configuration {k}"
        np.testing.assert_allclose(res.M[k], want, rtol=0, atol=1e-9)
    assert list(res.valid) == [True, False, False, False]


def test_matrices_are_numpy_finite_differences_of_the_row_values(engine):
    tables = [_table(*f) for f in _grid(8)]
    res = sweep_abcd_matrix(tables, 0, 1, scenes.abcd_rays(ob), disp=3e-5, rot=2e-5, engine=engine)
    M, counts = _numpy_fd(res, 1, 3e-5, 2e-5)
    assert np.array_equal(res.row_counts, counts) and _same(res.M, M)


def test_sweep_scene_equals_sweep_over_copies(engine):
    t = _table()
    lens, mon1 = t.components[1], t.monitors[1]
    restore = _poser([lens, mon1])
    F = _grid(12)
    calls = []

    def configure(k):
        calls.append(k)
        restore()
        lens.TX(F[k][0] + F[k][1] - 2 * F0)
        mon1.TX(F[k][0] + 2 * F[k][1] - 3 * F0)

    copies = []
    for k in range(len(F)):
        configure(k)
        copies.append(copy.deepcopy(t))
    rays = scenes.abcd_rays(ob)
    want = sweep_abcd_matrix(copies, 0, 1, rays, engine=engine)
    calls.clear()
    got = SweepScene(t, [lens, mon1]).abcd_matrix(t.monitors[0], mon1, rays, configure, len(F), engine=engine)
    assert calls == list(range(len(F)))
    assert _same(got.M, want.M) and np.array_equal(got.defined, want.defined)
    assert np.array_equal(got.row_counts, want.row_counts) and got.valid.all()
    for k in (0, 5, 11):
        np.testing.assert_allclose(got.M[k], _table_method(copies[k], rays), rtol=0, atol=1e-9)


def test_precondition_errors():
    rays = scenes.abcd_rays(ob)
    plate = lambda a: ob.GlassSlab([-5, 0, 0], width=6, height=6, thickness=1.0, n1=1, n2=1.5, reflectivity=0).RotZ(a)
    tables = [_table(extra=[plate(0.0)]), _table(extra=[plate(0.0)]), _table(extra=[plate(0.02)])]
    with pytest.raises(ValueError, match=r"in configuration 2, ray id 0 .*bundle per configuration"):
        sweep_abcd_matrix(tables, 0, 1, rays)
    missing = rays + [ob.Ray([-10, 4.0, 0], [1, 0, 0], wavelength=780e-7, w0=61e-4, id=99)]
    with pytest.raises(ValueError, match=r"Rays at mon0 do not match the input rays\..*ray id 99"):
        sweep_abcd_matrix([_table(), _table(44.0, 42.0)], 0, 1, missing)


def test_entry_points_ignore_row_order_and_repeat_bit_for_bit(engine):
    tables = _undefined_tables()
    res = sweep_abcd_matrix(tables, 0, 1, scenes.abcd_rays(ob), engine=engine)
    K, N = res.M.shape[:2]
    ha, hb = res.traces[0].hits, res.traces[1].hits
    frames = (A.MonitorFrame * K)(*[_frame(t.monitors[1]) for t in tables])
    g = torch.Generator(device="cpu").manual_seed(7)

    def permuted(h, how):
        n = h["hit_px"].numel()
        p = torch.randperm(n, generator=g) if how == "random" else torch.arange(n - 1, -1, -1)
        p = p.to(h["hit_px"].device)
        return {k: v[p].contiguous() for k, v in h.items()}

    def run(a, b):
        piv, bad = engine.sweep_abcd_pivots(a, N, K, 0)
        abcd, cnt = engine.sweep_abcd(a, b, N, K, 1, frames, 1e-5, 1e-5)
        return piv.cpu().numpy(), bad.cpu().numpy(), abcd.cpu().numpy(), cnt.cpu().numpy()

    ref = run(ha, hb)
    assert int(ref[1][0]) == -1 and _same(ref[2].reshape(K, N, 2, 2), res.M) and np.array_equal(ref[3], res.row_counts)
    for how in ("random", "reversed", "again"):
        a, b = (ha, hb) if how == "again" else (permuted(ha, how), permuted(hb, how))
        got = run(a, b)
        for x, y in zip(got, ref):
            assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), how


def test_documented_error_codes(engine):
    from optable_b200.backend import lib

    L = lib()
    tables = [_table(), _table(44.0, 42.0)]
    res = sweep_abcd_matrix(tables, 0, 1, scenes.abcd_rays(ob), engine=engine)
    K, N = 2, 7
    h = {k: v for k, v in res.traces[0].hits.items()}
    dev = h["hit_px"].device
    ws_n = int(L.optb_sweep_abcd_workspace_bytes(N, K))
    assert ws_n > 0
    ws = torch.empty(ws_n, dtype=torch.uint8, device=dev)
    piv = torch.empty((N, 3), dtype=torch.float64, device=dev)
    bad = torch.empty(1, dtype=torch.int64, device=dev)
    abcd = torch.empty((K, N, 4), dtype=torch.float64, device=dev)
    cnt = torch.empty((K, N, 3), dtype=torch.int32, device=dev)
    frames = torch.frombuffer(bytearray((A.MonitorFrame * K)(*[_frame(t.monitors[1]) for t in tables])),
                              dtype=torch.uint8).to(dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())

    def result(drop=()):
        r = A.Result()
        for k, v in h.items():
            if k not in drop:
                setattr(r, k, v.data_ptr())
        return r

    def pivots(r, n_rays=N, n_configs=K, mon=0, wsb=ws_n):
        rc = L.optb_sweep_abcd_pivots(engine._ctx, C.byref(r), h["hit_px"].numel(), n_rays, n_configs, mon, p(piv),
                                      p(bad), p(ws), wsb, st)
        return rc, L.optb_last_error(engine._ctx).decode()

    def matrix(ra, rb, n_rays=N, n_configs=K, mon=1, wsb=ws_n):
        rc = L.optb_sweep_abcd(engine._ctx, C.byref(ra), h["hit_px"].numel(), C.byref(rb), h["hit_px"].numel(), n_rays,
                               n_configs, mon, p(frames), 1e-5, 1e-5, p(abcd), p(cnt), p(ws), wsb, st)
        return rc, L.optb_last_error(engine._ctx).decode()

    assert pivots(result())[0] == 0 and matrix(result(), result())[0] == 0
    cases = [
        (dict(r=result(("hit_root", "hit_key"))), "hit_root or hit_key"),
        (dict(r=result(("hit_monitor", "hit_key"))), "hit_monitor or hit_key"),
        (dict(r=result(("hit_py",))), "hit_px/py/pz"),
        (dict(r=result(), mon=256), "monitor index"),
        (dict(r=result(), mon=-1), "monitor index"),
        (dict(r=result(), n_rays=1 << 31, n_configs=1), "below 2^32"),
        (dict(r=result(), wsb=ws_n - 1), "workspace too small"),
    ]
    for kw, msg in cases:
        rc, err = pivots(**kw)
        assert rc == -7 and msg in err and err.startswith("optb_sweep_abcd_pivots"), (kw, rc, err)
        r = kw.pop("r")
        rc, err = matrix(r, result(), **kw)
        assert rc == -7 and msg in err and err.startswith("optb_sweep_abcd"), (kw, rc, err)
    rc, err = matrix(result(), result(("hit_dz",)))
    assert rc == -7 and "hit_dx/dy/dz" in err
    assert pivots(result(("hit_dx",)))[0] == 0          # the pivots read no directions
    assert L.optb_sweep_abcd_workspace_bytes(0, 1) == -1 and L.optb_sweep_abcd_workspace_bytes(1, 0) == -1
    assert L.optb_sweep_abcd_workspace_bytes(1 << 31, 1) == -1
