"""CPU: sweeps built from one base scene plus the rows that differ (`SweepScene`). The configurations it hands to the
device equal fresh flattens of the table as `configure(k)` left it, and traced by the C oracle they give the rows of
`trace_sweep` over copies of the table taken after each `configure(k)`. Changes that cannot be made in place are
refused with ValueError."""
import copy

import numpy as np
import pytest
import torch

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.bundle import RayBundle
from optable_b200.flatten import FlatScene
from optable_b200.sweep import SweepRows, SweepScene, trace_sweep
from optable_b200.workloads import ripa, telescope_4f_grid
from tests import scenes

HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64


def _oracle(flats, rays, limit, record_hits=True, arrs=None):
    """The layout one sorted sweep trace produces, from K oracle traces (roots renumbered k * N + r)."""
    from oracle import oracle as O

    arrs = rays.materialise() if arrs is None else arrs
    n = len(arrs["ox"])
    parts = [O.trace(f, arrs, max_trace_num=limit, record_segments=False, record_hits=record_hits, record_hist=True)
             for f in flats]
    out = {}
    for k in HIT_COLS:
        v = np.concatenate([p[k].astype(np.int64) + c * n if k == "hit_root" else p[k] for c, p in enumerate(parts)])
        out[k] = torch.from_numpy(v.astype(np.uint32).view(np.int32) if k == "hit_root" else
                                  (v.view(np.int32) if v.dtype == np.uint32 else v))
    out["hist_y"] = torch.from_numpy(np.concatenate([p["hist_y"] for p in parts]))
    out["hist_yz"] = torch.from_numpy(np.concatenate([p["hist_yz"] for p in parts]))
    out["counters"] = np.sum([p["counters"] for p in parts], axis=0)
    return out


def _oracle_flats(flats, rays, limit, record_hits=True, record_hist=False, engine=None, unit=None, arrs=None):
    return _oracle(flats, rays, limit, record_hits, arrs)


class _Rows:
    """Tracer stand-in that keeps the SweepRows it was handed and traces its configurations with the oracle."""

    def __call__(self, rows, rays, limit, record_hits=True, record_hist=False, engine=None, unit=None, arrs=None):
        assert isinstance(rows, SweepRows)
        self.rows = rows
        return _oracle([rows.materialise(k) for k in range(rows.n_configs)], rays, limit, record_hits, arrs)


def _poser(objs):
    saved = []

    def walk(o):
        saved.append((o, o.origin.copy(), np.array(o.transform_matrix, dtype=np.float64), o._bbox))
        for c in getattr(o, "components", []):
            walk(c)

    for o in objs:
        walk(o)

    def restore():
        for o, org, T, box in saved:
            o.origin, o.transform_matrix, o._bbox = org.copy(), T.copy(), box

    return restore


def _four_f():
    t = telescope_4f_grid(ob, 43.17, 43.17)
    lens, mon = t.components[1], t.monitors[1]
    restore = _poser([lens, mon])

    def configure(k):
        restore()
        lens.TX(0.3 * k - 0.4)
        mon.TX(0.5 * k - 0.2)

    return t, [lens, mon], configure, RayBundle.collimated_disc(23, radius=2.5), None


def _slab():
    slab = ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=1, n2=1.5, reflectivity=0)
    t = scenes.Scene([ob.Mirror([-2, 0, 0], radius=3, reflectivity=0.9, transmission=0.0), slab,
                      ob.Mirror([2, 0, 0], radius=3, reflectivity=0.9, transmission=0.0).RotZ(np.pi)],
                     [], [ob.Monitor([1, 0, 0], 6, 6), ob.Monitor([-3, 0, 0], 6, 6)])
    restore = _poser([slab])

    def configure(k):
        restore()
        for face in slab.components:
            face.reflectivity = 0.05 * k
        slab.RotZ(0.02 * (k - 1))

    bundle = RayBundle.collimated_disc(9, x0=-1.5, radius=0.6, direction=(1.0, 0.01, 0.0))
    return t, [slab], configure, bundle, {"max_trace_num": 12}


@pytest.mark.parametrize("case", [_four_f, _slab])
def test_configurations_equal_fresh_flattens(case):
    t, vary, configure, bundle, limit = case()
    K = 4
    tracer = _Rows()
    SweepScene(t, vary).trace(bundle, configure, K, limit, tracer=tracer)
    rows = tracer.rows
    assert rows.n_configs == K and rows.nodes.size > 0
    for k in range(K):
        configure(k)
        fresh, got = FlatScene(t.components, t.monitors), rows.materialise(k)
        for name in ("node_i", "node_f", "mon_f", "mat_f", "aux"):
            assert np.array_equal(getattr(got, name), getattr(fresh, name)), (k, name)
        assert got.max_children == fresh.max_children
    # the properties that pick the trace path cover every configuration, not the base table
    assert rows.max_children == max(rows.materialise(k).max_children for k in range(K))


@pytest.mark.parametrize("case", [_four_f, _slab])
def test_rows_equal_trace_sweep_of_configured_copies(case):
    t, vary, configure, bundle, limit = case()
    K = 4
    copies = []
    for k in range(K):
        configure(k)
        copies.append(copy.deepcopy(t))
    want = trace_sweep(copies, bundle, limit, record_hist=True, tracer=_oracle_flats)
    got = SweepScene(t, vary).trace(bundle, configure, K, limit, record_hist=True, tracer=_Rows())
    for k in range(K):
        a, b = got.rows(k), want.rows(k)
        assert len(a["hit_root"]) == len(b["hit_root"]) > 0
        for c in HIT_COLS:
            assert np.array_equal(a[c].numpy().view(np.uint8), b[c].numpy().view(np.uint8)), (k, c)
    assert np.array_equal(got.hist_y.numpy(), want.hist_y.numpy())
    assert np.array_equal(got.counters, want.counters)
    # monitor frames are snapshots of each configuration
    M = len(t.monitors)
    for k in range(K):
        for m in range(M):
            assert np.array_equal(got.monitors[k][m].origin, want.tables[k].monitors[m].origin)
            assert np.array_equal(got.monitors[k][m].tangent_Y, want.tables[k].monitors[m].tangent_Y)


def _trace(t, vary, configure, K=2):
    return SweepScene(t, vary).trace(RayBundle.collimated_disc(4), configure, K, tracer=_Rows())


def test_rejections():
    t = telescope_4f_grid(ob, 43.17, 43.17)
    lens = t.components[1]
    with pytest.raises(ValueError, match=r"vary\[1\] \(Mirror\) is not a component or monitor of the table"):
        _trace(t, [lens, ob.Mirror([0, 0, 0], radius=1)], lambda k: None)
    leaf = next(c for c in lens.components if "_n2" in vars(c))
    # a new material value: refresh cannot keep the material table
    glass = vars(leaf)["_n2"]

    def new_glass(k):
        vars(leaf)["_n2"] = 1.7 + 0.01 * k

    with pytest.raises(ValueError, match=r"configuration 0 changes vary\[0\] \(.*\).*trace_sweep\(tables\)"):
        _trace(t, [lens], new_glass)
    vars(leaf)["_n2"] = glass
    # a node_i column the configurations must share (the ROC kind of a flat refracting face)
    sc = scenes.Scene([ob.CircleRefractive([5, 0, 0], radius=2, n1=1.0, n2=1.5)], [], [ob.Monitor([9, 0, 0], 4, 4)])
    face = sc.components[0]

    def curve(k):
        face.roc = 50.0

    with pytest.raises(ValueError, match=r"changes the ROC kind of vary\[0\] \(CircleRefractive\)"):
        _trace(sc, [face], curve)


def test_lattice_rejections():
    sc = ripa(ob, n_rays=0)
    mma = next(c for c in sc.components[1].components if type(c).__name__ == "MMA")
    with pytest.raises(ValueError, match=r"vary\[0\] \(MMA\) cannot be rewritten in place.*trace_sweep\(tables\)"):
        _trace(sc, [mma], lambda k: None)
    with pytest.raises(ValueError, match=r"vary\[0\] \(.*\) lies in a lattice group.*trace_sweep\(tables\)"):
        _trace(sc, [mma.components[0]], lambda k: None)
