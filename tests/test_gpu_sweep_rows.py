"""GPU: sweeps built from one base scene plus the rows that differ (`SweepScene`, `optb_scene_upload_sweep_rows`).
Every check is bit for bit: the sorted monitor rows in every column, the histograms, every OPTB_C_* counter (the
cull bits of the box hierarchy only show in OPTB_C_TESTS / OPTB_C_BOX_TESTS) and `stats()`. The references are
`trace_sweep` over deep copies of the table taken right after each `configure(k)`, and, for scenes whose flattening
builds box hierarchies, the one-scene path of a GUI loop (`FlatScene.refresh` + `optb_scene_update_nodes` + trace)."""
import copy
import ctypes as C

import numpy as np
import pytest

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.bundle import RayBundle, trace_bundle
from optable_b200.flatten import FlatScene, pack_rays
from optable_b200.sweep import SweepScene, trace_sweep
from optable_b200.workloads import ripa, telescope_4f_grid
from tests import scenes

pytestmark = pytest.mark.gpu

HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64
# every counter of a sweep, except the two that count the calls' launches and generations
SUMMED = [c for c in range(A.C_COUNT) if c not in (A.C_GENERATIONS, A.C_LAUNCHES)]


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _poser(objs):
    """A restore() that puts every object of the subtrees of `objs` back to its pose and cached box of now, so that
    `restore(); move(k)` is configuration k whatever ran before it (the pose methods are relative)."""
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


def _same_rows(got, want, what):
    assert len(got["hit_root"]) == len(want["hit_root"]), f"{what}: rows"
    for c in HIT_COLS:
        g, w = got[c], want[c]
        g = g.cpu().numpy() if hasattr(g, "cpu") else np.asarray(g)
        w = w.cpu().numpy() if hasattr(w, "cpu") else np.asarray(w)
        assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), f"{what}: {c}"


def _same_stats(a, b):
    for key in a:
        assert np.array_equal(np.asarray(a[key]), np.asarray(b[key]), equal_nan=True), key


def _against_copies(engine, table, vary, configure, K, bundle, limit=None):
    """SweepScene.trace == trace_sweep over deep copies taken after each configure(k), bit for bit. Returns both."""
    copies = []
    for k in range(K):
        configure(k)
        copies.append(copy.deepcopy(table))
    want = trace_sweep(copies, bundle, limit, record_hist=True, engine=engine)
    got = SweepScene(table, vary).trace(bundle, configure, K, limit, record_hist=True, engine=engine)
    assert got.n_configs == want.n_configs == K
    _same_rows(got.hits, want.hits, "all configurations")
    for k in range(K):
        _same_rows(got.rows(k), want.rows(k), f"configuration {k}")
    assert np.array_equal(got.hist_y.cpu().numpy(), want.hist_y.cpu().numpy())
    assert np.array_equal(got.hist_yz.cpu().numpy(), want.hist_yz.cpu().numpy())
    assert np.array_equal(np.asarray(got.counters), np.asarray(want.counters))
    _same_stats(got.stats(), want.stats())
    return got, want


def test_4f_grid_lens_and_monitor(engine):
    t = telescope_4f_grid(ob, 43.17, 43.17)
    lens, mon = t.components[1], t.monitors[1]
    restore = _poser([lens, mon])
    F = [(43.17 + 0.2 * (k // 4 - 1.5), 43.17 + 0.2 * (k % 4 - 1.5)) for k in range(16)]

    def configure(k):
        restore()
        lens.TX(F[k][0] + F[k][1] - 2 * 43.17)
        mon.TX(F[k][0] + 2 * F[k][1] - 3 * 43.17)

    got, want = _against_copies(engine, t, [lens, mon], configure, 16, RayBundle.collimated_disc(37, radius=2.5))
    # the monitor frames are configuration k's, not the live object's
    for k in (0, 7, 15):
        assert got.monitors[k][1].origin[0] == want.tables[k].monitors[1].origin[0]
        assert got.monitor(k, 1).stats()["count"] == got.stats()["count"][k, 1] > 0


@pytest.mark.parametrize("mirror_transmission", [0.1, 0.0])
def test_splitting_slab(engine, mirror_transmission):
    """Reflectivity 0 in configuration 0 (and, with opaque end mirrors, in the base table): whether the scene splits
    rays is decided by the varied rows of the other configurations."""
    slab = ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=1, n2=1.5, reflectivity=0)
    t = scenes.Scene([ob.Mirror([-2, 0, 0], radius=3, reflectivity=0.9, transmission=mirror_transmission), slab,
                      ob.Mirror([2, 0, 0], radius=3, reflectivity=0.9, transmission=mirror_transmission).RotZ(np.pi)],
                     [], [ob.Monitor([1, 0, 0], 6, 6), ob.Monitor([-3, 0, 0], 6, 6)])
    restore = _poser([slab])

    def configure(k):
        restore()
        for face in slab.components:
            face.reflectivity = 0.05 * k
        slab.RotZ(0.02 * (k - 2))

    bundle = RayBundle.collimated_disc(50, x0=-1.5, radius=0.6, direction=(1.0, 0.01, 0.0))
    got, _ = _against_copies(engine, t, [slab], configure, 5, bundle, {"max_trace_num": 40})
    assert int(got.counters[A.C_SEGMENTS]) > 0


def _f3_reference(engine, table, comps, configure, K, arrs, limit):
    """Configuration by configuration on ONE uploaded scene: refresh the moved components, send their rows
    (optb_scene_update_nodes), trace. Returns per-configuration (rows, hist_y, hist_yz, counters)."""
    flat = FlatScene(table.components, table.monitors)
    scene = engine.upload(flat)
    out = []
    for k in range(K):
        configure(k)
        changed = sorted({i for c in comps for i in flat.refresh(c)})
        scene.update_nodes(changed)
        out.append(engine.trace_arrays(scene, arrs, max_trace_num=limit, record_segments=False, record_hist=True))
    scene.close()
    return out


def _against_f3(engine, table, comps, configure, K, rays, limit):
    arrs, _, _ = pack_rays(rays)
    arrs["family"] = np.arange(len(rays), dtype=np.int32)   # every root its own family, as in a sweep
    got = SweepScene(table, comps).trace(rays, configure, K, {"max_trace_num": limit}, record_hist=True, engine=engine)
    want = _f3_reference(engine, table, comps, configure, K, arrs, limit)
    M = len(table.monitors)
    sums = np.zeros(A.C_COUNT, np.int64)
    for k, w in enumerate(want):
        _same_rows(got.rows(k), w, f"configuration {k}")
        assert np.array_equal(got.hist_y[k].cpu().numpy(), w["hist_y"][:M]), f"configuration {k}: hist_y"
        assert np.array_equal(got.hist_yz[k].cpu().numpy(), w["hist_yz"][:M]), f"configuration {k}: hist_yz"
        sums += np.asarray(w["counters"], np.int64)
    for c in SUMMED:
        assert int(got.counters[c]) == int(sums[c]), f"counter {c}"
    return got, want


def test_ripa_leaf_and_nested_group(engine):
    """ripa (7,689 leaves, lattice groups, box hierarchies): a mirror of the first group and the TriangularPrism next to
    the 6,401-cell lattice move. Equal to the one-scene path configuration by configuration, counters included."""
    sc = ripa(ob, n_rays=48)
    mirror, prism = sc.components[0].components[1], sc.components[1].components[1]
    restore = _poser([mirror, prism])

    def configure(k):
        restore()
        mirror.TX(2e-4 * k)
        prism.TY(1e-3 * (k - 3))
        prism.RotZ(1e-4 * k)

    got, _ = _against_f3(engine, sc, [mirror, prism], configure, 8, sc.rays, sc.limit["max_trace_num"])
    assert int(got.counters[A.C_HITS]) > 0


def test_stale_ancestor_box(engine):
    """A leaf that keeps a fresh box of its own moves sideways out of its group's cached box in the odd configurations:
    there, and only there, the group's box may no longer dismiss the group by distance. Equal to the one-scene path,
    whose optb_scene_update_nodes recomputes every cull bit of the table, configuration by configuration, counters
    included."""
    first = ob.CircleRefractive([10, 0, 0], radius=2.0, n1=1.0, n2=1.5)
    second = ob.CircleRefractive([12, 0, 0], radius=2.0, n1=1.5, n2=1.0)
    g = ob.ComponentGroup([0, 0, 0])
    g.add_components([first, second])
    _ = g.bbox
    sc = scenes.Scene([ob.BeamSplitter([5, 0, 0], width=4, height=4, eta=0.5), g], [], [ob.Monitor([20, 0, 0], 6, 6)])
    rays = [ob.Ray([0, y, z], [1, 0, 0], wavelength=633e-7, w0=50e-4) for y, z in np.linspace(-1, 1, 24).reshape(12, 2)]
    restore = _poser([second])

    def configure(k):
        restore()
        second.TY(3.0 * (k % 2))        # odd configurations: y from 1 to 5, beyond the group's cached box (|y| <= 2)
        second._bbox = tuple(second.get_bbox())

    got, _ = _against_f3(engine, sc, [second], configure, 4, rays, 50)
    assert int(got.counters[A.C_BOX_TESTS]) > 0


def test_one_configuration_equals_trace_bundle(engine):
    t = telescope_4f_grid(ob, 43.17, 43.17)
    bundle = RayBundle.collimated_disc(64, radius=2.5)
    got = SweepScene(t, [t.components[1]]).trace(bundle, lambda k: None, 1, record_hist=True, engine=engine)
    sep = trace_bundle(t, bundle, record_hist=True, engine=engine)
    want = {c: sep[c].cpu().numpy() for c in HIT_COLS}
    order = np.lexsort((want["hit_pop"].view(np.uint32), want["hit_monitor"], want["hit_root"].view(np.uint32)))
    _same_rows(got.rows(0), {c: v[order] for c, v in want.items()}, "K = 1")
    assert np.array_equal(got.hist_y[0].cpu().numpy(), sep["hist_y"][:2].cpu().numpy())
    for c in (A.C_SEGMENTS, A.C_INTERACTIONS, A.C_HITS, A.C_TESTS, A.C_DROPPED, A.C_STATUS, A.C_BOX_TESTS):
        assert int(got.counters[c]) == int(sep["counters"][c]), c


# -- documented errors --------------------------------------------------------------------------------------------
def _upload_rows(engine, flat, K, nodes, node_i, node_f, monitors=(), mon_f=None):
    from optable_b200.backend import lib

    nodes = np.ascontiguousarray(nodes, np.int32)
    monitors = np.ascontiguousarray(monitors, np.int32)
    node_i = np.ascontiguousarray(node_i, np.int32)
    node_f = np.ascontiguousarray(node_f, np.float64)
    mon_f = np.ascontiguousarray(np.zeros((K, 0, A.MON_STRIDE)) if mon_f is None else mon_f, np.float64)
    h = C.c_void_p()
    desc = flat.desc()
    rc = lib().optb_scene_upload_sweep_rows(engine._ctx, C.byref(desc), K, nodes.ctypes.data, nodes.size,
                                            node_f.ctypes.data, node_i.ctypes.data, monitors.ctypes.data, monitors.size,
                                            mon_f.ctypes.data, C.byref(h))
    msg = lib().optb_last_error(engine._ctx).decode()
    if rc == 0:
        lib().optb_scene_destroy(engine._ctx, h)
    return rc, msg


def test_documented_errors(engine):
    from optable_b200.backend import BackendError
    from optable_b200.sweep import SweepRows

    t = telescope_4f_grid(ob, 43.17, 43.17)
    flat = FlatScene(t.components, t.monitors)
    V = np.array([3, 4], np.int32)
    ni = np.stack([flat.node_i[V]] * 2)
    nf = np.stack([flat.node_f[V]] * 2)
    assert _upload_rows(engine, flat, 2, V, ni, nf)[0] == 0
    # node_i beyond ORTHO: configuration, row and column named
    bad = ni.copy()
    bad[1, 1, A.NI_MAT1] += 1
    rc, msg = _upload_rows(engine, flat, 2, V, bad, nf)
    assert rc == -5 and f"configuration 1 differs from the base in node_i row 4 column {A.NI_MAT1}" in msg
    ortho = ni.copy()
    ortho[1, 1, A.NI_ORTHO] ^= 1
    assert _upload_rows(engine, flat, 2, V, ortho, nf)[0] == 0
    # out of range and repeated node / monitor indices
    for nodes in ([3, flat.n_nodes], [3, -1], [4, 4]):
        rc, msg = _upload_rows(engine, flat, 2, nodes, ni, nf)
        assert rc == -5 and "out of range or repeated" in msg, nodes
    mon = np.zeros((2, 2, A.MON_STRIDE))
    for monitors in ([0, 2], [1, 1]):
        rc, msg = _upload_rows(engine, flat, 2, V, ni, nf, monitors, mon)
        assert rc == -5 and "varied monitor" in msg, monitors
    # a varied row that fails node validation: a composite aperture whose operation code (node_f) is unknown
    sc = scenes.nested_csg(ob)
    cf = FlatScene(sc.components, sc.monitors)
    i = int(np.nonzero(cf.node_i[:, A.NI_GEOM] == A.G_CSG)[0][0])
    rows_f = np.stack([cf.node_f[[i]]] * 2)
    rows_f[1, 0, A.NF_P] = 5.0
    rc, msg = _upload_rows(engine, cf, 2, [i], np.stack([cf.node_i[[i]]] * 2), rows_f)
    assert rc == -5 and f"configuration 1, node {i}: scene: bad CSG op" in msg
    # K blobs over the scene size limit
    big = 1 << 22   # configurations of a blob of more than 2 KB (6 nodes of 432 B of rows): over the 4 GB limit
    rc, msg = _upload_rows(engine, flat, big, [], np.zeros((big, 0, A.NI_STRIDE), np.int32), np.zeros((big, 0, A.NF_STRIDE)))
    assert rc == -6 and "too large" in msg
    # update_nodes on the scene
    scene = engine.upload_sweep(SweepRows(flat, 2, V, ni, nf, [], np.zeros((2, 0, A.MON_STRIDE))))
    with pytest.raises(BackendError, match=r"-7.*sweep scene"):
        scene.update_nodes([3])
    scene.close()


def test_python_rejections(engine):
    t = telescope_4f_grid(ob, 43.17, 43.17)
    bundle = RayBundle.collimated_disc(8)
    stranger = ob.Mirror([0, 0, 0], radius=1)
    with pytest.raises(ValueError, match=r"vary\[1\] \(Mirror\) is not a component or monitor"):
        SweepScene(t, [t.components[1], stranger]).trace(bundle, lambda k: None, 2, engine=engine)
    # ripa: an MMA holds a lattice (refresh cannot rewrite it), a leaf of the lattice lies in a lattice group
    sc = ripa(ob, n_rays=0)
    mma = next(c for c in sc.components[1].components if type(c).__name__.startswith("MMA"))
    with pytest.raises(ValueError, match=r"cannot be rewritten in place.*trace_sweep\(tables\)"):
        SweepScene(sc, [mma]).trace(bundle, lambda k: None, 2, engine=engine)
    with pytest.raises(ValueError, match=r"lattice group.*trace_sweep\(tables\)"):
        SweepScene(sc, [mma.components[0]]).trace(bundle, lambda k: None, 2, engine=engine)
    # a change refresh cannot express: a new material value
    lens = t.components[1]
    leaf = next(c for c in lens.components if "_n2" in vars(c))

    def new_glass(k):
        vars(leaf)["_n2"] = 1.7 + 0.01 * k

    with pytest.raises(ValueError, match=r"configuration 0 changes vary\[0\].*trace_sweep\(tables\)"):
        SweepScene(t, [lens]).trace(bundle, new_glass, 2, engine=engine)
