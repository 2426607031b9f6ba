"""GPU: scene sweeps. Every configuration of one `trace_sweep` is bit-identical to a separate `trace_bundle` of the same
table on the same device (sorted monitor rows, every column; histograms; summed counters), on scenes that cover every
sweep kernel kind: aspheres, splitting with the pop cap, lattice walks, pass-through leaves, glass changes."""
import ctypes as C

import numpy as np
import pytest

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.bundle import RayBundle, trace_bundle
from optable_b200.sweep import trace_sweep
from optable_b200.workloads import telescope_4f_grid
from tests import parity, scenes

pytestmark = pytest.mark.gpu

HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _np(rows):
    return {k: rows[k].cpu().numpy() for k in HIT_COLS}


def _key_order(o):
    return np.lexsort((o["hit_pop"].view(np.uint32), o["hit_monitor"], o["hit_root"].view(np.uint32)))


def _bundle_of(rays):
    """The RayBundle of a list of Ray (all alive with q: the bundle's default flags)."""
    from optable_b200.flatten import pack_rays

    arrs, _, _ = pack_rays(rays)
    assert (arrs["flags"] == A.RF_ALIVE | A.RF_HASQ).all()
    return RayBundle({k: arrs[k] for k in A.RAY_F64}, len(rays))


def _check_sweep(engine, tables, bundle, limit=None, rays=None):
    """trace_sweep == K separate trace_bundle calls, bit for bit. Returns the sweep result."""
    res = trace_sweep(tables, bundle if rays is None else rays, limit, record_hist=True, engine=engine)
    sums = np.zeros(A.C_COUNT, np.int64)
    for k, t in enumerate(tables):
        sep = trace_bundle(t, bundle, limit, record_hist=True, engine=engine)
        want = _np(sep)
        want = {c: v[_key_order(want)] for c, v in want.items()}
        got = _np(res.rows(k))
        assert len(got["hit_root"]) == len(want["hit_root"]), f"config {k}: rows"
        for c in HIT_COLS:
            assert np.array_equal(got[c].view(np.uint8), want[c].view(np.uint8)), f"config {k}: {c}"
        m = len(t.monitors)
        assert np.array_equal(res.hist_y[k].cpu().numpy(), sep["hist_y"][:m].cpu().numpy()), f"config {k}: hist_y"
        assert np.array_equal(res.hist_yz[k].cpu().numpy(), sep["hist_yz"][:m].cpu().numpy()), f"config {k}: hist_yz"
        sums += np.asarray(sep["counters"], np.int64)
    for c in (A.C_SEGMENTS, A.C_INTERACTIONS, A.C_HITS, A.C_DROPPED):
        assert int(res.counters[c]) == int(sums[c]), c
    assert int(res.counters[A.C_STATUS]) == 0
    return res


def _slab(n2, refl, tilt):
    """A glass slab with reflecting faces between two partially transmitting mirrors: every interaction splits and
    the cavity keeps its rays, so roots reach the pop cap."""
    return scenes.Scene([ob.Mirror([-2, 0, 0], radius=3, reflectivity=0.9, transmission=0.1),
                         ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=1, n2=n2, reflectivity=refl).RotZ(tilt),
                         ob.Mirror([2, 0, 0], radius=3, reflectivity=0.9, transmission=0.1).RotZ(np.pi)],
                        [], [ob.Monitor([3, 0, 0], 6, 6), ob.Monitor([-3, 0, 0], 6, 6)])


def _mma(dx):
    """scenes.mma_small with its second array moved along the cavity axis (a pose change that keeps the flattened
    topology; a sideways move can change the box hierarchy the flattener builds over the arrays)."""
    sc = scenes.mma_small(ob)
    grp = ob.ComponentGroup([0, 0, 0])
    pitch, roc = 420e-4, 2.2
    m0 = ob.MMA(origin=[-0.1, 0, 0], N=(6, 1), pitch=pitch, roc=roc, n=1.5, thickness=0.1, reflectivity=0.9999,
                transmission=0, back_transmission=0, back_reflectivity=1)
    m1 = ob.MMA(origin=[2.0, 0, 0], N=(6, 3), pitch=pitch, roc=roc, n=1.5, thickness=0.1, reflectivity=0.98,
                transmission=0.3, shifty_z=-0.002).TY(0.01).TX(dx)
    grp.add_components([m0, m1])
    return scenes.Scene([grp], sc.rays, sc.monitors)


def test_4f_grid_asphere(engine):
    grid = [(43.17 + a, 43.17 + b) for a in (-1.0, 0.0, 0.7) for b in (-0.5, 0.0, 1.1)]
    tables = [telescope_4f_grid(ob, f1, f2) for f1, f2 in grid]
    res = _check_sweep(engine, tables, RayBundle.collimated_disc(100, start=7))
    assert int(res.counters[A.C_INTERACTIONS]) == 4 * 100 * len(grid)


def test_splitting_slab_reaches_the_pop_cap_and_changes_index(engine):
    tables = [_slab(n2, refl, tilt) for n2, refl, tilt in ((1.5, 0.2, 0.0), (1.45, 0.3, 0.05), (1.6, 0.1, -0.08))]
    bundle = RayBundle.collimated_disc(45, x0=-3, radius=0.6, direction=(1.0, 0.01, 0.0))
    res = _check_sweep(engine, tables, bundle, {"max_trace_num": 300})
    assert int(res.counters[A.C_DROPPED]) > 0


def test_sellmeier_glass_change(engine):
    mk = lambda g1, g2: scenes.Scene([ob.Doublet([30.3964, 0, 0], CT1=1.359, CT2=0.6, R1=18.405, R2=-13.734, R3=-39.933,
                                                 n12=g1, n23=g2, diameter=7.5)], [], [ob.Monitor([62, 0, 0], 10, 10)])
    tables = [mk(ob.Glass_NBK7(), ob.Glass_NSF5()), mk(ob.Glass_NSK2(), ob.Glass_NSF11()), mk(ob.Glass_UVFS(), ob.Glass_NSF57())]
    _check_sweep(engine, tables, RayBundle.collimated_disc(33, x0=0, radius=2.5))


def test_mma_moved_group_lattice_walk(engine):
    tables = [_mma(dx) for dx in (0.0, 0.0015, -0.001, 0.003)]
    rays = tables[0].rays
    bundle = _bundle_of(rays)
    res = _check_sweep(engine, tables, bundle, {"max_trace_num": 120})
    # the same sweep from the list of Ray objects (pack_rays) gives the same rows
    res2 = trace_sweep(tables, rays, {"max_trace_num": 120}, engine=engine)
    for c in HIT_COLS:
        assert np.array_equal(res.hits[c].cpu().numpy().view(np.uint8), res2.hits[c].cpu().numpy().view(np.uint8)), c


def test_monitor_as_component_pass_through(engine):
    base = scenes.monitor_as_component(ob)
    tables = []
    for ang in (2.8, 2.75, 2.9):
        lens = ob.Lens([4, 0, 0], focal_length=9.0, radius=2.0)
        screen = ob.Monitor([8, 0.5, 0], 1.2, 1.2).RotZ(0.15)
        mirror = ob.Mirror([12, 0, 0], radius=3.0).RotZ(ang)
        far = ob.Monitor([6, -6, 0], 6, 6).RotZ(-1.2)
        tables.append(scenes.Scene([lens, screen, mirror], [], [screen, far]))
    _check_sweep(engine, tables, _bundle_of(base.rays), base.limit)


def test_single_configuration_equals_trace_bundle(engine):
    _check_sweep(engine, [telescope_4f_grid(ob, 43.17, 43.17)], RayBundle.collimated_disc(77))


def test_two_configurations_against_the_oracle(engine):
    from optable_b200.flatten import FlatScene
    from oracle import oracle as O
    from oracle import ref_harness as RH

    tables = [telescope_4f_grid(ob, 43.17, 43.17), telescope_4f_grid(ob, 42.5, 44.0)]
    bundle = RayBundle.collimated_disc(5000, start=991)
    res = trace_sweep(tables, bundle, engine=engine)
    for k, t in enumerate(tables):
        want = O.trace(FlatScene(t.components, t.monitors), bundle.materialise(), record_segments=False, nthreads=8)
        got = {c: v for c, v in want.items() if c.startswith("seg_")}
        got.update({c: (v.view(np.uint32) if c in A.HIT_U32 else v) for c, v in _np(res.rows(k)).items()})
        parity.compare(RH.arrays_from_result(want), RH.arrays_from_result(got), q_rtol=parity.Q_RTOL_FD, label=f"config {k}")


def test_monitor_statistics_per_configuration(engine):
    from optable_b200.analytics import DeviceMonitor

    tables = [telescope_4f_grid(ob, 43.17 + d, 43.17) for d in (0.0, 0.8)]
    bundle = RayBundle.collimated_disc(2000, start=3)
    res = trace_sweep(tables, bundle, record_hist=True, engine=engine)
    for k, t in enumerate(tables):
        sep = trace_bundle(t, bundle, record_hist=True, engine=engine)
        for m in range(2):
            a, b = res.monitor(k, m).stats(), DeviceMonitor(t.monitors[m], sep, m, engine=engine).stats()
            assert a["count"] == b["count"] > 0
            np.testing.assert_array_equal(a["hist_y"], b["hist_y"])
            for q in ("sum_intensity", "mean_y", "mean_z", "std_y", "min_y", "max_y", "mean_waist_distance"):
                assert a[q] == pytest.approx(b[q], rel=1e-12, abs=1e-15), q


def _sweep_scene(engine, tables):
    from optable_b200.flatten import FlatScene

    return engine.upload_sweep([FlatScene(t.components, t.monitors) for t in tables])


def test_documented_errors(engine):
    from optable_b200.backend import BackendError, lib

    tables = [telescope_4f_grid(ob, 43.17, 43.17), telescope_4f_grid(ob, 43.0, 43.5)]
    scene = _sweep_scene(engine, tables)
    # optb_scene_update_nodes on a sweep scene
    with pytest.raises(BackendError, match=r"-7.*sweep scene"):
        scene.update_nodes([0])
    # K * N >= 2^32: every column broadcast, so nothing of that size is allocated
    bundle = RayBundle.collimated_disc(1)
    rays_t = bundle.to_torch(device=f"cuda:{engine.device}")
    rs = engine._rays_struct(rays_t, n=1 << 31)
    res, _ = engine.alloc_result(scene, 0, 0, 1)
    prm = engine.make_params(record_segments=False, record_hits=False)
    ws = engine._ws(1 << 20)
    rc = lib().optb_trace(engine._ctx, scene._h, C.byref(rs), C.byref(prm), C.byref(res), ws.data_ptr(), int(ws.numel()), None)
    assert rc == -7 and b"2^32" in lib().optb_last_error(engine._ctx)
    scene.close()
    # a topology mismatch is refused by the library too
    from optable_b200.flatten import FlatScene

    f0 = FlatScene(tables[0].components, tables[0].monitors)
    f1 = FlatScene([tables[0].components[0]], tables[0].monitors)
    with pytest.raises(BackendError, match=r"-5.*configuration 1"):
        engine.upload_sweep([f0, f1])


def test_binding_caps_are_rejected(engine):
    from optable_b200.backend import BackendError

    sc = scenes.caps_binding(ob)
    # the Python entry point: a cap below the pop budget cannot be traced as a bundle
    with pytest.raises(NotImplementedError):
        trace_sweep([sc, sc], _bundle_of(sc.rays), sc.limit, engine=engine)
    # the library: a sweep scene with caps and no caps_slack would need the family-serial path
    scene = _sweep_scene(engine, [sc, sc])
    bundle = _bundle_of(sc.rays)
    n = bundle.n * 2
    res, _ = engine.alloc_result(scene, 0, 64, n)
    prm = engine.make_params(80, record_segments=False, n_families=n, caps_slack=0)
    with pytest.raises(BackendError, match=r"-7.*caps_slack"):
        engine.trace_device(scene, bundle.to_torch(device=f"cuda:{engine.device}"), prm, res)
    scene.close()
