"""CPU, build container only: the drop-in boundary on the reference's OWN classes.

`optable_b200.install(reference)` replaces `OpticalTable.ray_tracing`; everything around the device call (scene
flattening from reference objects, ray packing, rebuilding `table.rays`, filling `Monitor._data_raw`, updating
`_interact_count`) is exercised here with the C oracle standing in for the CUDA engine (same table/array
contract as `Engine.trace_arrays`), and compared object by object with what the reference's original method
produces on an identical scene."""
import numpy as np
import pytest

from oracle import oracle as O
from oracle import ref_harness as RH
from tests import parity, scenes

needs_reference = pytest.mark.skipif(not RH.reference_available(), reason="the unmodified optable reference package is not installed (baseline/_ref, or OPTABLE_REFERENCE_ROOT)")


class OracleEngine:
    """Stands in for optable_b200.backend.Engine in trace_table (test infrastructure)."""

    class _Scene:
        def __init__(self, flat):
            self.flat = flat

        def close(self):
            pass

    def upload(self, flat):
        return self._Scene(flat)

    def trace_arrays(self, scene, arrs, max_trace_num=2000, unit=1e-2, n_families=None, cap_counts=None, **kw):
        out = O.trace(scene.flat, arrs, max_trace_num=max_trace_num, unit=unit, n_families=n_families, cap_counts=cap_counts)
        order = np.lexsort((out["hit_pop"], out["hit_monitor"], out["hit_root"]))
        for k in list(out):
            if k.startswith("hit_"):
                out[k] = out[k][order]
        return out


from tests.install_check import fields as _fields  # noqa: E402


@needs_reference
@pytest.mark.parametrize("name", ["gaussian_beam", "chromatic", "doublet", "telescope_4f", "prism_refl", "caps_binding",
                                  "dove_prism", "misc_components", "mma_small"])
def test_installed_backend_equals_original_method(name):
    from tests.install_check import check_install

    check_install(name, OracleEngine())


@pytest.mark.parametrize("name", ["gaussian_beam", "chromatic", "telescope_4f", "prism_refl", "misc_components"])
def test_own_classes_through_trace_table_equal_reference(name):
    """This package's own scene classes + `OpticalTable.ray_tracing` host logic (ray packing, the `Ray` fast path
    of the segment builder, columnar monitors), oracle engine in place of the device: segment for segment equal
    to the reference's method on the reference's classes. Where the reference package is not installed, the
    segments and monitor rows are compared with the reference's stored results for the scene (tests/golden)."""
    import optable_b200 as ob
    from optable_b200.table import trace_table
    from tests import golden_io
    from tests.install_check import assert_same_segment, check_monitor_rows_against_golden, golden_fields

    live = RH.reference_available()
    b = scenes.REGISTRY[name](ob)
    tb = ob.OpticalTable()
    tb.add_components(b.components)
    tb.add_monitors(b.monitors)
    if live:
        ref = RH.load_reference()
        a = scenes.REGISTRY[name](ref)
        ta = ref.OpticalTable()
        ta.add_components(a.components)
        ta.add_monitors(a.monitors)
        ta.ray_tracing(a.rays, perfomance_limit=a.limit)
        want_fields = [_fields(r) for r in ta.rays]
    else:
        want = golden_io.load(name)[3]
        want_fields = [golden_fields(want, k) for k in range(len(want["seg_root"]))]
    before = [(_fields(r), dict(r.__dict__)) for r in b.rays]
    segs = trace_table(tb, list(b.rays), b.limit, engine=OracleEngine())
    assert len(segs) == len(want_fields)
    for fw, rg in zip(want_fields, segs):
        assert type(rg) is ob.Ray
        assert_same_segment(fw, _fields(rg))
        assert isinstance(rg.length, (float, type(None))) and isinstance(rg.alive, bool) and isinstance(rg.intensity, float)
    # every segment keeps the `_id` of the initial ray it descends from, and owns its arrays
    ids = {r._id for r in b.rays}
    assert {s._id for s in segs} <= ids
    segs[0].origin[0] += 1.0
    assert all(s.origin[0] != segs[0].origin[0] or s is segs[0] for s in segs[1:2])
    # inputs untouched
    for r, (f0, d0) in zip(b.rays, before):
        f1 = _fields(r)
        assert np.array_equal(f0[0], f1[0]) and np.array_equal(f0[1], f1[1]) and f0[2:] == f1[2:]
    if not live:
        check_monitor_rows_against_golden(tb.monitors, want, segs)
        return
    for mw, mg in zip(ta.monitors, tb.monitors):
        assert len(mw._data_raw) == mg.ndata
        if mw._data_raw:
            np.testing.assert_allclose(mg.get_yList(sort="YZ"), mw.get_yList(sort="YZ"), rtol=1e-9, atol=1e-12)
            np.testing.assert_allclose(mg.get_tYList(sort="YZ"), mw.get_tYList(sort="YZ"), rtol=1e-9, atol=1e-12)


@needs_reference
def test_monitor_record_explicit_segments_equals_reference():
    """`Monitor.record(list_of_rays)` called directly (monitor.py:183-193): finite, infinite and dead segments,
    misses, hits behind the origin; rows must reference the objects passed in."""
    import optable_b200 as ob

    ref = RH.load_reference()
    rng = np.random.default_rng(7)

    def build(mod):
        mon = mod.Monitor(origin=[5, 0.2, -0.1], width=2, height=1.5).RotZ(0.3).RotY(-0.2)
        rays = []
        for k in range(40):
            o = [rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(-1, 1)]
            d = [1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)]
            if k % 7 == 0:
                d[0] = -1.0                                   # monitor behind the ray
            kw = {}
            if k % 3 == 0:
                kw["length"] = float(rng.uniform(2.0, 9.0))   # may end before the plane
            if k % 5 == 0:
                kw["alive"] = False
            if k % 2 == 0:
                kw["w0"] = 0.01
            rays.append(mod.Ray(o, d, wavelength=780e-7, intensity=float(rng.uniform(0.1, 1.0)), **kw))
        return mon, rays

    state = rng.bit_generator.state
    mw, rw = build(ref)
    rng.bit_generator.state = state
    mg, rg = build(ob)
    mw.record(rw)
    mg.record(rg, engine=OracleEngine())
    assert mg._updated and mg.ndata == len(mw._data_raw) > 5
    for (Pw, Iw, tw, r_w), (Pg, Ig, tg, r_g) in zip(mw._data_raw, mg._data_raw):
        assert np.linalg.norm(np.asarray(Pw) - Pg) <= 1e-9 and Iw == pytest.approx(Ig, rel=1e-12) and tw == pytest.approx(tg, rel=1e-9)
        assert rw.index(r_w) == next(i for i, r in enumerate(rg) if r is r_g)
    np.testing.assert_allclose(mg.get_yList(), mw.get_yList(), rtol=1e-9, atol=1e-12)
    mg.record([], engine=OracleEngine())
    assert mg.ndata == len(mw._data_raw)


def test_ripa2_example_analysis_with_oracle_engine():
    """Host side of the same example (tests/test_gpu_api.py::test_ripa2_example_with_its_analysis) on the CPU."""
    import os

    import optable_b200 as ob
    from optable_b200.table import trace_table
    from tests import golden_io

    sc = scenes.ripa2_simplified(ob)
    table = ob.OpticalTable()
    table.add_components(sc.components)
    table.add_monitors(sc.monitors)
    table.rays.extend(trace_table(table, list(sc.rays), None, engine=OracleEngine()))
    got = scenes.ripa2_postprocess(ob, table, sc)
    want = np.load(os.path.join(golden_io.GOLDEN_DIR, "ripa2_post.npz"))
    np.testing.assert_allclose(got["P"], want["P"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(got["n"], want["n"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(got["pathlength"], want["pathlength"], rtol=1e-9)
    np.testing.assert_allclose(got["roc"], want["roc"], rtol=1e-5)


def test_abcd_matrix_batched_first_traces_equal_three_separate_traces(monkeypatch):
    """calculate_abcd_matrix traces the nominal and the shifted bundle as one batch (columns only). Same matrices,
    same final table state as the three separate ray_tracing calls it replaces (forced here by a third monitor on
    the table), and the reference's own values (tests/golden/abcd_4f.npz)."""
    import os

    import optable_b200 as ob
    from optable_b200 import backend
    from tests import golden_io

    monkeypatch.setattr(backend.Engine, "get", classmethod(lambda cls, device=None: OracleEngine()))
    z = np.load(os.path.join(golden_io.GOLDEN_DIR, "abcd_4f.npz"))
    F1, F2 = z["F"]

    def build(extra_monitor):
        lens = scenes.asphere_lens9(ob, [43.17, 0, 0])
        l0 = lens.copy()._Translate(np.array([F1, 0, 0]) - lens.origin)
        l1 = lens.copy()._Translate(np.array([F1 + 2 * F2, 0, 0]) - lens.origin).RotZ(np.pi)
        m0, m1 = ob.Monitor(origin=[0, 0, 0], width=5, height=5), ob.Monitor(origin=[2 * F1 + 2 * F2, 0, 0], width=5, height=5)
        table = ob.OpticalTable()
        table.add_components([l0, l1])
        table.add_monitors([m0, m1] + ([ob.Monitor(origin=[-5, 0, 0], width=1, height=1)] if extra_monitor else []))
        return table, m0, m1

    fast_t, fm0, fm1 = build(False)
    slow_t, sm0, sm1 = build(True)
    calls = []
    real = ob.OpticalTable.ray_tracing
    monkeypatch.setattr(ob.OpticalTable, "ray_tracing", lambda self, rays, perfomance_limit=None: (calls.append(self), real(self, rays, perfomance_limit))[1])
    # (the wrapper is installed on the class, so `type(self).ray_tracing is OpticalTable.ray_tracing` still holds)
    Mf = fast_t.calculate_abcd_matrix(fm0, fm1, scenes.abcd_rays(ob))
    Ms = slow_t.calculate_abcd_matrix(sm0, sm1, scenes.abcd_rays(ob))
    assert calls.count(fast_t) == 1 and calls.count(slow_t) == 3
    np.testing.assert_allclose(Mf, Ms, rtol=0, atol=1e-12)
    np.testing.assert_allclose(Mf, z["Ms"], rtol=1e-5, atol=2e-4)
    assert len(fast_t.rays) == len(slow_t.rays) and fm1.ndata == sm1.ndata == 7
    np.testing.assert_allclose(fm1.get_yList(sort="ID"), sm1.get_yList(sort="ID"), rtol=0, atol=1e-15)
    np.testing.assert_allclose([r.origin for r in fast_t.rays], [r.origin for r in slow_t.rays], rtol=0, atol=1e-15)


@needs_reference
def test_component_interact_single_pop_equals_reference():
    """`component.interact(ray)` (one pop against one component or group, optical_component.py:337-378) through the
    device path (oracle engine here): t, the truncated parent and every child ray against the reference's."""
    import optable_b200 as ob

    ref = RH.load_reference()
    rng = np.random.default_rng(5)
    n_checked = n_hits = 0
    for name in ("misc_components", "doublet", "telescope_4f", "prism_refl", "extras"):
        a, b = scenes.REGISTRY[name](ref), scenes.REGISTRY[name](ob)
        for ca, cb in zip(a.components, b.components):
            for ra, rb in list(zip(a.rays, b.rays))[:6]:
                tw, rw = ca.interact(ra)
                tg, rg = cb.interact(rb, engine=OracleEngine())
                n_checked += 1
                assert (tw is None) == (tg is None), (name, type(ca).__name__)
                if tw is None:
                    assert rg is None
                    continue
                n_hits += 1
                assert tg == pytest.approx(tw, rel=1e-9) and len(rg) == len(rw)
                for x, y in zip(rw, rg):
                    fx, fy = _fields(x), _fields(y)
                    assert parity._rel_vec(fx[0], fy[0], 1.0) <= 1e-9 and parity._rel_vec(fx[1], fy[1], 1.0) <= 1e-9
                    assert (fx[2] is None) == (fy[2] is None) and (fx[2] is None or abs(fx[2] - fy[2]) <= 1e-9 * max(abs(fx[2]), 1e-3))
                    assert fx[3] == fy[3] and fx[4] == pytest.approx(fy[4], rel=1e-9, abs=1e-300) and fx[5] == fy[5]
                    assert (fx[6] is None) == (fy[6] is None) and (fx[6] is None or abs(fx[6] - fy[6]) <= 1e-6 * abs(fx[6]))
                    assert fx[7] == pytest.approx(fy[7], rel=1e-9, abs=1e-12) and fx[8] == pytest.approx(fy[8], rel=1e-12)
        leaves_a, leaves_b = RH._leaves(a.components, []), RH._leaves(b.components, [])
        for la, lb in zip(leaves_a, leaves_b):   # interact counts moved the same way
            assert la.max_interact_count is None or sorted(la._interact_count.values()) == sorted(lb._interact_count.values())
    assert n_checked > 100 and n_hits > 20
