"""Shared check of the drop-in boundary on the reference's OWN classes: `optable_b200.install(reference)` with a
given engine (the C oracle in the CPU tests, the CUDA engine in the `-m gpu` tests) against the reference's original
`OpticalTable.ray_tracing` on an identically built scene. Compares `table.rays` object by object, the `_id`
family partition, every monitor's `_data_raw` rows (and that they point at the objects of `table.rays`), the
reference's own accessors on backend-filled monitors, and `_interact_count` of every leaf."""
import numpy as np
import pytest

from oracle import ref_harness as RH
from tests import parity, scenes


def fields(r):
    return (np.array(r.origin, float), np.array(r.direction, float), r.length, bool(r.alive), float(r.intensity),
            float(r.wavelength), r.qo, float(r._pathlength), float(r.n), r._id)


def assert_same_segment(fw, fg, q_rtol=1e-9):
    assert parity._rel_vec(fw[0], fg[0], 1.0) <= 1e-9 and parity._rel_vec(fw[1], fg[1], 1.0) <= 1e-9
    assert (fw[2] is None) == (fg[2] is None) and (fw[2] is None or abs(fw[2] - fg[2]) <= 1e-9 * max(abs(fw[2]), 1e-3))
    assert fw[3] == fg[3] and fw[4] == pytest.approx(fg[4], rel=1e-9) and fw[5] == fg[5]
    assert (fw[6] is None) == (fg[6] is None) and (fw[6] is None or abs(fw[6] - fg[6]) <= q_rtol * abs(fw[6]))
    assert fw[7] == pytest.approx(fg[7], rel=1e-9, abs=1e-12) and fw[8] == pytest.approx(fg[8], rel=1e-12)


def check_install(name, engine, q_rtol=1e-9):
    import optable_b200

    ref = RH.load_reference()
    a, b = scenes.REGISTRY[name](ref), scenes.REGISTRY[name](ref)
    ta, tb = ref.OpticalTable(), ref.OpticalTable()
    for t, sc in ((ta, a), (tb, b)):
        t.add_components(sc.components)
        t.add_monitors(sc.monitors)
    want = ta.ray_tracing(a.rays, perfomance_limit=a.limit)          # the reference's own method
    original = optable_b200.install(ref, engine=engine)
    try:
        got = tb.ray_tracing(b.rays, perfomance_limit=b.limit)       # same call, swapped back end
    finally:
        ref.OpticalTable.ray_tracing = original
    assert len(got) == len(want) == len(tb.rays)
    for rw, rg in zip(ta.rays, tb.rays):
        assert_same_segment(fields(rw), fields(rg), q_rtol)
    # ids: the reference keys families by Ray._id; copies made by the two scene builds differ in id(), so compare
    # the partition of segments into families instead of the raw values
    fam_w = {}
    fam_g = {}
    for k, (rw, rg) in enumerate(zip(ta.rays, tb.rays)):
        fam_w.setdefault(rw._id, []).append(k)
        fam_g.setdefault(rg._id, []).append(k)
    assert sorted(fam_w.values()) == sorted(fam_g.values())
    on_table = {id(s) for s in tb.rays}
    for mw, mg in zip(ta.monitors, tb.monitors):
        assert len(mw._data_raw) == len(mg._data_raw) and (mg._updated or not mw._data_raw)
        for (Pw, Iw, tw, rw), (Pg, Ig, tg, rg) in zip(mw._data_raw, mg._data_raw):
            assert np.linalg.norm(np.asarray(Pw) - np.asarray(Pg)) <= 1e-9 * max(np.linalg.norm(Pw), 1.0)
            assert Iw == pytest.approx(Ig, rel=1e-9) and tw == pytest.approx(tg, rel=1e-9)
            assert id(rg) in on_table                 # rows reference the segment objects of table.rays
        if mw._data_raw:                              # the reference's accessors run on backend-filled monitors
            np.testing.assert_allclose(mg.get_yList(), mw.get_yList(), rtol=1e-9, atol=1e-12)  # YZ order: ids are id() values
            np.testing.assert_allclose(mg.get_tYList(), mw.get_tYList(), rtol=1e-9, atol=1e-12)
    leaves_w, leaves_g = RH._leaves(ta.components, []), RH._leaves(tb.components, [])
    for cw, cg in zip(leaves_w, leaves_g):
        assert sorted(cw._interact_count.values()) == sorted(cg._interact_count.values()) or cw.max_interact_count is None
    return len(tb.rays), sum(len(m._data_raw) for m in tb.monitors)


def golden_fields(want, k):
    """`fields` of segment k of a stored reference result (tests/golden/<name>.npz, (root, pop) order)."""
    import math

    return (want["seg_o"][k], want["seg_d"][k], None if math.isinf(want["seg_length"][k]) else float(want["seg_length"][k]),
            bool(want["seg_alive"][k]), float(want["seg_intensity"][k]), float(want["seg_wavelength"][k]),
            complex(want["seg_q"][k]) if want["seg_hasq"][k] else None, float(want["seg_pathlength"][k]),
            float(want["seg_n"][k]))


def check_monitor_rows_against_golden(monitors, want, segments):
    """Every monitor's `_data_raw` rows against the stored reference rows, in order; each row must point at one of
    `segments` (the objects of the traced table)."""
    on_table = {id(s) for s in segments}
    for mi, mon in enumerate(monitors):
        sel = want["hit_monitor"] == mi
        assert mon.ndata == len(mon._data_raw) == int(sel.sum())
        for Pw, Iw, tw, (Pg, Ig, tg, rg) in zip(want["hit_P"][sel], want["hit_intensity"][sel], want["hit_t"][sel], mon._data_raw):
            assert np.linalg.norm(Pw - np.asarray(Pg)) <= 1e-9 * max(np.linalg.norm(Pw), 1.0)
            assert Iw == pytest.approx(Ig, rel=1e-9) and tw == pytest.approx(tg, rel=1e-9)
            assert id(rg) in on_table


def check_against_golden(name, q_rtol=1e-9):
    """`check_install` where the reference package is not installed: this package's own classes traced by its
    `OpticalTable.ray_tracing` (the CUDA engine) against the reference's results for the same scene as
    oracle/make_golden.py stored them (tests/golden/<name>.npz): `table.rays` segment by segment, the `_id` family
    partition, every monitor's `_data_raw` rows (pointing at the objects of `table.rays`) and `_interact_count`."""
    import optable_b200 as ob
    from optable_b200.flatten import pack_rays
    from tests import golden_io

    want = golden_io.load(name)[3]
    sc = scenes.REGISTRY[name](ob)
    table = ob.OpticalTable()
    table.add_components(sc.components)
    table.add_monitors(sc.monitors)
    got = table.ray_tracing(sc.rays, perfomance_limit=sc.limit)
    assert len(got) == len(table.rays) == len(want["seg_root"])
    for k, rg in enumerate(table.rays):
        assert_same_segment(golden_fields(want, k), fields(rg), q_rtol)
    # families: every segment descends from the initial ray of its root and keeps that ray's `_id`
    fam_w, fam_g = {}, {}
    for k, rg in enumerate(table.rays):
        fam_w.setdefault(sc.rays[int(want["seg_root"][k])]._id, []).append(k)
        fam_g.setdefault(rg._id, []).append(k)
    assert sorted(fam_w.values()) == sorted(fam_g.values())
    check_monitor_rows_against_golden(table.monitors, want, table.rays)
    flat = sc.flat()   # (the same component objects the table traced: cap slots point at their `_interact_count`)
    if flat.n_capslots:
        _, fam_ids, _ = pack_rays(sc.rays)
        for s, comp in enumerate(flat.capslots):
            for f, rid in enumerate(fam_ids):
                assert comp._interact_count.get(rid, 0) == int(want["cap_counts"][s, f])
    return len(table.rays), sum(len(m._data_raw) for m in table.monitors)
