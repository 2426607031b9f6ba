"""CPU, build container only: CSV exports (optical_table.py:447-523) against the reference's own, on the
reference's classes and on this package's, with the C oracle standing in for the device."""
import csv
import json

import numpy as np
import pytest

from oracle import ref_harness as RH
from tests import scenes
from tests.test_install_cpu import OracleEngine

needs_reference = pytest.mark.skipif(not RH.reference_available(), reason="the unmodified optable reference package is not installed (baseline/_ref, or OPTABLE_REFERENCE_ROOT)")


def _num(cell):
    """Parse a Mathematica-flavoured cell back into numbers (inverse of base.py:248-251)."""
    if cell == "None" or not isinstance(cell, str):
        return cell
    text = cell.replace("{", "[").replace("}", "]").replace("*10^", "e").replace("I", "j")
    try:
        return np.array(json.loads(text), dtype=float)
    except (ValueError, TypeError):
        pass
    try:
        return complex(text)
    except ValueError:
        return cell  # a name or a class


def _same_rows(want, got, rtol=1e-9):
    assert len(want) == len(got)
    for w, g in zip(want, got):
        assert list(w.keys()) == list(g.keys())
        for k in w:
            a, b = _num(w[k]), _num(g[k])
            if isinstance(a, str) or isinstance(b, str):
                assert a == b, (k, w[k], g[k])
            else:
                assert np.allclose(a, b, rtol=rtol, atol=1e-12), (k, w[k], g[k])


# The reference's ray CSV columns (optical_table.py:448-469), spelled out here rather than taken from the package.
REFERENCE_RAY_KEYS = ["origin", "transform_matrix", "intensity", "length", "qo", "n"]


def check_ray_rows_against_golden(name, rows):
    """Ray-export rows (dicts of cells, as gathered or as read back from the CSV file) against the reference's
    stored segments for the scene (tests/golden/<name>.npz, (root, pop) order), for where the reference package is
    not installed. The expected values come from the stored numbers, not from this package's exporter: every cell
    must parse to the reference's value, a falsy value (an infinite or zero length, no q, zero intensity) must be the
    cell "None" as the reference writes it, and transform_matrix must be a proper rotation taking the x axis onto the
    segment's direction (the stored results hold the direction, not the matrix)."""
    from tests import golden_io

    ref = golden_io.load(name)[3]
    assert len(rows) == len(ref["seg_root"]) > 0
    for k, row in enumerate(rows):
        assert list(row) == REFERENCE_RAY_KEYS
        length, q = float(ref["seg_length"][k]), complex(ref["seg_q"][k])
        want = {"origin": ref["seg_o"][k], "intensity": float(ref["seg_intensity"][k]) or None,
                "length": None if (np.isinf(length) or not length) else length,
                "qo": q if (ref["seg_hasq"][k] and q) else None, "n": float(ref["seg_n"][k]) or None}
        for key, w in want.items():
            cell = _num(row[key])
            if w is None:
                assert cell == "None", (k, key, row[key])
            else:
                assert not isinstance(cell, str) and np.allclose(cell, w, rtol=1e-9, atol=1e-12), (k, key, row[key], w)
        M = _num(row["transform_matrix"])
        d = ref["seg_d"][k] / np.linalg.norm(ref["seg_d"][k])
        assert M.shape == (3, 3) and np.allclose(M[:, 0], d, rtol=0, atol=1e-9), (k, row["transform_matrix"], d)
        assert np.allclose(M.T @ M, np.identity(3), rtol=0, atol=1e-9) and abs(np.linalg.det(M) - 1.0) <= 1e-9


@pytest.mark.parametrize("name", ["doublet", "misc_components", "telescope_4f", "mma_small"])
@needs_reference
def test_component_rows_equal_reference(name):
    import optable_b200 as ob

    ref = RH.load_reference()
    a, b = scenes.REGISTRY[name](ref), scenes.REGISTRY[name](ob)
    ta, tb = ref.OpticalTable(), ob.OpticalTable()
    ta.add_components(a.components)
    tb.add_components(b.components)
    _same_rows(ta.gather_components(), tb.gather_components(), rtol=1e-12)
    kw = dict(avoid_flatten_classname=["Doublet", "MMA"], ignore_classname=["Mirror", "Refraction"])
    _same_rows(ta.gather_components(**kw), tb.gather_components(**kw), rtol=1e-12)


@pytest.mark.parametrize("name", ["gaussian_beam", "chromatic", "prism_refl"])
def test_ray_rows_equal_reference(name, tmp_path):
    """Where the reference package is not installed, the three row sets are checked against its stored segments
    for the scene (check_ray_rows_against_golden)."""
    import optable_b200 as ob
    from optable_b200 import export
    from optable_b200.flatten import FlatScene, pack_rays, trace_cap
    from optable_b200.table import trace_table

    if not RH.reference_available():
        b = scenes.REGISTRY[name](ob)
        tb = ob.OpticalTable()
        tb.add_components(b.components)
        tb.add_monitors(b.monitors)
        tb.rays.extend(trace_table(tb, list(b.rays), b.limit, engine=OracleEngine()))
        arrs, fams, unit = pack_rays(b.rays)
        out = OracleEngine().trace_arrays(OracleEngine().upload(FlatScene(tb.components, tb.monitors)), arrs,
                                          max_trace_num=trace_cap(b.limit), unit=unit, n_families=len(fams))
        tb.export_rays_csv(str(tmp_path / "own.csv"))
        rb = list(csv.reader(open(tmp_path / "own.csv")))
        for rows in (tb.gather_rays_csv(), export.segment_rows(out), [dict(zip(rb[0], r)) for r in rb[1:]]):
            check_ray_rows_against_golden(name, rows)
        return
    ref = RH.load_reference()
    a, b = scenes.REGISTRY[name](ref), scenes.REGISTRY[name](ob)
    ta, tb = ref.OpticalTable(), ob.OpticalTable()
    for t, sc in ((ta, a), (tb, b)):
        t.add_components(sc.components)
        t.add_monitors(sc.monitors)
    ta.ray_tracing(a.rays, perfomance_limit=a.limit)
    tb.rays.extend(trace_table(tb, list(b.rays), b.limit, engine=OracleEngine()))
    want = ta.gather_rays_csv()
    _same_rows(want, tb.gather_rays_csv())
    # straight from the segment columns, no Ray objects in between
    arrs, fams, unit = pack_rays(b.rays)
    out = OracleEngine().trace_arrays(OracleEngine().upload(FlatScene(tb.components, tb.monitors)), arrs,
                                      max_trace_num=trace_cap(b.limit), unit=unit, n_families=len(fams))
    _same_rows(want, export.segment_rows(out))
    # files: same header, same number of lines, cells parse to the same numbers
    fa, fb = tmp_path / "ref.csv", tmp_path / "own.csv"
    ta.export_rays_csv(str(fa))
    tb.export_rays_csv(str(fb))
    ra, rb = list(csv.reader(open(fa))), list(csv.reader(open(fb)))
    assert ra[0] == rb[0] == list(export.RAY_KEYS) and len(ra) == len(rb)
    _same_rows([dict(zip(ra[0], r)) for r in ra[1:]], [dict(zip(rb[0], r)) for r in rb[1:]])


def test_empty_exports(tmp_path):
    import optable_b200 as ob

    t = ob.OpticalTable()
    t.export_rays_csv(str(tmp_path / "r.csv"))
    t.export_components_csv(str(tmp_path / "c.csv"))
    assert open(tmp_path / "r.csv").read().strip() == "" and open(tmp_path / "c.csv").read().strip() == ""
