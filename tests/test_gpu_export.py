"""GPU: the segment stream -> CSV exports of the reference (optical_table.py:447-523, SURVEY 8f item 4) fed by the
CUDA engine: cell for cell the numbers the unmodified reference (baseline/_ref) writes for the same scene, both
through Ray objects (`OpticalTable.export_rays_csv`) and straight from the device's segment columns
(`export.segment_rows`), plus the component table."""
import csv

import numpy as np
import pytest

from oracle import ref_harness as RH
from tests import scenes
from tests.test_export_cpu import _same_rows, check_ray_rows_against_golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["gaussian_beam", "chromatic", "prism_refl", "doublet", "callable_material"])
def test_ray_csv_rows_from_the_device_equal_reference(name, tmp_path):
    """Where the reference package is not installed, the same three row sets (Ray objects, device segment columns,
    the CSV file) are checked cell by cell against the reference's stored segments for the scene
    (tests/test_export_cpu.check_ray_rows_against_golden); the component table needs the live reference."""
    import optable_b200 as ob
    from optable_b200 import export
    from optable_b200.backend import Engine
    from optable_b200.flatten import pack_rays, trace_cap

    live = RH.reference_available()
    b = scenes.REGISTRY[name](ob)
    tb = ob.OpticalTable()
    tb.add_components(b.components)
    tb.add_monitors(b.monitors)
    tb.ray_tracing(b.rays, perfomance_limit=b.limit)      # liboptb.so
    # straight from the device's segment columns, no Ray objects in between
    engine = Engine.get(0)
    arrs, fams, unit = pack_rays(b.rays)
    scene = engine.upload(b.flat())
    out = engine.trace_arrays(scene, arrs, max_trace_num=trace_cap(b.limit), unit=unit, n_families=len(fams))
    scene.close()
    fb = tmp_path / "own.csv"
    tb.export_rays_csv(str(fb))
    rb = list(csv.reader(open(fb)))
    file_rows = [dict(zip(rb[0], r)) for r in rb[1:]]
    if not live:
        for rows in (tb.gather_rays_csv(), export.segment_rows(out), file_rows):
            check_ray_rows_against_golden(name, rows)
        return
    ref = RH.load_reference()
    a = scenes.REGISTRY[name](ref)
    ta = ref.OpticalTable()
    ta.add_components(a.components)
    ta.add_monitors(a.monitors)
    ta.ray_tracing(a.rays, perfomance_limit=a.limit)      # the reference, on the host
    want = ta.gather_rays_csv()
    _same_rows(want, tb.gather_rays_csv())
    _same_rows(want, export.segment_rows(out))
    fa = tmp_path / "ref.csv"
    ta.export_rays_csv(str(fa))
    ra = list(csv.reader(open(fa)))
    assert ra[0] == rb[0] == list(export.RAY_KEYS) and len(ra) == len(rb) > 1
    _same_rows([dict(zip(ra[0], r)) for r in ra[1:]], file_rows)
    _same_rows(ta.gather_components(), tb.gather_components(), rtol=1e-12)
