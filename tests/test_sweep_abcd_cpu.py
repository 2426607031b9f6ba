"""CPU: the host side of sweep ABCD matrices (optable_b200.sweep.sweep_abcd_matrix, SweepScene.abcd_matrix): the two
bundles the sweeps trace, and the refusals that come before any device call."""
import numpy as np
import pytest

import optable_b200 as ob
from optable_b200 import backend
from optable_b200 import table as table_mod
from optable_b200.flatten import pack_rays
from optable_b200.sweep import SweepScene, _abcd_bundle_a, _abcd_bundle_b, _abcd_work, sweep_abcd_matrix
from optable_b200.workloads import telescope_4f_grid
from tests import scenes
from tests.test_install_cpu import OracleEngine


def _table(F1=43.17, F2=43.17, extra=()):
    sc = telescope_4f_grid(ob, F1, F2)
    t = ob.OpticalTable()
    t.add_components(list(sc.components) + list(extra))
    t.add_monitors(list(sc.monitors))
    return t


def _no_device(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("a refusal must come before any device call")

    monkeypatch.setattr(backend.Engine, "get", classmethod(refuse))


def test_bundles_equal_what_calculate_abcd_matrix_traces(monkeypatch):
    """Sweep A's bundle is the batch of the table method's first (combined) trace and sweep B's the batch of its
    third, column for column after pack_rays, given the same pivots (the C oracle stands in for the device)."""
    monkeypatch.setattr(backend.Engine, "get", classmethod(lambda cls, device=None: OracleEngine()))
    batches, firsts = [], []
    real_pack, real_first = table_mod.pack_rays, ob.OpticalTable._abcd_first_two_traces
    # (packed when traced: the table method moves its ray objects in place between the traces)
    monkeypatch.setattr(table_mod, "pack_rays", lambda rays: (batches.append(real_pack(rays)), batches[-1])[1])
    monkeypatch.setattr(ob.OpticalTable, "_abcd_first_two_traces",
                        lambda self, *a: (firsts.append(real_first(self, *a)), firsts[-1])[1])
    t = _table(42.0, 44.5)
    mon0, mon1 = t.monitors
    rays = scenes.abcd_rays(ob)[::-1]            # out of id order: both sides sort by id
    disp, rot = 2e-5, 3e-5
    t.calculate_abcd_matrix(mon0, mon1, rays, disp=disp, rot=rot)
    assert len(batches) == 2 and len(firsts) == 1
    pivots = firsts[0][0][2]
    work, ids = _abcd_work(rays, None)
    assert ids == sorted(r._id for r in rays)
    for got, want in ((pack_rays(_abcd_bundle_a(work, mon0, disp)), batches[0]),
                      (pack_rays(_abcd_bundle_b(work, mon0, pivots, disp, rot)), batches[1])):
        assert got[2] == want[2]
        assert got[0].keys() == want[0].keys()
        for k in want[0]:
            np.testing.assert_array_equal(got[0][k], want[0][k], err_msg=k)


def test_repeated_ids_are_refused_with_the_reference_wording(monkeypatch):
    _no_device(monkeypatch)
    rays = scenes.abcd_rays(ob)
    rays[1]._id = rays[0]._id
    with pytest.raises(ValueError, match="Redundant ray ids in ABCD calculation."):
        sweep_abcd_matrix([_table(), _table(43.0, 43.5)], 0, 1, rays)
    sw = SweepScene(_table(), vary=[])
    with pytest.raises(ValueError, match="Redundant ray ids in ABCD calculation."):
        sw.abcd_matrix(0, 1, rays, lambda k: None, 2)


def test_interact_caps_and_sharding_are_refused(monkeypatch):
    _no_device(monkeypatch)
    capped = lambda: ob.Mirror([300, 0, 0], max_interact_count=3)
    rays = scenes.abcd_rays(ob)
    with pytest.raises(NotImplementedError, match="interact-capped"):
        sweep_abcd_matrix([_table(extra=[capped()]), _table(43.0, 43.5, extra=[capped()])], 0, 1, rays)
    calls = []
    sw = SweepScene(_table(extra=[capped()]), vary=[])
    with pytest.raises(NotImplementedError, match="interact-capped"):
        sw.abcd_matrix(0, 1, rays, calls.append, 2)
    assert calls == []
    with pytest.raises(NotImplementedError, match="group="):
        sweep_abcd_matrix([_table()], 0, 1, rays, group=True)
    with pytest.raises(NotImplementedError, match="group="):
        SweepScene(_table(), vary=[]).abcd_matrix(0, 1, rays, calls.append, 2, group=True)


def test_configurations_that_move_mon0_are_refused(monkeypatch):
    """mon0 must stand where configuration 0 put it: the three bundles are built from its frame."""
    _no_device(monkeypatch)
    rays = scenes.abcd_rays(ob)
    t = _table()
    mon0, mon1 = t.monitors
    lens2 = t.components[1]
    x2 = lens2.origin.copy()
    sw = SweepScene(t, vary=[lens2, mon0, mon1])

    def configure(k):
        lens2.origin = x2 + [0.1 * k, 0, 0]
        mon0.origin = np.array([0.0, 0.0, 0.0]) + ([0, 1e-3, 0] if k == 2 else 0)

    with pytest.raises(ValueError, match=r"configuration 2 changes the origin of mon0 \(monitor 0\).*bundle per configuration"):
        sw.abcd_matrix(mon0, mon1, rays, configure, 4)

    def turn(k):
        mon0.origin = np.array([0.0, 0.0, 0.0])
        if k == 1:
            mon0.RotZ(1e-3)

    with pytest.raises(ValueError, match="configuration 1 changes the tangent_Y of mon0"):
        sw.abcd_matrix(0, 1, rays, turn, 3)
    moved = _table()
    moved.monitors[0].width = 4.0
    with pytest.raises(ValueError, match="configuration 1 changes the width of mon0"):
        sweep_abcd_matrix([_table(), moved], 0, 1, rays)
    with pytest.raises(ValueError, match="not a monitor of the table"):
        sw.abcd_matrix(ob.Monitor([0, 0, 0], 1, 1), 1, rays, configure, 2)
