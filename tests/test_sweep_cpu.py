"""CPU: scene sweeps (optable_b200.sweep) -- topology checks, and the result layout with the C oracle standing in for
the device: rows(k), the root rebasing and the [K, M, ...] histograms equal K separate traces."""
import os
import re

import numpy as np
import pytest
import torch

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.bundle import RayBundle
from optable_b200.flatten import FlatScene
from optable_b200.sweep import SweepResult, check_topology, trace_sweep
from optable_b200.workloads import telescope_4f_grid
from tests import scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64


def _oracle_sweep(flats, rays, limit, record_hits=True, record_hist=False, engine=None, unit=None, arrs=None):
    """Stand-in for the CUDA sweep: K oracle traces, roots renumbered k * N + r, rows and histograms concatenated in
    configuration order (the layout one optb_trace on a sweep scene produces once its rows are sorted)."""
    from oracle import oracle as O

    arrs = rays.materialise() if arrs is None else arrs
    n = len(arrs["ox"])
    parts = [O.trace(f, arrs, max_trace_num=limit, record_segments=False, record_hits=record_hits, record_hist=True)
             for f in flats]
    out = {}
    if record_hits:
        for k in HIT_COLS:
            cols = [p[k].astype(np.int64) + c * n if k == "hit_root" else p[k] for c, p in enumerate(parts)]
            v = np.concatenate(cols)
            out[k] = torch.from_numpy(v.astype(np.uint32).view(np.int32) if k == "hit_root" else
                                      (v.view(np.int32) if v.dtype == np.uint32 else v))
    out["hist_y"] = torch.from_numpy(np.concatenate([p["hist_y"] for p in parts]))
    out["hist_yz"] = torch.from_numpy(np.concatenate([p["hist_yz"] for p in parts]))
    out["counters"] = np.sum([p["counters"] for p in parts], axis=0)
    return out


def _grid(F=((43.17, 43.17), (42.0, 44.5), (44.0, 41.9))):
    return [telescope_4f_grid(ob, f1, f2) for f1, f2 in F]


def test_sweep_rows_and_histograms_equal_separate_traces():
    from oracle import oracle as O

    tables = _grid()
    bundle = RayBundle.collimated_disc(37)   # not a multiple of 32: warps straddle configurations on the device
    res = trace_sweep(tables, bundle, record_hist=True, tracer=_oracle_sweep)
    assert isinstance(res, SweepResult) and res.n == 37 and res.n_configs == 3
    assert tuple(res.hist_y.shape) == (3, 2, A.HIST_BINS) and tuple(res.hist_yz.shape) == (3, 2, A.HIST_BINS, A.HIST_BINS)
    total = 0
    for k, t in enumerate(tables):
        want = O.trace(FlatScene(t.components, t.monitors), bundle.materialise(), record_segments=False, record_hist=True)
        got = res.rows(k)
        assert len(got["hit_root"]) == len(want["hit_root"]) > 0
        for c in HIT_COLS:
            np.testing.assert_array_equal(got[c].numpy().view(want[c].dtype) if want[c].dtype == np.uint32 else got[c].numpy(),
                                          want[c], err_msg=f"config {k} {c}")
        np.testing.assert_array_equal(got["hist_y"].numpy(), want["hist_y"])
        np.testing.assert_array_equal(got["hist_yz"].numpy(), want["hist_yz"])
        total += int(want["counters"][A.C_HITS])
    assert int(res.counters[A.C_HITS]) == total
    with pytest.raises(IndexError):
        res.rows(3)


def test_sweep_of_ray_objects_uses_their_packing():
    sc = scenes.glass_slab(ob)
    tables = [scenes.Scene([ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=1, n2=n2, reflectivity=0.2)],
                           [], [ob.Monitor([2, 0, 0], 4, 4)]) for n2 in (1.4, 1.5)]
    seen = {}

    def tracer(flats, rays, limit, **kw):
        seen.update(kw, limit=limit, n=len(flats))
        return _oracle_sweep(flats, rays, limit, **kw)

    res = trace_sweep(tables, sc.rays, perfomance_limit={"max_trace_num": 40}, tracer=tracer)
    assert seen["limit"] == 40 and seen["n"] == 2 and seen["unit"] == sc.rays[0].unit
    assert res.n == len(sc.rays)
    assert [int(v) for v in res.rows(1)["hit_root"].unique()] == [0]


def _flats(tables):
    return [FlatScene(t.components, t.monitors) for t in tables]


def test_mismatched_node_count_is_rejected():
    a = scenes.Scene([ob.Mirror([0, 0, 0])], [], [])
    b = scenes.Scene([ob.Mirror([0, 0, 0]), ob.Mirror([5, 0, 0])], [], [])
    with pytest.raises(ValueError, match=r"table 1 does not have the topology of table 0 \(n_nodes 2 != 1\)"):
        trace_sweep([a, b], RayBundle.collimated_disc(4), tracer=_oracle_sweep)
    with pytest.raises(ValueError, match=r"table 2 does not have the topology"):
        check_topology(_flats([a, a, b]))


def test_swapped_component_kind_is_rejected():
    a = scenes.Scene([ob.Mirror([0, 0, 0]), ob.Lens([5, 0, 0], focal_length=10)], [], [])
    b = scenes.Scene([ob.Mirror([0, 0, 0]), ob.Block([5, 0, 0])], [], [])
    with pytest.raises(ValueError, match=r"table 1 .*node 1: (interaction kind|geometry kind)"):
        check_topology(_flats([a, b]))


def test_different_material_kind_is_rejected():
    mk = lambda n2: scenes.Scene([ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=ob.Vacuum(), n2=n2)], [], [])
    check_topology(_flats([mk(ob.Glass_NBK7()), mk(ob.Glass_NSF5())]))     # Sellmeier coefficients may differ
    with pytest.raises(ValueError, match=r"table 1 .*material \d+: kind"):
        check_topology(_flats([mk(ob.Glass_NBK7()), mk(1.5)]))


def test_ortho_only_difference_is_accepted():
    f0, f1 = _flats(_grid()[:2])
    f1.node_i[:, A.NI_ORTHO] = 1 - f1.node_i[:, A.NI_ORTHO]
    check_topology([f0, f1])
    f1.node_i[0, A.NI_LEAF] += 1
    with pytest.raises(ValueError, match="leaf index"):
        check_topology([f0, f1])


def test_header_declares_the_sweep_entry_point_and_stays_c99():
    import subprocess

    src = open(os.path.join(ROOT, "include", "optb.h")).read()
    assert "optb_scene_upload_sweep" in A.EXPORTED_SYMBOLS
    proto = re.search(r"int optb_scene_upload_sweep\(([^)]*)\);", src).group(1)
    assert [p.split()[-1].lstrip("*") for p in proto.split(",")] == ["ctx", "descs", "n_configs", "out"]
    assert "const optb_scene_desc* descs" in proto and "int32_t n_configs" in proto
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-x", "c",
                    os.path.join(ROOT, "include", "optb.h")], check=True)
    import ctypes as C

    from optable_b200 import backend

    assert backend.lib().optb_scene_upload_sweep.argtypes == [C.c_void_p, C.POINTER(A.SceneDesc), C.c_int32,
                                                              C.POINTER(C.c_void_p)]
