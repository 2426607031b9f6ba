"""GPU: sweeps of Ray objects whose interact caps bind run the family-serial sweep kernel. Every configuration of one
`trace_sweep` is bit-identical to `engine.trace_arrays` of that configuration alone from its starting counts: sorted
monitor rows (every column), histograms, summed counters and the final interact counts. `optb_trace_host` gives the
same, the plan reports SERIAL | SWEEP, and the refusals that remain leave the counters untouched."""
import numpy as np
import pytest
import torch

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.flatten import FlatScene, pack_rays
from optable_b200.sweep import initial_counts, trace_sweep
from tests import scenes

pytestmark = pytest.mark.gpu

HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64
SUMMED = (A.C_SEGMENTS, A.C_INTERACTIONS, A.C_HITS, A.C_DROPPED)


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _prism(refl, tilt, cap=3, extra=()):
    """tests.scenes.caps_binding (24 rays, 6 wavelengths per id) with reflectivity, tilt and caps varied."""
    sc = scenes.caps_binding(ob)
    ps = ob.TriangularPrism(origin=[0, 0, 0], width=6, height=6, n1=1, n2=ob.Glass_NBK7(), alpha=np.pi / 4,
                            beta=np.pi / 2, reflectivity_1=refl, reflectivity_2=0.5, reflectivity_3=0.4,
                            max_interact_count_2=cap, max_interact_count_3=cap).RotZ(tilt)
    return scenes.Scene([ps, *extra], sc.rays, sc.monitors + [m for m in extra if isinstance(m, ob.Monitor)])


def _seed(tables, fam_ids):
    for k, t in enumerate(tables):
        for s, comp in enumerate(FlatScene(t.components, t.monitors).capslots):
            comp._interact_count = {rid: (f + s + k) % 3 for f, rid in enumerate(fam_ids) if (f + k) % 2 == 0}


def _check(engine, tables, rays, limit):
    """trace_sweep == one trace_arrays per configuration from its starting counts, bit for bit."""
    arrs, fam_ids, unit = pack_rays(rays)
    F = len(fam_ids)
    res = trace_sweep(tables, rays, {"max_trace_num": limit}, record_hist=True, engine=engine)
    sums = np.zeros(A.C_COUNT, np.int64)
    for k, t in enumerate(tables):
        flat = FlatScene(t.components, t.monitors)
        caps0 = initial_counts([flat.capslots], fam_ids)
        scene = engine.upload(flat)
        want = engine.trace_arrays(scene, arrs, max_trace_num=limit, unit=unit, record_segments=False, record_hist=True,
                                   n_families=F, cap_counts=caps0)
        scene.close()
        got = {c: v.cpu().numpy() for c, v in res.rows(k).items()}
        assert len(got["hit_root"]) == len(want["hit_root"]) > 0, f"config {k}: rows"
        for c in HIT_COLS:
            assert np.array_equal(got[c].view(np.uint8), np.ascontiguousarray(want[c]).view(np.uint8)), f"config {k}: {c}"
        m = len(t.monitors)
        assert np.array_equal(got["hist_y"], want["hist_y"][:m]) and np.array_equal(got["hist_yz"], want["hist_yz"][:m])
        np.testing.assert_array_equal(res.interact_counts[k], want["cap_counts"], err_msg=f"config {k}: counts")
        sums += np.asarray(want["counters"], np.int64)
    for c in SUMMED:
        assert int(res.counters[c]) == int(sums[c]), c
    assert int(res.counters[A.C_STATUS]) == 0
    return res


def test_prism_grid_with_starting_counts(engine):
    tables = [_prism(r, t) for r, t in ((0.3, 0.0), (0.2, 0.03), (0.45, -0.05))]   # K N = 72: warps straddle
    _, fam_ids, _ = pack_rays(tables[0].rays)
    _seed(tables, fam_ids)
    res = _check(engine, tables, tables[0].rays, 80)
    assert res.interact_counts.max() >= 3


def test_shared_ids_bind_beyond_one_root(engine):
    # caps of 100 against 80 pops: only the 6 rays that share an id can reach them, as in ray_tracing
    tables = [_prism(0.3, t, cap=100) for t in (0.0, 0.02, -0.01)]
    res = _check(engine, tables, tables[0].rays, 80)
    assert res.interact_counts.max() > 80


def test_non_splitting_cavity_with_distinct_ids(engine):
    def cavity(tilt):
        a = ob.Mirror([-2, 0, 0], radius=3, reflectivity=1, transmission=0, max_interact_count=7).RotZ(tilt)
        b = ob.Mirror([2, 0, 0], radius=3, reflectivity=1, transmission=0).RotZ(np.pi)
        return scenes.Scene([a, b], [], [ob.Monitor([0, 0, 0], 8, 8)])

    rays = [ob.Ray([0, 0.1 * i - 1.0, 0], [1, 0.01 * (i % 5), 0], wavelength=780e-7, w0=61e-4, id=i) for i in range(37)]
    tables = [cavity(t) for t in (0.0, 0.001, -0.002)]
    assert max(FlatScene(t.components, t.monitors).max_children for t in tables) == 1
    _check(engine, tables, rays, 60)


def test_pass_through_leaf(engine):
    screen = lambda: ob.Monitor([4.5, 3, 0], 6, 6)
    tables = [_prism(r, 0.0, extra=(screen(),)) for r in (0.3, 0.25)]
    assert FlatScene(tables[0].components, tables[0].monitors).has_pass
    _check(engine, tables, tables[0].rays, 80)


def test_plan_and_host_trace(engine):
    from tests.test_gpu_trace_host import host_trace, sorted_params

    tables = [_prism(r, t) for r, t in ((0.3, 0.0), (0.2, 0.03))]
    rays = tables[0].rays
    arrs, fam_ids, unit = pack_rays(rays)
    _seed(tables, fam_ids)
    K, n, F, limit = len(tables), len(arrs["ox"]), len(fam_ids), 80
    flats = [FlatScene(t.components, t.monitors) for t in tables]
    caps0 = initial_counts([f.capslots for f in flats], fam_ids)
    scene = engine.upload_sweep(flats)
    bits = engine.trace_plan(scene, arrs, max_trace_num=limit, unit=unit)["bits"]
    assert bits & A.PLAN_SERIAL and bits & A.PLAN_SWEEP
    res = trace_sweep(tables, rays, {"max_trace_num": limit}, record_hist=True, engine=engine)
    prm = sorted_params(engine.make_params(limit, unit, record_segments=False, record_hist=True, n_families=F))
    got = host_trace(engine, scene, arrs, prm, 1, K * n * limit, n_hist=K * len(tables[0].monitors), cap_counts=caps0)
    for c in HIT_COLS:
        want = res.hits[c].cpu().numpy()
        assert np.array_equal(np.asarray(got[c]).view(np.uint8), want.view(np.uint8)), c
    np.testing.assert_array_equal(got["hist_y"].reshape(res.hist_y.shape), res.hist_y.cpu().numpy())
    np.testing.assert_array_equal(got["cap_counts"].reshape(-1, K, F).transpose(1, 0, 2), res.interact_counts)
    for c in SUMMED:
        assert int(got["counters"][c]) == int(res.counters[c]), c
    scene.close()


def test_remaining_refusals_leave_the_counters(engine):
    from optable_b200.backend import BackendError

    tables = [_prism(0.3, t) for t in (0.0, 0.02)]
    arrs, fam_ids, unit = pack_rays(tables[0].rays)
    scene = engine.upload_sweep([FlatScene(t.components, t.monitors) for t in tables])
    rays_t = engine.rays_to_device(arrs)
    n, F = len(arrs["ox"]), len(fam_ids)

    def refused(pattern, rays, **kw):
        res, t = engine.alloc_result(scene, 0, 64, 2 * max(n, F))
        t["counters"].fill_(-1)
        prm = engine.make_params(80, unit, record_segments=False, **kw)
        with pytest.raises(BackendError, match=pattern):
            engine.trace_device(scene, rays, prm, res)
        torch.cuda.synchronize()
        assert (t["counters"] == -1).all()

    no_family = {k: v for k, v in rays_t.items() if k != "family"}
    refused(r"-7.*caps_slack.*rays\.family", no_family, n_families=2 * n)
    refused(r"-7.*flag_ambiguity and reference_roots", rays_t, n_families=F, flag_ambiguity=True)
    refused(r"-7.*flag_ambiguity and reference_roots", rays_t, n_families=F, reference_roots=True)
    refused(r"-7.*rays\.family must be NULL", rays_t, n_families=F, caps_slack=1)
    scene.close()
