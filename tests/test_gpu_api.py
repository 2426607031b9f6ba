"""GPU: the object-level API (OpticalTable.ray_tracing with Ray objects, Monitor accessors, interact counts)
against the reference's results in tests/golden/."""
import math

import numpy as np
import pytest

import optable_b200 as ob
from optable_b200 import _abi as A
from tests import golden_io, parity, scenes

pytestmark = pytest.mark.gpu


def _objects_to_arrays(segs, roots):
    index = {id(r): k for k, r in enumerate(roots)}
    out = {
        "seg_o": np.array([s.origin for s in segs], float).reshape(-1, 3),
        "seg_d": np.array([s.direction for s in segs], float).reshape(-1, 3),
        "seg_length": np.array([math.inf if s.length is None else s.length for s in segs], float),
        "seg_alive": np.array([bool(s.alive) for s in segs]),
        "seg_intensity": np.array([s.intensity for s in segs], float),
        "seg_wavelength": np.array([s.wavelength for s in segs], float),
        "seg_q": np.array([0j if s.qo is None else s.qo for s in segs], complex),
        "seg_hasq": np.array([s.qo is not None for s in segs]),
        "seg_pathlength": np.array([s._pathlength for s in segs], float),
        "seg_n": np.array([s.n for s in segs], float),
    }
    return out


@pytest.mark.parametrize("name", ["gaussian_beam", "chromatic", "doublet", "prism_refl", "caps_binding", "misc_components", "mirror_pair"])
def test_ray_tracing_objects_match_reference(name):
    _, _, _, ref = golden_io.load(name)
    sc = scenes.REGISTRY[name](ob)
    table = ob.OpticalTable()
    table.add_components(sc.components)
    table.add_monitors(sc.monitors)
    before = [(r.origin.copy(), r.direction.copy(), r.alive, r.length) for r in sc.rays]
    returned = table.ray_tracing(sc.rays, perfomance_limit=sc.limit)
    assert len(returned) == len(table.rays) == len(ref["seg_root"])
    got = _objects_to_arrays(table.rays, sc.rays)
    q_rtol = 1e-9
    for k in ("seg_alive", "seg_hasq"):
        np.testing.assert_array_equal(got[k], ref[k])
    for k in ("seg_o", "seg_d"):
        assert parity._rel_vec(ref[k], got[k], 1.0).max() <= 1e-9
    for k in ("seg_length", "seg_intensity", "seg_wavelength", "seg_pathlength", "seg_n"):
        assert parity._rel(ref[k], got[k], 1e-3).max() <= 1e-9, k
    hq = ref["seg_hasq"]
    if hq.any():
        assert (np.abs(ref["seg_q"][hq] - got["seg_q"][hq]) / np.abs(ref["seg_q"][hq])).max() <= q_rtol
    # inputs untouched, ids inherited, copies returned
    for r, (o, d, alive, length) in zip(sc.rays, before):
        assert np.array_equal(r.origin, o) and np.array_equal(r.direction, d) and r.alive == alive and r.length == length
    assert {s._id for s in table.rays} <= {r._id for r in sc.rays}
    assert returned[0] is not table.rays[0]
    # monitors: rows per monitor in (root, pop) order, same as Monitor.record after sequential traces
    for mi, mon in enumerate(table.monitors):
        sel = ref["hit_monitor"] == mi
        assert mon.ndata == int(sel.sum())
        if mon.ndata:
            raw = mon._data_raw
            P = np.array([row[0] for row in raw])
            assert parity._rel_vec(ref["hit_P"][sel], P, 1.0).max() <= 1e-9
            np.testing.assert_allclose([row[2] for row in raw], ref["hit_t"][sel], rtol=1e-9)
            assert all(row[3] is not None for row in raw)
            assert len(mon.get_yList()) == mon.ndata and len(mon.get_tYList(sort="ID")) == mon.ndata
    # interact counts of capped components (SURVEY A.6)
    from optable_b200.flatten import FlatScene, pack_rays

    flat = FlatScene(table.components, table.monitors)
    if flat.n_capslots:
        _, fam_ids, _ = pack_rays(sc.rays)
        for s, comp in enumerate(flat.capslots):
            for f, rid in enumerate(fam_ids):
                assert comp._interact_count.get(rid, 0) == int(ref["cap_counts"][s, f])


def test_second_call_extends_and_bundle_entry():
    sc = scenes.gaussian_beam(ob)
    table = ob.OpticalTable()
    table.add_components(sc.components)
    table.ray_tracing(sc.rays[:2])
    n1 = len(table.rays)
    out = table.ray_tracing(sc.rays[2])      # a single Ray is accepted; self.rays is extended, not replaced
    assert len(table.rays) > n1 and len(out) == len(table.rays)
    from optable_b200.bundle import RayBundle

    sc2 = scenes.telescope_4f(ob, n_rays=0)
    t2 = ob.OpticalTable()
    t2.add_components(sc2.components)
    t2.add_monitors(sc2.monitors)
    res = t2.trace_bundle(RayBundle.collimated_disc(50_000), record_hist=True)
    assert int(res["counters"][1]) == 4 * 50_000 and int(res["hist_y"].sum()) == len(res["hit_monitor"])


def test_abcd_matrix_and_4f_calibration_callers():
    """The callers of ray_tracing the reference ships on OpticalTable (optical_table.py:211-422) on the GPU back
    end: finite-difference ABCD matrices and the symmetric-4f simulate step against the reference's own values.
    The matrices are differences of traced positions divided by 1e-5, so 1e-9 parity of the traces gives ~1e-4
    absolute on the entries; the fixture's entries are O(1) (and O(100) for B)."""
    import os

    z = np.load(os.path.join(golden_io.GOLDEN_DIR, "abcd_4f.npz"))
    lens = scenes.asphere_lens9(ob, [43.17, 0, 0])
    rays = scenes.abcd_rays(ob)
    F1, F2 = z["F"]
    Ms, y, ty = ob.OpticalTable.calibrate_symmetric_4f(lens, rays, F10=F1, F20=F2, optimize=False)
    np.testing.assert_allclose(y, z["yList"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(ty, z["tYList"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(Ms, z["Ms"], rtol=1e-5, atol=2e-4)
    assert Ms.shape == (7, 2, 2) and abs(Ms[3, 0, 0] + 1) < 0.2   # a 4f relay images with magnification about -1
    F = ob.OpticalTable.calibrate_symmetric_4f(lens, rays[2:5], F10=F1, F20=F2, criterion="min_stdtY", optimize=True)
    assert len(F) == 2 and all(np.isfinite(F)) and abs(F[0] - F1) < 5
    # the whole Nelder-Mead calibration (94 cost evaluations x 2 device calls) lands where the reference's does
    F = ob.OpticalTable.calibrate_symmetric_4f(lens, scenes.abcd_rays(ob), F10=F1, F20=F2, criterion="M=-I", optimize=True)
    np.testing.assert_allclose(F, z["F_opt"], rtol=1e-6)


def test_scene_upload_rejects_malformed_tables():
    """The kernels index the tables without bounds checks, so optb_scene_upload validates them."""
    from optable_b200 import _abi as A
    from optable_b200.backend import BackendError, Engine

    engine = Engine.get(0)
    flat, _, _, _ = golden_io.load("dove_prism")
    for col, val in ((A.NI_SKIP, 0), (A.NI_GEOM, 99), (A.NI_MAT1, 1000), (A.NI_AUX, 10 ** 6)):
        bad, _, _, _ = golden_io.load("dove_prism")
        leaf = int(np.nonzero(bad.node_i[:, A.NI_GEOM] == A.G_POLY3D)[0][0])
        bad.node_i[leaf, col] = val
        with pytest.raises(BackendError):
            engine.upload(bad)
    engine.upload(flat).close()


def test_scene_upload_rejects_malformed_csg_programs():
    """Nested composite apertures travel as postfix programs in the aux pool (include/optb.h OPTB_G_CSG, p0 = 2): the
    upload checks that a program is well formed before a kernel ever evaluates it on its bit stack."""
    from optable_b200 import _abi as A
    from optable_b200.backend import BackendError, Engine

    engine = Engine.get(0)
    flat, _, _, _ = golden_io.load("nested_csg")
    leaves = np.nonzero((flat.node_i[:, A.NI_GEOM] == A.G_CSG) & (flat.node_f[:, A.NF_P] == 2.0))[0]
    assert len(leaves) == 3
    off = int(flat.node_i[leaves[0], A.NI_AUX])
    n_tok = int(flat.aux[off])
    assert n_tok == 5 and int(flat.aux[off + 1 + 3 * (n_tok - 1)]) == A.CSG_SUBTRACT   # rect circle rect union subtract
    for where, val in ((off, 4.0),                      # one token short: two values left on the stack
                       (off + 1 + 3 * 2, float(A.CSG_UNION)),   # operator where the third shape was: stack underflow later
                       (off + 1, 99.0),                 # unknown token
                       (off, 1e9)):                     # program runs past the aux pool
        bad, _, _, _ = golden_io.load("nested_csg")
        bad.aux[where] = val
        with pytest.raises(BackendError):
            engine.upload(bad)
    engine.upload(flat).close()


def test_edge_cases_empty_inputs_and_long_chains():
    """Empty ray list, empty table, one ray bouncing 1e5 times in a closed cavity (the ripa example's pop budget)."""
    table = ob.OpticalTable()
    assert table.ray_tracing([]) == [] and table.rays == []
    out = table.ray_tracing([ob.Ray([0, 0, 0], [1, 0, 0])])          # nothing to hit: the ray itself comes back
    assert len(out) == 1 and out[0].alive and out[0].length is None
    sc = scenes.cavity(ob, 0.0, 0.0, gaussian=True)
    t2 = ob.OpticalTable()
    t2.add_components(sc.components)
    segs = t2.ray_tracing(sc.rays, perfomance_limit={"max_trace_num": 1e5})
    assert len(segs) == 100000 and all(s.length is not None for s in segs[:10])
    assert segs[-1].intensity == 0.0 or segs[-1].intensity < 1e-300   # 0.9^1e5 underflows, no cutoff in the reference
    L = 10 * 4 / 3
    assert segs[-1]._pathlength == pytest.approx(99999 * L - 2, rel=1e-9)


def test_monitor_record_explicit_segments():
    """Monitor.record(list) through the device (empty scene, one pop per ray) against the oracle's rows."""
    from optable_b200.flatten import FlatScene, pack_rays
    from oracle import oracle as O

    rng = np.random.default_rng(11)
    mon = ob.Monitor(origin=[5, 0.2, -0.1], width=2, height=1.5).RotZ(0.3).RotY(-0.2)
    rays = []
    for k in range(500):
        d = [1.0 if k % 7 else -1.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)]
        kw = {"length": float(rng.uniform(2.0, 9.0))} if k % 3 == 0 else {}
        rays.append(ob.Ray(rng.uniform(-1, 1, 3), d, wavelength=780e-7, alive=bool(k % 5), w0=0.01 if k % 2 else None, **kw))
    mon.record(rays)
    arrs, fam, unit = pack_rays(rays)
    want = O.trace(FlatScene([], [mon]), arrs, max_trace_num=1, unit=unit, n_families=len(fam))
    order = np.argsort(want["hit_root"], kind="stable")
    assert mon.ndata == len(order) > 50
    got_rays = [r for (_, _, _, r) in mon._data_raw]
    assert [rays.index(r) for r in got_rays[:20]] == want["hit_root"][order][:20].tolist()
    np.testing.assert_allclose(mon._P, np.stack([want["hit_px"], want["hit_py"], want["hit_pz"]], 1)[order], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(mon._t, want["hit_t"][order], rtol=1e-9)
    mon.record([])
    assert mon.ndata == len(order)


def test_ripa2_example_with_its_analysis():
    """examples/ripa_gen2_2nd_simplified.py end to end on the new back end: scene held by a ComponentGroup, trace,
    then the script's own analysis (monitor rows looked up by ray id, ray-ray intersections, beam helpers) against
    what the reference computes for it (tests/golden/ripa2_post.npz)."""
    import os

    sc = scenes.ripa2_simplified(ob)
    table = ob.OpticalTable()
    table.add_components(sc.components)
    table.add_monitors(sc.monitors)
    table.ray_tracing(sc.rays)
    got = scenes.ripa2_postprocess(ob, table, sc)
    want = np.load(os.path.join(golden_io.GOLDEN_DIR, "ripa2_post.npz"))
    assert got["P"].shape == want["P"].shape == (8, 3)
    np.testing.assert_allclose(got["P"], want["P"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(got["n"], want["n"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(got["pathlength"], want["pathlength"], rtol=1e-9)
    np.testing.assert_allclose(got["roc"], want["roc"], rtol=1e-5)   # q behind finite-difference asphere curvatures


def test_device_monitor_analytics_match_host_monitor(tmp_path):
    """optable_b200.analytics.DeviceMonitor (rows stay in HBM) against the host Monitor fed the same rows."""
    import torch

    from optable_b200.analytics import DeviceMonitor
    from optable_b200.bundle import RayBundle

    sc = scenes.telescope_4f(ob)
    table = ob.OpticalTable()
    table.add_components(sc.components)
    table.add_monitors(sc.monitors)
    bundle = RayBundle.collimated_disc(20000, radius=2.0)
    out = table.trace_bundle(bundle, record_hist=True)
    for m, mon in enumerate(table.monitors):
        dm = DeviceMonitor(mon, out, m)
        sel = (out["hit_monitor"] == m).cpu().numpy()
        h = {k: out[k].cpu().numpy()[sel] for k in out if k.startswith("hit_")}
        host = ob.Monitor(origin=mon.origin, width=mon.width, height=mon.height)
        host.transform_matrix = mon.transform_matrix
        host._extend(np.stack([h["hit_px"], h["hit_py"], h["hit_pz"]], 1), h["hit_intensity"], h["hit_t"],
                     np.stack([h["hit_dx"], h["hit_dy"], h["hit_dz"]], 1), h["hit_q_re"] + 1j * h["hit_q_im"],
                     h["hit_root"].astype(np.int64).tolist())
        assert dm.ndata == host.ndata > 1000
        for name in ("get_yList", "get_zList", "get_tYList", "get_tZList", "get_IList", "get_tList"):
            for sort in ("YZ", "ID"):
                np.testing.assert_allclose(getattr(dm, name)(sort=sort).cpu().numpy(), getattr(host, name)(sort=sort), rtol=1e-14,
                                           atol=1e-16, err_msg=f"{name}/{sort}")
        np.testing.assert_allclose(dm.get_waist_distance().cpu().numpy(), host.get_waist_distance(), rtol=1e-14)
        assert float(dm.sum_intensity) == pytest.approx(host.sum_intensity, rel=1e-12)
        assert float(dm.std_histy) == pytest.approx(host.std_histy, rel=1e-12)
        counts, _ = host._get_hist_y()
        np.testing.assert_array_equal(dm._get_hist_y()[0], counts)           # the statistics kernels' own binning
        np.testing.assert_array_equal(out["hist_y"][m].cpu().numpy(), counts)  # = the histogram the trace accumulated
        y, z = dm.get_yList(sort=None).cpu().numpy(), dm.get_zList(sort=None).cpu().numpy()
        hw, hh = float(mon.width) / 2, float(mon.height) / 2
        want2 = np.histogram2d(y, z, 30, [[-hw, hw], [-hh, hh]])[0].astype(np.int64)
        np.testing.assert_array_equal(out["hist_yz"][m].cpu().numpy(), want2)
        dy, dz = dm.get_delta_pos()
        hy, hz = host.get_delta_pos()
        np.testing.assert_allclose(dy.cpu().numpy(), hy, rtol=0, atol=1e-15)
        dm.export_rays_npz(str(tmp_path / f"m{m}.npz"))
        host.export_rays_npz(str(tmp_path / f"h{m}.npz"))
        a, b = np.load(tmp_path / f"m{m}.npz"), np.load(tmp_path / f"h{m}.npz")
        for k in b.files:
            np.testing.assert_allclose(a[k], b[k], rtol=1e-14, atol=1e-16)


def test_bench_line_contract_small():
    """bench.py end to end on a small bundle: one JSON line carrying every key of the contract."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    run = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--rays", "200000", "--steps", "3", "--warmup", "3",
                          "--e2e-steps", "1", "--cpu-rays", "500", "--flag-rays", "20000"], capture_output=True, text=True, cwd=root, timeout=900)
    assert run.returncode == 0, run.stderr[-2000:]
    lines = [l for l in run.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "clocks", "gpu_launches", "e2e", "roofline", "cpu_baseline"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["gpu_launches"] > 0 and d["value"] > 1e8
    assert d["e2e"]["value"] > 1e7 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and 0 < d["roofline"]["frac"] < 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert d["config"]["interactions_per_step_per_gpu"] == 4 * 200000
    # the other BASELINE configs ride in the same line, each with its own device value, e2e, roofline and CPU baseline
    assert set(d["workloads"]) == {"c3_doublets_16wl", "c4_cavity_4000", "c5_ripa_64"}
    for name, w in d["workloads"].items():
        assert w["value"] > 1e8 and w["e2e"]["value"] > 1e6 and 0 < w["roofline"]["frac"] < 1.5, name
        assert w["cpu_baseline"]["value"] > 0 and w["config"]["rays_per_gpu"] == 200000, name
    assert d["workloads"]["c4_cavity_4000"]["config"]["interactions_per_step_per_gpu"] == 4001 * 200000
    assert d["roofline_hbm"]["frac"] < 1 and d["roofline"]["bound"] == "fp64" and d["fp64_peak"]["tflops"] > 10


def test_component_interact_single_pop_on_device():
    """`component.interact(ray)`: one pop against one component/group on the device, against the oracle engine."""
    from tests.test_install_cpu import OracleEngine

    hits = 0
    for name in ("misc_components", "prism_refl", "doublet"):
        a, b = scenes.REGISTRY[name](ob), scenes.REGISTRY[name](ob)
        for ca, cb in zip(a.components, b.components):
            for ra, rb in list(zip(a.rays, b.rays))[:5]:
                tw, rw = ca.interact(ra, engine=OracleEngine())
                tg, rg = cb.interact(rb)
                assert (tw is None) == (tg is None)
                if tw is None:
                    continue
                hits += 1
                assert tg == pytest.approx(tw, rel=1e-9) and len(rg) == len(rw)
                for x, y in zip(rw, rg):
                    np.testing.assert_allclose(y.origin, x.origin, rtol=1e-9, atol=1e-12)
                    np.testing.assert_allclose(y.direction, x.direction, rtol=1e-9, atol=1e-12)
                    assert y.alive == x.alive and y.intensity == pytest.approx(x.intensity, rel=1e-9, abs=1e-300)
                    assert y.length == x.length or y.length == pytest.approx(x.length, rel=1e-9)
    assert hits > 10


@pytest.mark.parametrize("name", ["doublet", "telescope_4f", "callable_material", "ripa2_simplified"])
def test_device_monitor_analytics_match_reference_monitor_methods(name):
    """f2: optable_b200.analytics.DeviceMonitor (optb_monitor_stats_grouped over rows that stay in HBM) against
    what the REFERENCE's own Monitor methods returned after the reference's own trace (monitor.py:78-253; fixture
    tests/golden/monitor_analytics.npz, made by oracle/make_golden.py analytics)."""
    import os

    from optable_b200.analytics import DeviceMonitor
    from optable_b200.bundle import RayBundle
    from optable_b200.flatten import pack_rays

    z = np.load(os.path.join(golden_io.GOLDEN_DIR, "monitor_analytics.npz"))
    sc = scenes.REGISTRY[name](ob)
    table = ob.OpticalTable()
    table.add_components(sc.components)
    table.add_monitors(sc.monitors)
    arrs, fam_ids, unit = pack_rays(sc.rays)
    bundle = RayBundle({k: arrs[k] for k in A.RAY_F64}, len(sc.rays))
    out = table.trace_bundle(bundle, sc.limit)
    checked = 0
    q_tol = parity.Q_RTOL_FD * 5 if name in ("telescope_4f", "ripa2_simplified") else 1e-9   # Re(q) behind FD-curvature aspheres (SURVEY A.11); the real part alone can be much smaller than |q|
    for m, mon in enumerate(table.monitors):
        pre = f"{name}__{m}__"
        if pre + "yList" not in z.files:
            continue
        dm = DeviceMonitor(mon, out, m)
        assert dm.ndata == len(z[pre + "yList"]) == dm.stats()["count"], (dm.ndata, len(z[pre + "yList"]), dm.stats()["count"], out["counters"])
        host = lambda t: t.cpu().numpy()
        np.testing.assert_allclose(host(dm.get_yList()), z[pre + "yList"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(host(dm.get_zList()), z[pre + "zList"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(host(dm.get_tYList()), z[pre + "tYList"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(host(dm.get_tZList()), z[pre + "tZList"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(host(dm.get_IList()), z[pre + "IList"], rtol=1e-9)
        np.testing.assert_allclose(host(dm.get_tList()), z[pre + "tList"], rtol=1e-9)
        np.testing.assert_allclose(host(dm.get_waist_distance()), z[pre + "waist_distance"], rtol=q_tol, atol=1e-9)
        counts, edges = dm._get_hist_y()
        np.testing.assert_array_equal(counts, z[pre + "hist_counts"])
        np.testing.assert_allclose(edges, z[pre + "hist_edges"], rtol=0, atol=1e-15)
        if np.isfinite(z[pre + "std_histy"]):
            assert dm.std_histy == pytest.approx(float(z[pre + "std_histy"]), rel=1e-12)
        dy, dz = dm.get_delta_pos()
        np.testing.assert_allclose(host(dy), z[pre + "delta_y"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(host(dz), z[pre + "delta_z"], rtol=1e-9, atol=1e-12)
        assert dm.sum_intensity == pytest.approx(float(z[pre + "sum_intensity"]), rel=1e-12)
        assert dm.avg_intensity == pytest.approx(float(z[pre + "avg_intensity"]), rel=1e-12)
        st = dm.stats()
        assert st["min_y"] == pytest.approx(z[pre + "yList"].min(), rel=1e-9, abs=1e-12)
        assert st["mean_y"] == pytest.approx(z[pre + "yList"].mean(), rel=1e-9, abs=1e-12)
        checked += 1
    assert checked >= 1


def test_gui_loop_refresh_update_nodes_and_graph_replay():
    """f3 (optable/interact.py:455-457: one slider event = the scene with ONE component moved, traced again): the moved
    component is re-read in place (FlatScene.refresh), its rows go to the device copy of the scene
    (optb_scene_update_nodes) and the captured CUDA graph of the trace is replayed. Every replay must equal a trace
    of a freshly flattened, freshly uploaded scene."""
    import torch

    from optable_b200.backend import Engine
    from optable_b200.bundle import DeviceTrace, RayBundle
    from optable_b200.flatten import FlatScene

    engine = Engine.get(0)
    sc = scenes.telescope_4f(ob, n_rays=0)
    n = 50_000
    rays = RayBundle.collimated_disc(n, radius=2.5).to_torch(device="cuda:0")
    flat = FlatScene(sc.components, sc.monitors)
    live = DeviceTrace(engine, flat, n, 2 * n + 64, record_hist=True)
    live.capture(rays)
    lens2 = sc.components[1]
    for step in range(4):
        lens2.TX(0.05).RotZ(2e-3)
        changed = flat.refresh(lens2)
        assert changed is not None and len(changed) == 3
        live.scene.update_nodes(changed)
        live.replay()
        fresh = DeviceTrace(engine, FlatScene(sc.components, sc.monitors), n, 2 * n + 64, record_hist=True)
        fresh.run(rays)
        a, b = live.counters(), fresh.counters()
        assert a[A.C_STATUS] == 0 and list(a[:5]) == list(b[:5]) and a[A.C_INTERACTIONS] > 3 * n
        assert torch.equal(live.t["hist_yz"], fresh.t["hist_yz"]) and torch.equal(live.t["hist_y"], fresh.t["hist_y"])
        nh = int(a[A.C_HITS])
        for col in ("hit_py", "hit_t", "hit_q_im"):
            assert torch.equal(torch.sort(live.t[col][:nh]).values, torch.sort(fresh.t[col][:nh]).values), col
        fresh.close()
    live.close()


def test_rejected_option_combinations_enqueue_nothing():
    """Option combinations the library refuses fail with -7 and their message before anything is enqueued: the
    caller's counters are left as they were."""
    import re

    import torch

    from optable_b200.backend import BackendError, Engine
    from optable_b200.bundle import DeviceTrace, RayBundle
    from optable_b200.flatten import FlatScene

    engine = Engine.get(0)
    n = 64
    rays = RayBundle.collimated_disc(n, radius=2.5).to_torch(device="cuda:0")
    root_flags = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    sc = scenes.telescope_4f(ob, n_rays=0)
    flat = FlatScene(sc.components, sc.monitors)
    caps = scenes.caps_binding(ob)

    def refused(scene, msg, rays_t=rays, **kw):
        res, t = engine.alloc_result(scene, 0, 0, n * scene.n_configs)
        res.root_flags = root_flags.data_ptr()
        t["counters"].fill_(-1)
        prm = engine.make_params(80, record_segments=False, record_hits=False, n_families=n * scene.n_configs, **kw)
        with pytest.raises(BackendError, match=re.escape(f"liboptb error -7: {msg}")):
            engine.trace_device(scene, rays_t, prm, res)
        torch.cuda.synchronize()
        assert (t["counters"] == -1).all()

    single, sweep, capped = engine.upload(flat), engine.upload_sweep([flat, flat]), engine.upload(FlatScene(caps.components, caps.monitors))
    refused(single, "reference_roots and flag_ambiguity are separate diagnostics modes", reference_roots=True, flag_ambiguity=True)
    sweep_msg = "sweep: flag_ambiguity and reference_roots are not available on sweep scenes"
    refused(sweep, sweep_msg, flag_ambiguity=True)
    refused(sweep, sweep_msg, reference_roots=True)
    refused(sweep, "sweep: rays.family must be NULL (every root is its own family)",
            rays_t=dict(rays, family=torch.arange(n, dtype=torch.int32, device="cuda:0")))
    refused(capped, "flag_ambiguity is not available on the family-serial path (binding interact caps)", flag_ambiguity=True)
    for s in (single, sweep, capped):
        s.close()
    # the graph capture of a flag_ambiguity trace (one host round trip per generation) is refused before it begins
    dt = DeviceTrace(engine, flat, n, 2 * n + 64, flag_ambiguity=True)
    dt.t["counters"].fill_(-1)
    with pytest.raises(NotImplementedError):
        dt.capture(rays)
    assert not torch.cuda.is_current_stream_capturing()
    assert (dt.t["counters"] == -1).all()   # not even the warm-up run
    dt.close()
