"""GPU: the CUDA path against the C oracle on seeded batches far larger than the golden fixtures (sizes the oracle
finishes in seconds), one scene per BASELINE.json config family, plus size-independent properties at full size."""
import numpy as np
import pytest

from tests import parity, scenes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _both(engine, sc, arrs, limit=2000, q_rtol=parity.RTOL, nthreads=8, **kw):
    from optable_b200.flatten import FlatScene
    from oracle import oracle as O
    from oracle import ref_harness as RH

    flat = FlatScene(sc.components, sc.monitors)
    scene = engine.upload(flat)
    got = engine.trace_arrays(scene, arrs, max_trace_num=limit, **kw)
    want = O.trace(flat, arrs, max_trace_num=limit, nthreads=nthreads if not flat.n_capslots else 1)
    errs = parity.compare(RH.arrays_from_result(want), RH.arrays_from_result(got), q_rtol=q_rtol, label="scale")
    for c in (1, 2, 4):  # interactions, monitor rows, dropped
        assert int(got["counters"][c]) == int(want["counters"][c]), c
    # OPTB_C_TESTS is a work counter, not a result. The engine may do LESS work than the reference's loop (a box
    # entered beyond the closest hit so far dismisses its subtree: DESIGN.md, front-to-back dismissal), never more --
    # up to the last bit of a child ray's origin: it starts ON the surface it left, so whether that surface's
    # zero-thickness box is entered at t = +-1 ulp (leaf test attempted, then rejected by t >= 1e-9) is a coin flip.
    assert int(got["counters"][3]) <= 1.05 * int(want["counters"][3])
    return got, errs


def test_c2_4f_asphere_200k(engine):
    import optable_b200 as ob
    from optable_b200.bundle import RayBundle

    sc = scenes.telescope_4f(ob, n_rays=0)
    arrs = RayBundle.collimated_disc(200_000, start=12345).materialise()
    got, errs = _both(engine, sc, arrs, q_rtol=parity.Q_RTOL_FD)
    assert int(got["counters"][1]) == 4 * 200_000


def test_c3_doublets_16_wavelengths(engine):
    import optable_b200 as ob

    mk = lambda x: ob.Doublet([x, 0, 0], CT1=1.359, CT2=0.6, R1=18.405, R2=-13.734, R3=-39.933, n12=ob.Glass_NBK7(),
                              n23=ob.Glass_NSF5(), diameter=7.5)
    sc = scenes.Scene([mk(30.3964), mk(90.3964)], [], [ob.Monitor([150, 0, 0], 10, 10)])
    arrs = scenes.ray_arrays(120_000, [0, 0, 0], [0, 2.1, 2.1], [1, 0, 0], [0, 0.004, 0.004],
                             wavelengths=np.linspace(400e-7, 1100e-7, 16))
    got, errs = _both(engine, sc, arrs)
    assert int(got["counters"][1]) > 6 * 100_000


def test_c4_cavity_long_chains(engine):
    import optable_b200 as ob

    sc = scenes.cavity(ob, 0.0, 0.0)
    arrs = scenes.ray_arrays(3000, [2, 0, 0], [0, 1, 1], [1, 0, 0], [0, 1e-5, 1e-5])
    got, errs = _both(engine, sc, arrs, limit=401)
    assert int(got["counters"][1]) == 3000 * 401  # every pop hits a mirror; the cap stops the chain


def test_splitting_scene_with_pop_cap(engine):
    import optable_b200 as ob

    sc = scenes.misc_components(ob)
    arrs = scenes.ray_arrays(20_000, [-3, 0, 0], [0, 15, 0.4], [1, 0, 0], [0, 0.03, 0.03], wavelengths=(633e-7, 500e-7))
    got, errs = _both(engine, sc, arrs, limit=40, max_live=400_000)
    assert int(got["counters"][4]) > 0  # the cap really dropped queued rays


def test_c5_style_nested_mma(engine):
    import optable_b200 as ob

    sc = scenes.mma_small(ob)
    arrs = scenes.ray_arrays(20_000, [0, 0, 0], [0, 0.1, 0.03], [1, 0, 0], [0, 0.02, 0.02])
    _both(engine, sc, arrs, limit=60, max_live=400_000)


def test_full_size_properties_c2(engine):
    """1e7 rays (BASELINE size): every ray refracts exactly 4 times; monitor rows = rays inside the 5x5 windows;
    the device histogram equals np.histogram of the returned rows; intensities unchanged (T = 1)."""
    import torch

    import bench
    from optable_b200 import _abi as A
    from optable_b200.bundle import DeviceTrace

    n = 10_000_000
    flat = bench.build_scene()
    bundle = bench.make_bundle(n, 0)
    dt = DeviceTrace(engine, flat, n, 2 * n, record_hist=True)
    dt.run(bundle.to_torch(device="cuda:0"))
    cnt = dt.counters()
    assert int(cnt[A.C_STATUS]) == 0
    assert int(cnt[A.C_INTERACTIONS]) == 4 * n and int(cnt[A.C_SEGMENTS]) == 5 * n and int(cnt[A.C_DROPPED]) == 0
    nh = int(cnt[A.C_HITS])
    mon = dt.t["hit_monitor"][:nh]
    py = dt.t["hit_py"][:nh]
    pz = dt.t["hit_pz"][:nh]
    oy, oz = torch.from_numpy(bundle.columns["oy"]).cuda(), torch.from_numpy(bundle.columns["oz"]).cuda()
    inside0 = int(((oy.abs() <= 2.5) & (oz.abs() <= 2.5)).sum())
    assert int((mon == 0).sum()) == inside0
    assert bool((dt.t["hit_intensity"][:nh] == 1.0).all())
    assert int(dt.t["hist_y"].sum()) == nh
    for m in (0, 1):
        sel = mon == m
        mf = flat.mon_f[m]
        assert list(mf[A.MON_TY:A.MON_TY + 3]) == [0.0, 1.0, 0.0]   # unrotated: the histogram's y is hit_py itself
        hw = float(mf[A.MON_HW])
        want = np.histogram(py[sel].cpu().numpy(), bins=30, range=(-hw, hw))[0]
        np.testing.assert_array_equal(dt.t["hist_y"][m].cpu().numpy(), want, err_msg=f"monitor {m}")
    # a 4f relay images the input plane inverted: monitor-1 position = -input position within aberrations
    r1 = dt.t["hit_root"][:nh][mon == 1].long()
    assert float((py[mon == 1] + oy[r1]).abs().max()) < 0.05 and float((pz[mon == 1] + oz[r1]).abs().max()) < 0.05


def test_c5_ripa_7689_leaves(engine):
    """The full ripa_gen2_lensless scene (scene tables 2.8 MB: read through L2, not staged in shared memory):
    2,000 jittered rays x 48 pops against the oracle; caps of 1e5 cannot bind -> parallel path."""
    import optable_b200 as ob

    sc = scenes.ripa(ob, n_rays=0)
    p = sc.params
    arrs = scenes.ray_arrays(2000, p["origin"], [0, p["R1w0"], p["R1w0"]], p["direction"], [0, 1e-3, 1e-3],
                             wavelengths=(p["wavelength"],), w0=p["R1w0"])
    got, _ = _both(engine, sc, arrs, limit=48, max_live=200_000)
    assert int(got["counters"][1]) > 40 * 2000


def test_pipelined_host_trace_equals_device_trace(engine):
    """optb_trace_host switches to the chunked three-stream pipeline above 3 Mi rays: same rows (as a set, keyed by
    (root, monitor)), same histograms, same counters (but launches and generations) as one device-resident launch."""
    import torch

    import bench
    from optable_b200 import _abi as A
    from optable_b200.bundle import DeviceTrace
    from optable_b200.flatten import rays_struct

    n = 3_300_000
    flat = bench.build_scene()
    bundle = bench.make_bundle(n, 777)
    dt = DeviceTrace(engine, flat, n, 2 * n, record_hist=True)
    dt.run(bundle.to_torch(device="cuda:0"))
    cnt = dt.counters()
    nh = int(cnt[A.C_HITS])
    host = {k: v.numpy() for k, v in bundle.to_torch(pin=True).items()}
    host["length"] = None
    rs = rays_struct({**{k: None for k in A.RAY_F64}, **host})
    res = A.Result()
    res.seg_capacity, res.hit_capacity = 0, 2 * n
    out = {}
    for k in dt.hit_columns:
        out[k] = torch.empty(2 * n, dtype=dt.t[k].dtype).pin_memory()
        setattr(res, k, out[k].data_ptr())
    hy, hyz = torch.zeros(2, 30, dtype=torch.int64).pin_memory(), torch.zeros(2, 30, 30, dtype=torch.int64).pin_memory()
    hc = torch.zeros(A.C_COUNT, dtype=torch.int64).pin_memory()
    res.hist_y, res.hist_yz, res.counters = hy.data_ptr(), hyz.data_ptr(), hc.data_ptr()
    engine.trace_host(dt.scene, rs, dt.prm, res)
    assert int(hc[A.C_STATUS]) == 0
    for c in range(A.C_COUNT):  # chunk counters add up (status: OR); launches and generations count per chunk
        if c not in (A.C_LAUNCHES, A.C_GENERATIONS):
            assert int(hc[c]) == int(cnt[c]), c
    assert torch.equal(hy, dt.t["hist_y"].cpu()) and torch.equal(hyz, dt.t["hist_yz"].cpu())

    def keyed(cols, rows):
        key = cols["hit_root"][:rows].to(torch.int64) * 4 + cols["hit_monitor"][:rows].to(torch.int64)
        order = torch.argsort(key)
        return key[order], {k: v[:rows][order] for k, v in cols.items()}

    ka, a = keyed({k: v.cpu() for k, v in dt.t.items() if k in dt.hit_columns}, nh)
    kb, b = keyed(out, nh)
    assert torch.equal(ka, kb)
    for k in dt.hit_columns:
        assert torch.equal(a[k], b[k]), k


def test_one_ray_whose_generation_outgrows_64_live_rays(engine):
    """ADVICE r1: the wavefront capacity used to be clamped to 64x the batch, so ONE initial ray through a stack of
    partial mirrors (every pop queues two rays) overflowed the workspace although the reference traces it to its
    2000-pop cap. The capacity now follows the workspace and `trace_arrays` grows it on overflow."""
    import optable_b200 as ob

    comps = [ob.Mirror([float(x), 0, 0], radius=3, reflectivity=0.6, transmission=0.4).RotZ(0.002 * k)
             for k, x in enumerate(range(0, 16, 2))]
    sc = scenes.Scene(comps, [], [ob.Monitor([20, 0, 0], 8, 8)])
    arrs = scenes.ray_arrays(1, [-1, 0.01, 0.02], [0, 0, 0], [1, 0, 0], [0, 0, 0])
    got, errs = _both(engine, sc, arrs, limit=2000, nthreads=1)
    assert len(got["seg_root"]) == 2000 and int(got["counters"][4]) > 64  # the pop cap bound with > 64 rays still queued
    # same through the object API (trace_table has no max_live knob: it must grow on its own)
    table = ob.OpticalTable()
    table.add_components(comps)
    ray = ob.Ray([-1, 0.01, 0.02], [1, 0, 0], wavelength=780e-7, w0=61e-4)
    assert len(table.ray_tracing(ray)) == 2000


@pytest.mark.parametrize("case", ["mma_oblique", "mla_dmd", "ripa", "mma_small"])
def test_lattice_window_walk_equals_reference_walk(engine, case, monkeypatch):
    """OPTB_G_GRID groups (flatten._grid): the device lists the children inside the ray's lattice window instead of
    descending the box hierarchy. The oracle ignores the descriptor and box-tests every child like the reference
    (component_group.py:104-115): same segments, same monitor rows, same leaf-test count. Rays come from all
    directions, including nearly in-plane ones (window refused -> hierarchy) and axis-parallel ones (parallel-axis
    branch of the slab test -> hierarchy)."""
    import optable_b200 as ob
    from optable_b200 import _abi as A
    from optable_b200.flatten import FlatScene

    monkeypatch.setattr(FlatScene, "GRID_MIN_CHILDREN", 6)
    rng = np.random.default_rng(11)
    if case == "mma_oblique":
        mma = ob.MMA(origin=[5, 0, 0], N=(12, 9), pitch=0.3, roc=2.0, n=1.5, thickness=0.2, reflectivity=0.9,
                     transmission=0.1, shifty_z=0.02).RotZ(0.3).RotY(-0.2)
        sc = scenes.Scene([mma, ob.Mirror([-3, 0, 0], radius=6)], [], [ob.Monitor([2, 0, 0], 8, 8)])
        n = 30_000
        o = np.column_stack([rng.uniform(-2, 4, n), rng.uniform(-3, 3, n), rng.uniform(-3, 3, n)])
        tgt = np.array([5.0, 0, 0]) + np.column_stack([rng.uniform(-0.3, 0.3, n), rng.uniform(-2.5, 2.5, n), rng.uniform(-2, 2, n)])
        d = tgt - o
        d[: n // 20] = [0.0, 1.0, 0.0]           # axis-parallel rays along the array
        d[n // 20: n // 10, 0] *= 1e-4           # nearly in-plane
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        arrs = scenes.ray_arrays(n, [0, 0, 0], [0, 0, 0], [1, 0, 0], [0, 0, 0])
        for k, ax in enumerate("xyz"):
            arrs["o" + ax], arrs["d" + ax] = np.ascontiguousarray(o[:, k]), np.ascontiguousarray(d[:, k])
        limit = 12
    elif case == "mla_dmd":
        mla = ob.MLA([4, 0, 0], N=(7, 6), pitch=0.5, focal_length=3.0, radius=0.3)
        dmd = ob.DMD([8, 0, 0], N=(8, 8), pitch=0.4, tilt_angle=0.2)
        sc = scenes.Scene([mla, dmd], [], [ob.Monitor([0.5, 0, 0], 6, 6)])
        arrs = scenes.ray_arrays(30_000, [0, 0, 0], [0, 1.6, 1.4], [1, 0, 0], [0, 0.05, 0.05])
        limit = 10
    elif case == "ripa":
        sc = scenes.ripa(ob, n_rays=0)
        import bench

        arrs = bench.make_bundle(20_000, 0, "c5_ripa_64").materialise()
        limit = 40
    else:
        sc = scenes.mma_small(ob)
        arrs = scenes.ray_arrays(20_000, [0, 0, 0], [0, 0.1, 0.03], [1, 0, 0], [0, 0.02, 0.02])
        limit = 60
    flat = FlatScene(sc.components, sc.monitors)
    assert (flat.node_i[:, A.NI_GEOM] == A.G_GRID).any(), "the scene was meant to contain a lattice group"
    got, errs = _both(engine, sc, arrs, limit=limit, max_live=max(40 * len(arrs["ox"]), 1 << 20))
    assert int(got["counters"][A.C_INTERACTIONS]) > len(arrs["ox"]) // 4


def test_ambiguity_flags_in_kernel(engine):
    """SURVEY A.9 on the device (params.flag_ambiguity): rays aimed at an aperture edge, at a shared edge of two
    coplanar mirrors (equal-distance tie), at grazing incidence and at the TIR threshold get their bits; a clean ray
    through the middle of everything gets none; OPTB_C_FLAGGED counts the flagged initial rays."""
    import optable_b200 as ob
    from optable_b200 import _abi as A
    from optable_b200.flatten import FlatScene

    m1 = ob.SquareMirror([5, 0.5, 0], width=1, height=1, reflectivity=1.0)       # y in [0, 1]
    m2 = ob.SquareMirror([5, -0.5, 0], width=1, height=1, reflectivity=1.0)      # y in [-1, 0]: shares the edge y = 0
    slab = ob.SquareRefractive([9, 5, 0], width=2, height=2, n1=1.0, n2=1.5)     # glass on the -x side
    sc = scenes.Scene([m1, m2, slab], [], [])
    crit = np.arcsin(1.0 / 1.5)
    rays = {
        "clean": ([0, 0.4, 0.1], [1, 0, 0]),
        "edge": ([0, 1.0, 0.2], [1, 0, 0]),                       # on the outer edge of m1 -> APERTURE
        "tie_edge": ([0, 0.0, 0.3], [1, 0, 0]),                   # on the edge shared by m1 and m2 -> APERTURE (+ TIE)
        "grazing": ([5 - 2e-8, 0.2, 0.0], [1e-7, 1.0, 0]),        # skims m1 (meets it at y = 0.4) -> GRAZING
        "tir": ([8.0, 5.0, 0.0], [np.cos(crit), np.sin(crit), 0]),  # from inside the glass at the critical angle -> TIR
    }
    names = list(rays)
    arrs = scenes.ray_arrays(len(names), [0, 0, 0], [0, 0, 0], [1, 0, 0], [0, 0, 0])
    for k, nm in enumerate(names):
        o, d = np.array(rays[nm][0], float), np.array(rays[nm][1], float)
        d /= np.linalg.norm(d)
        for j, ax in enumerate("xyz"):
            arrs["o" + ax][k], arrs["d" + ax][k] = o[j], d[j]
    arrs["n_medium"][names.index("tir")] = 1.5
    flat = FlatScene(sc.components, sc.monitors)
    scene = engine.upload(flat)
    out = engine.trace_arrays(scene, arrs, max_trace_num=4, flag_ambiguity=True)
    fl = dict(zip(names, out["root_flags"].tolist()))
    assert fl["clean"] == 0, fl
    assert fl["edge"] & A.AMB_APERTURE and fl["tie_edge"] & A.AMB_APERTURE, fl
    assert fl["grazing"] & A.AMB_GRAZING, fl
    assert fl["tir"] & A.AMB_TIR, fl
    assert int(out["counters"][A.C_FLAGGED]) == sum(1 for v in fl.values() if v)
    # same result with and without the diagnostics pass
    plain = engine.trace_arrays(scene, arrs, max_trace_num=4)
    for k in ("seg_leaf", "seg_length", "seg_ox"):
        np.testing.assert_array_equal(out[k], plain[k])
