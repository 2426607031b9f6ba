"""GPU: every single-scene trace kernel variant, in both table placements, against its twin and the oracle.

A scene's tables are staged in shared memory (the SMEM variants) when its blob fits the opt-in window less the largest
static shared memory of those kernels, and read from global memory otherwise. The fixtures are all small, so the
global-memory variants only ran on thousand-leaf scenes. Here any scene is forced to global tables by padding its
aux pool with zeros: nothing reads past the offsets the nodes reference, so the results must not change, and the blob
grows in steps of 16 bytes. optb_trace_plan (Engine.trace_plan) tells which variant a trace runs, so every case can
assert that it ran the variant it claims to.

  * the variant matrix: 12 parallel kinds (box mode x aspheres x split) and 5 general kinds (reference roots with and
    without the family-serial path, the ambiguity mask, family-serial, pass-through leaves), each with its tables in
    shared memory and in global memory: the two are bit-identical and both match the oracle;
  * histograms through global atomics in a non-sweep trace (blob + histograms over the window; more than 64 KiB of
    histograms) against the same monitors' shared-memory histograms and numpy;
  * blobs at the edges of the shared-memory plan: one to seven 32 KiB bulk copies, and the top of the opt-in window.
"""
import numpy as np
import pytest

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200.bundle import RayBundle
from optable_b200.flatten import FlatScene
from optable_b200.workloads import asphere_lens9, telescope_4f_grid
from tests import hist_cases as H
from tests import parity, scenes
from tests.test_gpu_trace_host import host_trace, sorted_params

pytestmark = pytest.mark.gpu

SEG_COLS = A.SEG_F64 + A.SEG_U32 + A.SEG_I32
HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64
# OPTB_C_TESTS is a work counter: the only result-independent slot the twins may disagree on
SAME_COUNTERS = [c for c in range(A.C_COUNT) if c != A.C_TESTS]
GLOBAL_BLOB = 256 << 10   # above the opt-in window of any device: tables in global memory
OBSERVED = {}             # plan bits (without HIST_SMEM) -> case that ran them


@pytest.fixture(scope="module")
def engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


# ---- blob layout and padding --------------------------------------------------------------------------------------
def _a16(x):
    return (x + 15) // 16 * 16


def blob_bytes(flat):
    """Bytes of the scene blob optb_scene_upload builds (optb.cu blob_layout)."""
    n = flat.n_nodes
    parts = [max(n, 1) * 64, n * A.NF_STRIDE * 8, n * A.NI_STRIDE * 4, flat.n_materials * 4, flat.n_materials * A.MF_STRIDE * 8,
             max(flat.n_monitors, 1) * (A.MON_STRIDE + 4) * 8, max(flat.aux.size, 1) * 8]
    return sum(_a16(p) for p in parts)


def padded(flat, blob):
    """`flat` with zeros appended to its aux pool so that its blob is exactly `blob` bytes (a multiple of 16)."""
    fixed = blob_bytes(flat) - _a16(max(flat.aux.size, 1) * 8)
    n_aux = (blob - fixed) // 8
    assert blob % 16 == 0 and n_aux >= flat.aux.size, (blob, blob_bytes(flat))
    d = flat.to_arrays()
    d["aux"] = np.concatenate([flat.aux, np.zeros(n_aux - flat.aux.size)])
    out = FlatScene.from_arrays(d)
    assert blob_bytes(out) == blob
    return out


def expect(boxes, asph=False, split=False, serial=False, flag=False, brent=False, passk=False):
    return ((boxes << A.PLAN_BOX_SHIFT) | (A.PLAN_ASPH if asph else 0) | (A.PLAN_SPLIT if split else 0)
            | (A.PLAN_SERIAL if serial else 0) | (A.PLAN_FLAG if flag else 0) | (A.PLAN_BRENT if brent else 0)
            | (A.PLAN_PASSK if passk else 0))


def describe(bits):
    names = [n for n, b in (("SMEM", A.PLAN_SMEM), ("SERIAL", A.PLAN_SERIAL), ("ASPH", A.PLAN_ASPH), ("SPLIT", A.PLAN_SPLIT),
                            ("FLAG", A.PLAN_FLAG), ("BRENT", A.PLAN_BRENT), ("PASSK", A.PLAN_PASSK), ("SWEEP", A.PLAN_SWEEP)) if bits & b]
    return f"box{(bits & A.PLAN_BOX_MASK) >> A.PLAN_BOX_SHIFT}" + "".join("+" + n for n in names)


# ---- scenes -------------------------------------------------------------------------------------------------------
def _flat(sc):
    return FlatScene(sc.components, sc.monitors)


def _no_box_tests(flat):
    """The scene with every box test switched off (box mode 0; groups are then always entered)."""
    d = flat.to_arrays()
    d["node_i"] = flat.node_i.copy()
    d["node_i"][:, A.NI_AABB] = 0
    return FlatScene.from_arrays(d)


def _mma_lattice(ns, extra=()):
    """scenes.mma_small with 8 x 4 lenslet arrays: enough children for a lattice group (flatten.GRID_MIN_CHILDREN)."""
    pitch, roc = 420e-4, 2.2
    m0 = ns.MMA(origin=[-0.1, 0, 0], N=(8, 4), pitch=pitch, roc=roc, n=1.5, thickness=0.1, reflectivity=0.9999,
                transmission=0, back_transmission=0, back_reflectivity=1)
    m1 = ns.MMA(origin=[2.0, 0, 0], N=(8, 4), pitch=pitch, roc=roc, n=1.5, thickness=0.1, reflectivity=0.98,
                transmission=0.3, shifty_z=-0.002).TY(0.01)
    grp = ns.ComponentGroup([0, 0, 0])
    grp.add_components([m0, m1])
    return scenes.Scene([grp, *extra], [], [ns.Monitor([2.0 - 1e-4, 0, 0], width=1, height=1), ns.Monitor([12, 0, 0], 8, 8)])


def _mla_lattice(ns, extra=()):
    mla = ns.MLA([5, 0, 0], N=(8, 4), pitch=0.5, focal_length=4.0, radius=0.25)
    return scenes.Scene([mla, *extra], [], [ns.Monitor([30, 0, 0], 8, 8)])


def _lens9(x):
    return asphere_lens9(ob, [x, 0, 0])


def _caps_rays(n):
    """caps_binding's geometry with n rays in families of six wavelengths (a family column: the serial path)."""
    arrs = scenes.ray_arrays(n, [3, 3, 0], [0, 2.5, 0.25], [-1, 0, 0], [0, 0.02, 0.0], wavelengths=np.linspace(450e-7, 900e-7, 6))
    arrs["family"] = (np.arange(n) // 6).astype(np.int32)
    return arrs


N = 2400
_disc = lambda n, **kw: scenes.ray_arrays(n, [0, 0, 0], [0, 2.0, 2.0], [1, 0, 0], [0, 0.004, 0.004], **kw)
# The 4f relay gets the benchmark's collimated disc, the bundle its q bar (parity.Q_RTOL_FD) was set on: the q behind an
# asphere inherits the reference's finite-difference curvature noise, which grows towards the lens rim (a 1-ulp change of
# the inputs moves the oracle's own q by 1.6e-7 on this disc and by 3.5e-7 on the wider square of `_disc`).
_c2 = lambda n: RayBundle.collimated_disc(n, start=7).materialise()
_cavity = lambda n: scenes.ray_arrays(n, [2, 0, 0], [0, 1, 1], [1, 0, 0], [0, 1e-5, 1e-5])
_slab_rays = lambda n: scenes.ray_arrays(n, [-3 - 2 * np.cos(np.pi / 6), 2 + 2 * np.sin(np.pi / 6), 0], [0, 0.3, 0.3],
                                         [np.cos(np.pi / 6), -np.sin(np.pi / 6), 0], [0, 0.01, 0.01])
_mma_rays = lambda n: scenes.ray_arrays(n, [0, 0, 0], [0, 0.1, 0.03], [1, 0, 0], [0, 0.02, 0.02])

# name -> (flat builder, rays builder, trace options, expected bits without SMEM, equal-distance ties allowed)
CASES = {
    "cavity_aligned": (lambda: _flat(scenes.cavity_aligned(ob)), _cavity, dict(max_trace_num=120), expect(0), False),
    "cavity_aligned_split": (lambda: _flat(scenes.cavity_aligned(ob)), _cavity, dict(max_trace_num=120, chain_len=1),
                             expect(0, split=True), False),
    "telescope_4f_no_boxes": (lambda: _no_box_tests(_flat(scenes.telescope_4f(ob, n_rays=0))), _c2,
                              dict(record_hist=True), expect(0, asph=True), False),
    "telescope_4f_no_boxes_split": (lambda: _no_box_tests(_flat(scenes.telescope_4f(ob, n_rays=0))), _c2,
                                    dict(record_hist=True, chain_len=1), expect(0, asph=True, split=True), False),
    "doublet": (lambda: _flat(scenes.doublet(ob)), lambda n: _disc(n, wavelengths=(780e-7, 560e-7, 400e-7)),
                dict(record_hist=True), expect(1), False),
    "glass_slab": (lambda: _flat(scenes.glass_slab(ob)), _slab_rays, dict(max_trace_num=100), expect(1, split=True), False),
    "gaussian_beam_split": (lambda: _flat(scenes.gaussian_beam(ob)), lambda n: scenes.ray_arrays(n, [-10, 4, 0], [0, 5, 0.3], [1, 0, 0], [0, 0.01, 0.01]),
                            dict(max_trace_num=60, chain_len=1), expect(1, split=True), False),
    "telescope_4f": (lambda: _flat(scenes.telescope_4f(ob, n_rays=0)), _c2, dict(record_hist=True), expect(1, asph=True), False),
    "telescope_4f_grid_split": (lambda: _flat(telescope_4f_grid(ob, 42.5, 44.0)),
                                _c2, dict(record_hist=True, chain_len=1), expect(1, asph=True, split=True), False),
    "mla_lattice": (lambda: _flat(_mla_lattice(ob)), lambda n: scenes.ray_arrays(n, [0, 0, 0], [0, 2.2, 1.2], [1, 0, 0], [0, 0.01, 0.01]),
                    dict(record_hist=True), expect(2), True),
    "mma_lattice": (lambda: _flat(_mma_lattice(ob)), _mma_rays, dict(max_trace_num=60, record_hist=True), expect(2, split=True), True),
    "mla_lattice_asphere": (lambda: _flat(_mla_lattice(ob, [_lens9(15.0)])),
                            lambda n: scenes.ray_arrays(n, [0, 0, 0], [0, 2.2, 1.2], [1, 0, 0], [0, 0.01, 0.01]),
                            dict(record_hist=True), expect(2, asph=True), True),
    "mma_lattice_asphere": (lambda: _flat(_mma_lattice(ob, [_lens9(6.0)])), _mma_rays, dict(max_trace_num=60, record_hist=True),
                            expect(2, asph=True, split=True), True),
    "reference_roots": (lambda: _flat(scenes.telescope_4f(ob, n_rays=0)), _c2, dict(reference_roots=True, record_hist=True),
                        expect(1, asph=True, split=True, brent=True), False),
    "reference_roots_serial": (lambda: _flat(scenes.caps_binding(ob)), _caps_rays, dict(max_trace_num=80, reference_roots=True),
                               expect(1, asph=True, split=True, serial=True, brent=True), True),
    "flag_ambiguity": (lambda: _flat(scenes.doublet(ob)), lambda n: _disc(n, wavelengths=(780e-7, 560e-7, 400e-7)),
                       dict(flag_ambiguity=True, record_hist=True), expect(1, asph=True, split=True, flag=True), False),
    "caps_serial": (lambda: _flat(scenes.caps_binding(ob)), _caps_rays, dict(max_trace_num=80, record_hist=True),
                    expect(1, asph=True, split=True, serial=True), True),
    "monitor_as_component": (lambda: _flat(scenes.monitor_as_component(ob)),
                             lambda n: scenes.ray_arrays(n, [0, 0, 0], [0, 1.5, 1.5], [1, 0, 0], [0, 0.01, 0.01], wavelengths=(633e-7,)),
                             dict(max_trace_num=25, record_hist=True), expect(1, asph=True, split=True, passk=True), False),
}


def _trace(engine, flat, arrs, opts):
    """Plan and result of one trace_arrays call on a fresh upload of `flat`."""
    scene = engine.upload(flat)
    try:
        plan = engine.trace_plan(scene, arrs, **opts)
        out = engine.trace_arrays(scene, arrs, **opts)
    finally:
        scene.close()
    return plan, out


def assert_twins(got, want, label, counters=SAME_COUNTERS):
    """Bit-identical rows (reference key order, every column), histograms, counters, interact counts, flags."""
    for k in SEG_COLS + HIT_COLS:
        assert len(got[k]) == len(want[k]), f"{label}: {k} rows {len(got[k])} != {len(want[k])}"
        assert np.array_equal(np.asarray(got[k]).view(np.uint8), np.asarray(want[k]).view(np.uint8)), f"{label}: {k}"
    for k in ("hist_y", "hist_yz", "cap_counts", "root_flags"):
        if k in want and k in got:
            np.testing.assert_array_equal(got[k], want[k], err_msg=f"{label}: {k}")
    np.testing.assert_array_equal(np.asarray(got["counters"])[counters], np.asarray(want["counters"])[counters], err_msg=f"{label}: counters")


def assert_plan(plan, bits, smem, label):
    assert plan["dynamic"] + plan["static"] <= plan["optin"], f"{label}: {plan}"
    want = bits | (A.PLAN_SMEM if smem else 0)
    got = plan["bits"] & ~A.PLAN_HIST_SMEM
    assert got == want, f"{label}: ran {describe(got)}, expected {describe(want)}"
    OBSERVED.setdefault(got, label)


def _oracle(flat, arrs, opts, nthreads=8):
    from oracle import oracle as O

    n_fam = int(arrs["family"].max()) + 1
    return O.trace(flat, arrs, max_trace_num=opts.get("max_trace_num", 2000), n_families=n_fam,
                   nthreads=1 if flat.n_capslots else nthreads)


@pytest.mark.parametrize("name", list(CASES))
def test_variant_twins_and_oracle(engine, name):
    from oracle import ref_harness as RH

    build, rays, opts, bits, ties_ok = CASES[name]
    flat = build()
    arrs = rays(N)
    plan_s, smem = _trace(engine, flat, arrs, opts)
    assert plan_s["blob"] == blob_bytes(flat) and plan_s["blob"] <= plan_s["optin"] - plan_s["static"]
    assert_plan(plan_s, bits, True, f"{name} (shared memory)")
    plan_g, glob = _trace(engine, padded(flat, GLOBAL_BLOB), arrs, opts)
    assert plan_g["blob"] == GLOBAL_BLOB
    assert_plan(plan_g, bits, False, f"{name} (global memory)")
    assert_twins(glob, smem, name)
    assert int(smem["counters"][A.C_STATUS]) == 0
    # real work: several generations where rays split or chains are cut, rows on the monitors when there are any
    if opts.get("chain_len") or (flat.max_children > 1 and not bits & A.PLAN_SERIAL):
        assert int(smem["counters"][A.C_GENERATIONS]) > 2, smem["counters"]
    if flat.n_monitors:
        assert len(smem["hit_root"]) > 0
    raw = _oracle(flat, arrs, opts)
    want = RH.arrays_from_result(raw)
    got = RH.arrays_from_result(smem)
    q = parity.q_rtol_for(flat)
    if ties_ok:
        _, ties = parity.compare_flagging_ties(flat, want, got, q_rtol=q, label=name)
        assert len(ties) <= 2e-3 * N, (name, ties)
    else:
        parity.compare(want, got, q_rtol=q, label=name)
        ties = []
    if flat.n_capslots and not ties:
        np.testing.assert_array_equal(smem["cap_counts"], raw["cap_counts"])
    if not ties:
        for c in (A.C_INTERACTIONS, A.C_HITS, A.C_DROPPED):
            assert int(smem["counters"][c]) == int(raw["counters"][c]), (name, c)


# ---- histogram placement ------------------------------------------------------------------------------------------
def _hist_scene(n_mons):
    """n_mons axis-aligned monitors along the beam (local y, z = the ray's), an absorber behind them."""
    hw = H.HALF_WIDTHS
    mons = [ob.Monitor([1.0 + k, 0, 0], width=2 * hw[k % 5], height=2 * hw[(k + 2) % 5]) for k in range(n_mons)]
    return FlatScene([ob.Block([n_mons + 5.0, 0, 0], width=40, height=40)], mons)


def _hist_rays(n):
    arrs = scenes.ray_arrays(n, [0, 0, 0], [0, 5.2, 5.2], [1, 0, 0], [0, 0, 0], w0=0)
    ys = np.concatenate([H.on_edge_grid(hw) for hw in H.HALF_WIDTHS[:5]])
    arrs["oy"][: ys.size] = ys[: n]
    arrs["oz"][: ys.size] = ys[::-1][: n]
    return arrs


def _check_numpy(flat, out, label):
    mon, py, pz = out["hit_monitor"], out["hit_py"], out["hit_pz"]
    mf = flat.mon_f.reshape(-1, A.MON_STRIDE)
    for m in range(flat.n_monitors):
        hw, hh = mf[m, A.MON_HW], mf[m, A.MON_HH]
        y, z = py[mon == m], pz[mon == m]
        assert y.size > 0
        assert np.array_equal(out["hist_y"][m], H.numpy_hist(y, hw)), f"{label} monitor {m}: " + H.explain_hist(y, out["hist_y"][m], hw)
        want2 = np.histogram2d(y, z, H.BINS, [[-hw, hw], [-hh, hh]])[0].astype(np.int64)
        assert np.array_equal(out["hist_yz"][m], want2), f"{label} monitor {m}: hist_yz"


def test_histograms_through_global_atomics_past_the_window(engine):
    """Tables in shared memory, histograms not: blob + histograms cross the window. Bit-identical to the same scene with
    shared-memory histograms, and np.histogram / np.histogram2d of the rows."""
    flat = _hist_scene(4)
    arrs = _hist_rays(4000)
    opts = dict(record_hist=True, max_trace_num=20)
    plan, small = _trace(engine, flat, arrs, opts)
    assert plan["bits"] & A.PLAN_SMEM and plan["bits"] & A.PLAN_HIST_SMEM, describe(plan["bits"])
    top = (plan["optin"] - max(plan["static"], _static_max(engine, flat, arrs))) // 16 * 16
    hist = 4 * A.HIST_BINS * (A.HIST_BINS + 1) * 4
    plan2, big = _trace(engine, padded(flat, top - 16), arrs, opts)
    assert top - 16 + hist > top   # blob + histograms over the budget, the blob alone within it
    assert plan2["bits"] & A.PLAN_SMEM and not plan2["bits"] & A.PLAN_HIST_SMEM, describe(plan2["bits"])
    assert plan2["dynamic"] == top - 16 and plan2["dynamic"] + plan2["static"] <= plan2["optin"]
    assert_twins(big, small, "global-atomic histograms")
    _check_numpy(flat, small, "4 monitors")


def test_histograms_of_twenty_monitors(engine):
    """20 monitors: 74 KiB of histograms, over the 64 KiB shared-memory limit, so global atomics with the tables in
    shared memory. Each group of four monitors traced on its own (shared-memory histograms) gives the same histograms."""
    flat = _hist_scene(20)
    arrs = _hist_rays(4000)
    opts = dict(record_hist=True, max_trace_num=30)
    plan, out = _trace(engine, flat, arrs, opts)
    assert plan["bits"] & A.PLAN_SMEM and not plan["bits"] & A.PLAN_HIST_SMEM, describe(plan["bits"])
    _check_numpy(flat, out, "20 monitors")
    d = flat.to_arrays()
    for g in range(5):
        sub = dict(d, mon_f=flat.mon_f.reshape(-1, A.MON_STRIDE)[4 * g:4 * g + 4].copy())
        sub["counts"] = d["counts"].copy()
        sub["counts"][2] = 4
        part = FlatScene.from_arrays(sub)
        p, o = _trace(engine, part, arrs, opts)
        assert p["bits"] & A.PLAN_HIST_SMEM
        np.testing.assert_array_equal(o["hist_y"], out["hist_y"][4 * g:4 * g + 4])
        np.testing.assert_array_equal(o["hist_yz"], out["hist_yz"][4 * g:4 * g + 4])


# ---- the edges of the shared-memory plan --------------------------------------------------------------------------
def _static_max(engine, flat, arrs):
    """Static shared memory of the general kind (flag_ambiguity): the largest of the shared-memory trace kernels."""
    scene = engine.upload(flat)
    try:
        return engine.trace_plan(scene, arrs, flag_ambiguity=True)["static"]
    finally:
        scene.close()


BOUNDARY_SCENES = {
    # aspheres + boxes (the 11.6 KiB static kinds) and a box-free scene of thin lenses (the 5.6 KiB ones)
    "telescope_4f": (lambda: _flat(scenes.telescope_4f(ob, n_rays=0)), lambda n: _disc(n, wavelengths=(780e-7,))),
    "gaussian_telescope": (lambda: _flat(scenes.gaussian_telescope(ob)),
                           lambda n: scenes.ray_arrays(n, [0, 0, 0], [0, 0.8, 0.8], [1, 0, 0], [0, 0.002, 0.002])),
}
SIZES = ([f"{32768 * k - 16}" for k in range(1, 7)] + [f"{32768 * k + 16}" for k in range(1, 7)]
         + [f"{s}{d:+d}" for s in ("sel", "max") for d in (-16, 0, 16)] + ["224992", "230400"])


def boundary_size(label, optin, s_sel, s_max):
    for name, s in (("sel", s_sel), ("max", s_max)):
        if label.startswith(name):
            return optin - s + int(label[len(name):])
    return int(label)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("scene_name", list(BOUNDARY_SCENES))
def test_blob_at_the_edges_of_the_window(engine, scene_name, size):
    """A blob of the given size (the unpadded scene, aux zeros appended) traces through optb_trace and optb_trace_host,
    with results bit-identical to the unpadded scene's; the plan launches within the opt-in limit and stages the
    tables in shared memory exactly when the blob fits the opt-in limit less the largest static shared memory."""
    build, rays = BOUNDARY_SCENES[scene_name]
    flat = build()
    arrs = rays(512)
    opts = dict(record_hist=True, max_trace_num=40)
    plan0, want = _trace(engine, flat, arrs, opts)
    s_max = _static_max(engine, flat, arrs)
    assert s_max >= plan0["static"] and plan0["bits"] & A.PLAN_SMEM
    blob = boundary_size(size, plan0["optin"], plan0["static"], s_max)
    assert blob % 16 == 0
    big = padded(flat, blob)
    scene = engine.upload(big)
    try:
        plan = engine.trace_plan(scene, arrs, **opts)
        assert plan["blob"] == blob and plan["dynamic"] + plan["static"] <= plan["optin"], plan
        assert bool(plan["bits"] & A.PLAN_SMEM) == (blob <= plan["optin"] - s_max), (plan, s_max)
        assert (plan["bits"] | A.PLAN_SMEM) & ~A.PLAN_HIST_SMEM == plan0["bits"] & ~A.PLAN_HIST_SMEM
        got = engine.trace_arrays(scene, arrs, **opts)
        assert_twins(got, want, f"{scene_name} blob {blob}")
        n, m = len(arrs["ox"]), flat.n_monitors
        prm = sorted_params(engine.make_params(40, record_hist=True, n_families=n))
        host = host_trace(engine, scene, arrs, prm, 64 * n, 64 * n, n_hist=m)
        assert_twins(host, want, f"{scene_name} blob {blob} (optb_trace_host)",
                     counters=[c for c in SAME_COUNTERS if c not in (A.C_LAUNCHES, A.C_GENERATIONS)])
    finally:
        scene.close()


def test_every_single_scene_variant_ran():
    """The variant matrix above ran all 34 single-scene trace_kernel instantiations: 12 parallel kinds and 5 general
    kinds, each with its tables in shared memory and in global memory."""
    if not OBSERVED:
        pytest.skip("runs after the variant matrix of this module")
    want = set()
    for smem in (0, A.PLAN_SMEM):
        for boxes in range(3):
            for asph in (False, True):
                for split in (False, True):
                    want.add(smem | expect(boxes, asph, split))
        general = expect(1, asph=True, split=True)
        for extra in (A.PLAN_BRENT, A.PLAN_BRENT | A.PLAN_SERIAL, A.PLAN_FLAG, A.PLAN_SERIAL, A.PLAN_PASSK):
            want.add(smem | general | extra)
    assert len(want) == 34
    missing = sorted(describe(b) for b in want - set(OBSERVED))
    assert not missing, f"variants never run: {missing}"
    print("trace_kernel variants run:", ", ".join(f"{describe(b)} ({OBSERVED[b]})" for b in sorted(OBSERVED)))
