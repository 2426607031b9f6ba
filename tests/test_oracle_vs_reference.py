"""CPU: the C restatement against the Python reference on every fixture scene (live where the reference package is
installed, otherwise its stored results); the random-scene sweeps need the live reference."""
import pytest

from oracle import oracle as O
from oracle import ref_harness as RH
from optable_b200.flatten import FlatScene, pack_rays, trace_cap
from tests import golden_io, parity, scenes

needs_reference = pytest.mark.skipif(not RH.reference_available(), reason="the unmodified optable reference package is not installed (baseline/_ref, or OPTABLE_REFERENCE_ROOT)")


@pytest.mark.parametrize("name", list(scenes.REGISTRY))
def test_oracle_vs_live_reference(name, capsys):
    """Without the reference package, the scene is built with this package's own classes and compared with the
    reference's results for it as oracle/make_golden.py stored them (tests/golden/<name>.npz)."""
    if RH.reference_available():
        sc = scenes.REGISTRY[name](RH.load_reference())
        want = RH.run_reference(sc)
    else:
        import optable_b200 as ob

        sc = scenes.REGISTRY[name](ob)
        want = golden_io.load(name)[3]
    flat = sc.flat()
    arrs, fam_ids, unit = pack_rays(sc.rays)
    got = O.trace(flat, arrs, max_trace_num=trace_cap(sc.limit), unit=unit, n_families=len(fam_ids))
    q_rtol = parity.q_rtol_for(flat) if name.startswith("fuzz_") else parity.RTOL
    parity.compare(want, RH.arrays_from_result(got), q_rtol=q_rtol, label=name)


@needs_reference
@pytest.mark.parametrize("block", range(6))
def test_fuzz_scenes_oracle_equals_reference(block):
    """Random scenes over the whole component zoo (tests/scenes.fuzz): 60 scenes here; 8,900 were run when the
    generator was written (1.69 million segments): no index or pop-count difference except 33 initial rays at
    equal-distance ties between overlapping coplanar lenslets (parity.compare_flagging_ties), where numpy's and the
    C restatement's last bit of t decide differently; fields within 1e-9 except behind rotated finite-difference
    aspheres (q 4e-6 once) and 1.0-1.4e-9 on a length in 3 scenes (profiles/r1_parity_sweep.md)."""
    ref = RH.load_reference()
    flagged = rays = 0
    for seed in range(100 + 10 * block, 110 + 10 * block):
        sc = scenes.fuzz(ref, seed)
        flat = sc.flat()
        arrs, fam_ids, unit = pack_rays(sc.rays)
        want = RH.run_reference(sc)
        got = O.trace(flat, arrs, max_trace_num=trace_cap(sc.limit), unit=unit, n_families=len(fam_ids))
        fd = parity.q_rtol_for(flat) > parity.RTOL   # finite-difference asphere normals/curvatures: 1e-6 along whole paths
        _, ties = parity.compare_flagging_ties(flat, want, RH.arrays_from_result(got), rtol=1e-6 if fd else parity.RTOL,
                                               q_rtol=1e-4 if fd else parity.RTOL, label=f"fuzz seed {seed}")
        flagged += len(ties)
        rays += len(sc.rays)
    assert flagged <= max(1, 2e-3 * rays)


@needs_reference
def test_random_nested_composite_apertures():
    """40 random composites of circles, rectangles and polygons, up to four operator levels deep
    (tests/scenes.random_csg): the postfix programs of the flattener evaluated by the C restatement against the live
    reference's nested closures (surfaces.py:100-136), ray by ray."""
    from optable_b200 import _abi as A

    ref = RH.load_reference()
    nested = 0
    for seed in range(40):
        sc = scenes.random_csg(ref, seed)
        flat = sc.flat()
        nested += int(((flat.node_i[:, A.NI_GEOM] == A.G_CSG) & (flat.node_f[:, A.NF_P] == 2.0)).sum())
        arrs, fam_ids, unit = pack_rays(sc.rays)
        want = RH.run_reference(sc)
        got = O.trace(flat, arrs, max_trace_num=trace_cap(sc.limit), unit=unit, n_families=len(fam_ids))
        parity.compare(want, RH.arrays_from_result(got), label=f"random_csg seed {seed}")
    assert nested >= 30   # (a few draws end up with two simple operands: the flat record)


@needs_reference
def test_fuzz_scenes_with_binding_interact_caps():
    """Random scenes in which a third of the leaves carry max_interact_count 1-3 and rays come in three-wavelength
    families sharing one id (tests/scenes.fuzz(caps=True)): the visible set depends on the reference's sequential
    order (SURVEY A.6). Oracle against the live reference, interact-count tables included."""
    import numpy as np

    ref = RH.load_reference()
    reached = 0
    for seed in range(300, 316):
        sc = scenes.fuzz(ref, seed, caps=True)
        flat = sc.flat()
        arrs, fam_ids, unit = pack_rays(sc.rays)
        want = RH.run_reference(sc)
        want.pop("_leaves", None)
        got = O.trace(flat, arrs, max_trace_num=trace_cap(sc.limit), unit=unit, n_families=len(fam_ids))
        parity.compare_flagging_ties(flat, want, RH.arrays_from_result(got), q_rtol=1e-5, label=f"caps fuzz seed {seed}")
        for s, comp in enumerate(flat.capslots):
            for f, rid in enumerate(fam_ids):
                assert got["cap_counts"][s, f] == comp._interact_count.get(rid, 0)
            reached += int(got["cap_counts"][s].max() >= comp.max_interact_count)
    assert reached > 10


@needs_reference
@pytest.mark.parametrize("block", range(3))
def test_fuzz_scenes_whole_zoo(block):
    """tests/scenes.fuzz(extended=True): the remaining component classes (MMA, MirrorPair, MirrorPrism,
    TriangularPrism with its built-in caps, DovePrism polygons, the exact-spherical asphere, bare refractive faces)
    mixed into the random scenes, every third scene with binding caps. Fields behind finite-difference aspheres
    (normal and curvature from numerical derivatives, surfaces.py:351-369) are compared to 1e-6 along whole paths."""
    ref = RH.load_reference()
    for seed in range(800 + 12 * block, 812 + 12 * block):
        caps = seed % 3 == 0
        sc = scenes.fuzz(ref, seed, caps=caps, extended=True)
        flat = sc.flat()
        arrs, fam_ids, unit = pack_rays(sc.rays)
        want = RH.run_reference(sc)
        want.pop("_leaves", None)
        got = O.trace(flat, arrs, max_trace_num=trace_cap(sc.limit), unit=unit, n_families=len(fam_ids))
        fd = parity.q_rtol_for(flat) > parity.RTOL
        parity.compare_flagging_ties(flat, want, RH.arrays_from_result(got), rtol=1e-6 if fd else parity.RTOL,
                                     q_rtol=1e-4 if fd else parity.RTOL, label=f"zoo fuzz seed {seed}")
        for s, comp in enumerate(flat.capslots):
            for f, rid in enumerate(fam_ids):
                assert got["cap_counts"][s, f] == comp._interact_count.get(rid, 0)
