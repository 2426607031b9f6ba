"""CPU: optable_b200's own scene classes describe the same scenes as the reference's constructors.

Every fixture scene of tests/scenes.py is built with `ns = optable_b200`, flattened, and compared with the tables
stored in tests/golden/ (which came from the reference's classes): integer columns exact, floats to 1e-12."""
import numpy as np
import pytest

import optable_b200 as ob
from optable_b200.flatten import FlatScene, pack_rays, trace_cap
from tests import golden_io, scenes


@pytest.mark.parametrize("name", golden_io.names())
def test_flattened_tables_match_reference_classes(name):
    want_flat, want_rays, want_params, _ = golden_io.load(name)
    sc = scenes.REGISTRY[name](ob)
    flat = sc.flat()
    # Leaves (and their order) must agree exactly; the synthetic box hierarchy above them may be cut at
    # different, equally valid places when box coordinates differ in the last bits, so `skip` and the wrapper
    # rows are not compared (the wrappers are exact by construction, see FlatScene._wrap_runs).
    from optable_b200 import _abi as A

    cols = [A.NI_GEOM, A.NI_INTER, A.NI_AABB, A.NI_MAT1, A.NI_MAT2, A.NI_CAPSLOT, A.NI_AUX, A.NI_ROCKIND, A.NI_LEAF]
    mine, ref = flat.node_i[:, A.NI_LEAF] >= 0, want_flat.node_i[:, A.NI_LEAF] >= 0
    assert flat.n_leaves == want_flat.n_leaves == int(mine.sum()) == int(ref.sum())
    np.testing.assert_array_equal(flat.node_i[mine][:, cols], want_flat.node_i[ref][:, cols])
    np.testing.assert_allclose(flat.node_f[mine], want_flat.node_f[ref], rtol=1e-12, atol=1e-12)
    if flat.n_nodes == want_flat.n_nodes and np.array_equal(flat.node_i[:, A.NI_SKIP], want_flat.node_i[:, A.NI_SKIP]):  # same hierarchy
        np.testing.assert_array_equal(flat.node_i, want_flat.node_i)
        np.testing.assert_allclose(flat.node_f, want_flat.node_f, rtol=1e-12, atol=1e-12)
    np.testing.assert_array_equal(flat.mat_kind, want_flat.mat_kind)
    np.testing.assert_allclose(flat.mat_f, want_flat.mat_f, rtol=1e-15, atol=0)
    np.testing.assert_allclose(flat.mon_f, want_flat.mon_f, rtol=1e-12, atol=1e-12)
    # aux pool: polygon records + lattice descriptors (OPTB_G_GRID). A descriptor lists its children by NODE index,
    # which depends on where the synthetic hierarchy was cut: compare those through the leaf numbers they point at.
    assert flat.aux.shape == want_flat.aux.shape
    cellmask = np.zeros(flat.aux.size, bool)
    ga, gb = np.nonzero(flat.node_i[:, A.NI_GEOM] == A.G_GRID)[0], np.nonzero(want_flat.node_i[:, A.NI_GEOM] == A.G_GRID)[0]
    assert len(ga) == len(gb)
    for x, y in zip(ga, gb):
        ox, oy = int(flat.node_i[x, A.NI_AUX]), int(want_flat.node_i[y, A.NI_AUX])
        assert ox == oy
        ncell = int(flat.aux[ox + A.GRID_NOUTER] * flat.aux[ox + A.GRID_NINNER] + flat.aux[ox + A.GRID_NEXT])
        sl = slice(ox + A.GRID_CELLS, ox + A.GRID_CELLS + ncell)
        cellmask[sl] = True
        np.testing.assert_array_equal(flat.node_i[flat.aux[sl].astype(int), A.NI_LEAF],
                                      want_flat.node_i[want_flat.aux[sl].astype(int), A.NI_LEAF])
    np.testing.assert_allclose(flat.aux[~cellmask], want_flat.aux[~cellmask], rtol=1e-9, atol=1e-12)
    assert flat.max_children == want_flat.max_children
    arrs, fam_ids, unit = pack_rays(sc.rays)
    for k, v in want_rays.items():
        if k == "family":
            np.testing.assert_array_equal(arrs[k], v)
        elif arrs[k].dtype.kind == "f":
            np.testing.assert_allclose(arrs[k], v, rtol=1e-13, atol=1e-15)
        else:
            np.testing.assert_array_equal(arrs[k], v)
    assert trace_cap(sc.limit) == want_params["max_trace_num"]
    assert unit == want_params["unit"] and len(fam_ids) == want_params["n_families"]


def test_pose_verbs():
    m = ob.Mirror([1, 2, 3]).RotZ(0.3).TX(1).RotYAroundLocal([0, 0, 1], 0.2)
    assert np.allclose(m.transform_matrix @ m.transform_matrix.T, np.eye(3), atol=1e-14)
    g = ob.ComponentGroup([0, 0, 0])
    g.add_components([ob.Mirror([1, 0, 0]), ob.Lens([2, 0, 0], focal_length=3)])
    g.RotZ(np.pi / 2)
    assert np.allclose(g.components[0].origin, [0, 1, 0], atol=1e-14)
    g.TX(1)
    assert np.allclose(g.components[1].origin, [1, 2, 0], atol=1e-14)
    r = ob.Ray([0, 0, 0], [2, 0, 0], wavelength=780e-7, w0=61e-4)
    assert np.allclose(r.direction, [1, 0, 0]) and r.qo.imag > 0 and r.n == 1.0
    r2 = r.Propagate(-2)
    assert r2._id == r._id and r2.qo.real == -2


def test_error_behaviour_matches_reference():
    with pytest.raises(TypeError):
        ob.Sphere(1.0)  # height=None crashes in the reference too (surfaces.py:292)
    with pytest.raises(ValueError):
        ob.Polygon([[0, 0], [1, 1]])
    from optable_b200.flatten import FlattenError

    with pytest.raises(FlattenError):
        FlatScene([ob.BaseRefraciveSurface([0, 0, 0], n1=1, n2=1.5)])  # bare Plane has no boundary
    with pytest.raises(FlattenError):
        FlatScene([ob.CircleRefractive([0, 0, 0], n1=ob.Material("x", lambda wl: 1.5), n2=1)])


def _compare_flat(flat, want_flat):
    from optable_b200 import _abi as A

    cols = [A.NI_GEOM, A.NI_INTER, A.NI_AABB, A.NI_MAT1, A.NI_MAT2, A.NI_CAPSLOT, A.NI_AUX, A.NI_ROCKIND, A.NI_LEAF]
    mine, ref = flat.node_i[:, A.NI_LEAF] >= 0, want_flat.node_i[:, A.NI_LEAF] >= 0
    assert flat.n_leaves == want_flat.n_leaves == int(mine.sum()) == int(ref.sum())
    np.testing.assert_array_equal(flat.node_i[mine][:, cols], want_flat.node_i[ref][:, cols])
    np.testing.assert_allclose(flat.node_f[mine], want_flat.node_f[ref], rtol=1e-12, atol=1e-12)
    np.testing.assert_array_equal(flat.mat_kind, want_flat.mat_kind)
    np.testing.assert_allclose(flat.mat_f, want_flat.mat_f, rtol=1e-15, atol=0)
    np.testing.assert_allclose(flat.mon_f, want_flat.mon_f, rtol=1e-12, atol=1e-12)
    # aux pool: polygon records + lattice descriptors (OPTB_G_GRID). A descriptor lists its children by NODE index,
    # which depends on where the synthetic hierarchy was cut: compare those through the leaf numbers they point at.
    assert flat.aux.shape == want_flat.aux.shape
    cellmask = np.zeros(flat.aux.size, bool)
    ga, gb = np.nonzero(flat.node_i[:, A.NI_GEOM] == A.G_GRID)[0], np.nonzero(want_flat.node_i[:, A.NI_GEOM] == A.G_GRID)[0]
    assert len(ga) == len(gb)
    for x, y in zip(ga, gb):
        ox, oy = int(flat.node_i[x, A.NI_AUX]), int(want_flat.node_i[y, A.NI_AUX])
        assert ox == oy
        ncell = int(flat.aux[ox + A.GRID_NOUTER] * flat.aux[ox + A.GRID_NINNER] + flat.aux[ox + A.GRID_NEXT])
        sl = slice(ox + A.GRID_CELLS, ox + A.GRID_CELLS + ncell)
        cellmask[sl] = True
        np.testing.assert_array_equal(flat.node_i[flat.aux[sl].astype(int), A.NI_LEAF],
                                      want_flat.node_i[want_flat.aux[sl].astype(int), A.NI_LEAF])
    np.testing.assert_allclose(flat.aux[~cellmask], want_flat.aux[~cellmask], rtol=1e-9, atol=1e-12)
    assert flat.max_children == want_flat.max_children and flat.n_capslots == want_flat.n_capslots


@pytest.mark.parametrize("block", range(4))
def test_random_constructions_match_reference_classes(block):
    """Every component class with random constructor arguments and poses (tests/scenes.fuzz, 200 scenes, with and
    without interact caps): this package's classes and the reference's flatten to the same tables."""
    from oracle import ref_harness as RH

    if not RH.reference_available():
        pytest.skip("the unmodified optable reference package is not installed (baseline/_ref, or OPTABLE_REFERENCE_ROOT)")
    ref = RH.load_reference()
    for seed in range(7000 + 50 * block, 7050 + 50 * block):
        caps, extended = bool(seed % 2), bool(seed % 4 < 2)   # extended: the whole zoo incl. MMA, roof mirrors, prisms
        a, b = scenes.fuzz(ref, seed, caps=caps, extended=extended), scenes.fuzz(ob, seed, caps=caps, extended=extended)
        _compare_flat(FlatScene(b.components, b.monitors), FlatScene(a.components, a.monitors))
        ra, fa, ua = pack_rays(a.rays)
        rb, fb, ub = pack_rays(b.rays)
        assert ua == ub and len(fa) == len(fb)
        for k in ra:
            if ra[k].dtype.kind == "f":
                np.testing.assert_allclose(rb[k], ra[k], rtol=1e-13, atol=1e-15)
            else:
                np.testing.assert_array_equal(rb[k], ra[k])


def test_callable_material_becomes_a_per_wavelength_table():
    """a19: Material(n=<callable>) -> OPTB_MAT_LUT rows evaluated by the host at the batch's distinct wavelengths
    (metres); without the wavelengths the flattener refuses (there is no CPU fallback to hide behind)."""
    from optable_b200 import _abi as A
    from optable_b200.flatten import FlattenError

    sc = scenes.callable_material(ob)
    with pytest.raises(FlattenError):
        FlatScene(sc.components, sc.monitors)
    flat = sc.flat()
    lut = np.nonzero(flat.mat_kind == A.MAT_LUT)[0]
    assert len(lut) == 2
    wl = sorted({r.wavelength * r.unit for r in sc.rays})
    for m in lut:
        off, cnt = int(flat.mat_f[m, 0]), int(flat.mat_f[m, 1])
        tab = flat.aux[off:off + 2 * cnt].reshape(-1, 2)
        np.testing.assert_array_equal(tab[:, 0], wl)
        assert np.all(tab[:, 1] > 1.4) and np.all(np.diff(tab[:, 1]) < 0)   # normal dispersion of both laws


def test_refresh_rewrites_a_moved_component_in_place():
    """f3: FlatScene.refresh(component) = the rows a full re-flatten would produce, for a top-level leaf, a small group
    and a leaf deep inside the 7,689-leaf ripa scene (where it also has to take well under 5 ms); changes that cannot
    be expressed in place (a group with a synthetic box hierarchy, a new material) are refused with None."""
    import time

    sc = scenes.gaussian_beam(ob)
    flat = FlatScene(sc.components, sc.monitors)
    sc.components[0].TX(0.5).RotZ(0.1)
    assert flat.refresh(sc.components[0]) == [0]
    sc.components[4].TX(0.3)                                  # GlassSlab: a group of two faces
    changed = flat.refresh(sc.components[4])
    fresh = FlatScene(sc.components, sc.monitors)
    assert changed == [4, 5, 6]
    np.testing.assert_array_equal(flat.node_i, fresh.node_i)
    np.testing.assert_array_equal(flat.node_f, fresh.node_f)
    assert flat.leaves[int(flat.node_i[5, 9])] is sc.components[4].components[0]
    # a change of material adds a table row: not expressible in place
    sc.components[4].components[0]._n2 = ob.Material("other", n=1.7)
    assert flat.refresh(sc.components[4]) is None

    big = scenes.ripa(ob, n_rays=0)
    flat = FlatScene(big.components, big.monitors)
    fold = big.components[0].components[1]                    # a fold mirror inside the first ripa group
    fold.RotY(1e-3)
    flat.refresh(fold)                                        # (first call builds the parent table)
    fold.RotY(1e-3)
    t0 = time.perf_counter()
    changed = flat.refresh(fold)
    dt = time.perf_counter() - t0
    fresh = FlatScene(big.components, big.monitors)
    np.testing.assert_array_equal(flat.node_i, fresh.node_i)
    np.testing.assert_array_equal(flat.node_f, fresh.node_f)
    assert changed and len(changed) <= 3 and dt < 5e-3, (changed, dt)
    assert flat.refresh(big.components[0].components[3]) is None   # an MMA: box hierarchy + lattice descriptor
