"""CPU: host-side solver helpers against the reference's (optable/solver.py) and against the oracle's slab."""
import numpy as np
import pytest

from oracle import ref_harness as RH

pytestmark = pytest.mark.skipif(not RH.reference_available(), reason="the unmodified optable reference package is not installed (baseline/_ref, or OPTABLE_REFERENCE_ROOT)")


def test_solver_helpers_equal_reference():
    import optable_b200 as ob

    ref = RH.load_reference()
    rng = np.random.default_rng(3)
    for k in range(200):
        o1, d1, o2, d2 = rng.normal(size=(4, 3))
        if k % 20 == 0:
            d2 = d1 * rng.uniform(0.5, 2.0)             # parallel branch
        got, want = ob.solve_ray_ray_intersection(o1, d1, o2, d2), ref.solve_ray_ray_intersection(o1, d1, o2, d2)
        for g, w in zip(got, want):
            np.testing.assert_allclose(g, w, rtol=1e-12, atol=1e-12)
        a, b = rng.normal(size=(2, 3))
        if k % 25 == 0:
            b = 3.0 * a
        (ax_g, th_g), (ax_w, th_w) = ob.solve_normal_to_normal_rotation(a, b), ref.solve_normal_to_normal_rotation(a, b)
        np.testing.assert_allclose(ax_g, ax_w, rtol=1e-12, atol=1e-12)
        assert th_g == pytest.approx(th_w, rel=1e-12, abs=1e-15)
        boxes = np.sort(rng.uniform(-3, 3, size=(12, 3, 2)), axis=2).reshape(12, 6)
        o, d = rng.uniform(-4, 4, 3), rng.normal(size=3)
        if k % 10 == 0:
            d[k % 3] = 0.0                                # containment-only axis
        g1, g2, gh = ob.solve_ray_bboxes_intersections(o, d, boxes)
        w1, w2, wh = ref.solve_ray_bboxes_intersections(o, d, boxes)
        np.testing.assert_array_equal(gh, wh)
        np.testing.assert_array_equal(g1, w1)
        np.testing.assert_array_equal(g2, w2)
