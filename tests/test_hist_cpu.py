"""CPU: the C oracle's histogram binning is np.histogram's, at the bin edges too. The oracle stands in for the device in
every CPU test and is the device's reference in the GPU parity tests, so its binning is pinned to numpy here."""
import numpy as np
import pytest

from tests import golden_io
from tests import hist_cases as H


def _oracle_bins(x, hw):
    from oracle import oracle as O

    f = O.lib().optb_oracle_hist_bin
    return np.array([f(float(v), -hw, hw) for v in x], np.int64)


@pytest.mark.parametrize("hw", H.HALF_WIDTHS)
def test_oracle_hist_bin_is_np_histogram_at_the_edges(hw):
    x = H.edge_values(hw)
    b = _oracle_bins(x, hw)
    finite_in = np.isfinite(x) & (np.abs(x) <= hw)
    assert ((b >= 0) == finite_in).all(), "binned outside the range, or NaN / inf binned"
    got = np.bincount(b[b >= 0], minlength=H.BINS)
    assert got.size == H.BINS
    np.testing.assert_array_equal(got, H.numpy_hist(x, hw), err_msg=H.explain(x, b, hw))
    np.testing.assert_array_equal(b, H.numpy_bin(x, hw), err_msg=H.explain(x, b, hw))


def test_edge_values_reach_the_edges():
    """The value set really holds values on interior edges that a fused i * step + lo misplaces (hw = 2.5, and the
    plain y = -0.5000000000000001 of the 5 x 5 benchmark monitor)."""
    x = H.edge_values(2.5)
    assert np.float64(-0.5000000000000001) in x and H.numpy_bin(np.array([-0.5000000000000001]), 2.5)[0] == 11
    assert H.numpy_bin(np.array([-1.0]), 3.0)[0] == 10


def _yz(flat, arrs, m):
    """y, z of monitor m's rows as the C oracle forms them: the monitor-local point dotted with the lab tangents."""
    from optable_b200 import _abi as A

    sel = arrs["hit_monitor"] == m
    P = np.stack([arrs["hit_px"][sel], arrs["hit_py"][sel], arrs["hit_pz"][sel]], 1)
    mf = flat.mon_f[m]
    ty, tz = mf[A.MON_TY:A.MON_TY + 3], mf[A.MON_TZ:A.MON_TZ + 3]
    dot = lambda t: P[:, 0] * t[0] + P[:, 1] * t[1] + P[:, 2] * t[2]   # (a0 b0 + a1 b1) + a2 b2, unfused like the C
    return dot(ty), dot(tz), mf[A.MON_HW], mf[A.MON_HH]


@pytest.mark.parametrize("name", ["telescope_4f", "nested_csg", "monitor_as_component", "misc_components"])
def test_oracle_trace_histograms_are_numpy_of_its_rows(name):
    """hist_y / hist_yz that the oracle accumulates while tracing = np.histogram / np.histogram2d of its own rows."""
    from oracle import oracle as O

    flat, rays, params, _ = golden_io.load(name)
    assert flat.n_monitors > 0
    out = O.trace(flat, rays, record_segments=False, record_hist=True, **params)
    assert out["hist_y"].sum() > 0
    for m in range(flat.n_monitors):
        y, z, hw, hh = _yz(flat, out, m)
        np.testing.assert_array_equal(out["hist_y"][m], H.numpy_hist(y, hw), err_msg=f"{name} monitor {m}")
        want2, _, _ = np.histogram2d(y, z, H.BINS, [[-hw, hw], [-hh, hh]])
        np.testing.assert_array_equal(out["hist_yz"][m], want2.astype(np.int64), err_msg=f"{name} monitor {m}")
