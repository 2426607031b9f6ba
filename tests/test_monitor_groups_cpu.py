"""CPU: the summaries `stats_arrays` derives from stats slots, which `SweepResult.stats`, `analytics.monitor_stats` and
`DeviceMonitor.stats` return, against the same formulas written for one group's slots with scalars."""
import numpy as np
import pytest

from optable_b200 import _abi as A
from optable_b200.analytics import stats_arrays


def _reference(s, width):
    """The summaries of one group's slots s [OPTB_MS_STRIDE] and monitor width, one scalar at a time."""
    n = max(s[A.MS_COUNT], 1.0)
    counts = s[A.MS_HIST:A.MS_HIST + A.HIST_BINS].astype(np.int64)
    c, left = counts.astype(np.float64), np.linspace(-width / 2, width / 2, 31)[:-1]
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = (c * left).sum() / c.sum()
        std_histy = float(np.sqrt((c * left ** 2).sum() / c.sum() - mean ** 2))
    return {
        "count": int(s[A.MS_COUNT]), "sum_intensity": float(s[A.MS_SUM_I]), "avg_intensity": float(s[A.MS_SUM_I] / n),
        "mean_y": float(s[A.MS_SUM_Y] / n), "mean_z": float(s[A.MS_SUM_Z] / n),
        "std_y": float(np.sqrt(s[A.MS_M2_Y] / n)), "std_z": float(np.sqrt(s[A.MS_M2_Z] / n)),
        "min_y": float(s[A.MS_MIN_Y]), "max_y": float(s[A.MS_MAX_Y]), "min_z": float(s[A.MS_MIN_Z]), "max_z": float(s[A.MS_MAX_Z]),
        "mean_waist_distance": float(s[A.MS_SUM_WD] / n), "mean_tY": float(s[A.MS_SUM_TY] / n), "hist_y": counts,
        "std_tY": float(np.sqrt(s[A.MS_M2_TY] / n)), "std_histy": std_histy,
    }


def _slots(rng, K, M):
    s = np.zeros((K, M, A.MS_STRIDE))
    n = rng.integers(0, 5000, (K, M)).astype(np.float64)
    n[0, 0] = 0.0                                    # a group without rows
    s[..., A.MS_COUNT] = n
    for q in (A.MS_SUM_I, A.MS_SUM_Y, A.MS_SUM_Z, A.MS_SUM_WD, A.MS_SUM_TY):
        s[..., q] = rng.normal(0, 3, (K, M)) * n
    for q in (A.MS_SUM_YY, A.MS_SUM_ZZ, A.MS_SUM_TYTY, A.MS_M2_Y, A.MS_M2_Z, A.MS_M2_TY):
        s[..., q] = rng.uniform(0, 2, (K, M)) * n
    s[..., A.MS_MIN_Y], s[..., A.MS_MAX_Y] = -rng.uniform(0, 3, (K, M)), rng.uniform(0, 3, (K, M))
    s[..., A.MS_MIN_Z], s[..., A.MS_MAX_Z] = -rng.uniform(0, 3, (K, M)), rng.uniform(0, 3, (K, M))
    hist = rng.integers(0, 200, (K, M, A.HIST_BINS)).astype(np.float64)
    hist[0, 0] = 0.0
    hist[-1, -1, :] = 0.0
    hist[-1, -1, 7] = 5.0                            # every row in one bin: std_histy of a single bin
    s[..., A.MS_HIST:A.MS_HIST + A.HIST_BINS] = hist
    s[0, 0, A.MS_MIN_Y] = s[0, 0, A.MS_MIN_Z] = np.inf
    s[0, 0, A.MS_MAX_Y] = s[0, 0, A.MS_MAX_Z] = -np.inf
    return s


@pytest.mark.parametrize("K,M", [(1, 3), (7, 2), (16, 5)])
def test_stats_arrays_against_scalar_formulas(K, M):
    rng = np.random.default_rng(K * 10 + M)
    s = _slots(rng, K, M)
    widths = rng.choice([5.0, 2.54, 1.0, 0.2, 12.7], (K, M))
    got = stats_arrays(s, widths)
    assert got["count"].shape == (K, M) and got["hist_y"].shape == (K, M, A.HIST_BINS)
    for k in range(K):
        for m in range(M):
            want = _reference(s[k, m], widths[k, m])
            one = stats_arrays(s[k, m], widths[k, m])   # one group's slots, as DeviceMonitor.stats reads them
            assert set(got) == set(one) == set(want)
            for q, v in want.items():
                assert np.array_equal(got[q][k, m], v, equal_nan=q == "std_histy"), (k, m, q)
                assert np.array_equal(one[q], v, equal_nan=q == "std_histy"), (k, m, q)
            if s[k, m, A.MS_HIST:A.MS_HIST + A.HIST_BINS].sum() == 0:
                assert np.isnan(got["std_histy"][k, m])
