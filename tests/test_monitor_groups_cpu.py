"""CPU: the [K, M] summaries of SweepResult.stats / analytics.monitor_stats are DeviceMonitor.stats() and
DeviceMonitor.std_histy of each group's slots, evaluated by DeviceMonitor's own code on the same slots."""
from types import SimpleNamespace

import numpy as np
import pytest

from optable_b200 import _abi as A
from optable_b200.analytics import DeviceMonitor, stats_arrays


class _Slots(DeviceMonitor):
    """A DeviceMonitor whose fused pass already ran: only its stats slots and its monitor's width."""

    def __init__(self, slots, width):
        import torch

        self._stats, self._stats_dev = None, torch.from_numpy(slots)
        self.monitor = SimpleNamespace(width=width)


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
def test_stats_arrays_are_device_monitor_stats(K, M):
    rng = np.random.default_rng(K * 10 + M)
    s = _slots(rng, K, M)
    widths = rng.choice([5.0, 2.54, 1.0, 0.2, 12.7], (K, M))
    got = stats_arrays(s, widths)
    assert got["count"].shape == (K, M) and got["hist_y"].shape == (K, M, A.HIST_BINS)
    for k in range(K):
        for m in range(M):
            dm = _Slots(np.ascontiguousarray(s[k, m]), widths[k, m])
            want = dm.stats()
            for q, v in want.items():
                assert np.array_equal(got[q][k, m], v), (k, m, q)
            assert got["std_tY"][k, m] == np.sqrt(s[k, m, A.MS_M2_TY] / max(s[k, m, A.MS_COUNT], 1.0))
            if s[k, m, A.MS_HIST:A.MS_HIST + A.HIST_BINS].sum() == 0:
                assert np.isnan(got["std_histy"][k, m])
            else:
                assert got["std_histy"][k, m] == dm.std_histy, (k, m)
