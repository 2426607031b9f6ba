"""Monitor analytics on the device: the reference's `Monitor` accessors (optable/monitor.py:53-269) evaluated on
the row columns a bundle trace leaves in HBM, without copying rows to the host or building Python tuples.

`trace_bundle` returns one set of row columns for all monitors; `DeviceMonitor(table.monitors[m], out, m)` selects
monitor m's rows. The per-row quantities (y, z, slopes, waist distances) and every summary that needs no ordering
(row count, intensity sum / mean, moments and extrema of the spot, the 30-bin histogram behind `std_histy`) come from
the library's grouped statistics kernels (`optb_monitor_stats_grouped`, include/optb.h), which reduce every group of
rows in a fixed order: the same rows give the same bits on every call. `grouped_stats` and `monitor_stats` give the
summaries of every (configuration, monitor) of a result in one call; a `DeviceMonitor` is one group of such a call.
Only the accessors the reference defines through a sort (`sort="YZ"` / `"ID"` views, `get_delta_pos`) order those
columns with torch.sort (PyTorch as the array library). Row order "YZ" = lexicographic (y, z) of the monitor-local
point like `Monitor.sortYZIndex`; "ID" = by initial ray (a bundle ray's id is its index); None = device append order.
"""
from __future__ import annotations

import numpy as np

from . import _abi as A


def _frame(monitor) -> A.MonitorFrame:
    fr = A.MonitorFrame()
    fr.tangent_y[:] = [float(v) for v in monitor.tangent_Y]
    fr.tangent_z[:] = [float(v) for v in monitor.tangent_Z]
    fr.normal[:] = [float(v) for v in monitor.normal]
    fr.half_width, fr.half_height = float(monitor.width) / 2, float(monitor.height) / 2
    return fr


def stats_arrays(s, widths) -> dict:
    """`DeviceMonitor.stats()` of many monitors at once: stats slots s [..., OPTB_MS_STRIDE] (numpy) -> its keys as
    arrays shaped s.shape[:-1] (hist_y: [..., 30]), among them `std_tY` (from OPTB_MS_M2_TY) and `std_histy` (the
    reference's Monitor.std_histy: the spread of the left bin edges weighted by the counts; NaN for a monitor without
    rows in its histogram) for monitors of widths `widths`."""
    s = np.asarray(s, np.float64)
    n = np.maximum(s[..., A.MS_COUNT], 1.0)
    hist = s[..., A.MS_HIST:A.MS_HIST + A.HIST_BINS].astype(np.int64)
    w = np.asarray(widths, np.float64)
    c = hist.astype(np.float64)
    left = np.linspace(-w / 2, w / 2, A.HIST_BINS + 1, axis=-1)[..., :-1]
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = (c * left).sum(-1) / c.sum(-1)
        std_histy = np.sqrt((c * left ** 2).sum(-1) / c.sum(-1) - mean ** 2)
    return {
        "count": s[..., A.MS_COUNT].astype(np.int64), "sum_intensity": s[..., A.MS_SUM_I],
        "avg_intensity": s[..., A.MS_SUM_I] / n, "mean_y": s[..., A.MS_SUM_Y] / n, "mean_z": s[..., A.MS_SUM_Z] / n,
        "std_y": np.sqrt(s[..., A.MS_M2_Y] / n), "std_z": np.sqrt(s[..., A.MS_M2_Z] / n),
        "min_y": s[..., A.MS_MIN_Y], "max_y": s[..., A.MS_MAX_Y], "min_z": s[..., A.MS_MIN_Z], "max_z": s[..., A.MS_MAX_Z],
        "mean_waist_distance": s[..., A.MS_SUM_WD] / n, "mean_tY": s[..., A.MS_SUM_TY] / n,
        "hist_y": hist, "std_tY": np.sqrt(s[..., A.MS_M2_TY] / n), "std_histy": std_histy,
    }


def grouped_stats(out: dict, monitors, rays_per_config=0, engine=None):
    """Summaries of every (configuration k, monitor m) of the hit rows in `out` (CUDA tensors of one result) in one
    device call (`optb_monitor_stats_grouped`), each group in the frame of monitors[k][m]. A row's configuration is
    root // rays_per_config (0: one configuration). Returns (stats_arrays dict of [K, M] arrays, per-row values
    [5, n]: y, z, tY, tZ, waist distance as a CUDA tensor aligned with the rows). Raises ValueError when a row belongs
    to no group (its monitor or configuration is out of range): the counts would not add up to the rows."""
    s, per_row = grouped_slots(out, monitors, rays_per_config, engine)
    return stats_arrays(s, monitor_widths(monitors)), per_row


def monitor_widths(monitors):
    """[K][M] widths of monitors[k][m], the second argument of `stats_arrays`."""
    return [[float(m.width) for m in row] for row in monitors]


def grouped_slots(out: dict, monitors, rays_per_config=0, engine=None):
    """The raw stats slots [K, M, OPTB_MS_STRIDE] (numpy) and per-row values of `grouped_stats`."""
    from .backend import Engine

    K, M = len(monitors), len(monitors[0])
    any_col = out["hit_px"]
    engine = engine or Engine.get(any_col.device.index or 0)
    frames = (A.MonitorFrame * (K * M))(*[_frame(monitors[k][m]) for k in range(K) for m in range(M)])
    stats, per_row = engine.monitor_stats_grouped(out, frames, K, M, rays_per_config)
    s = stats.cpu().numpy().reshape(K, M, A.MS_STRIDE)
    n, counted = int(any_col.numel()), int(s[..., A.MS_COUNT].sum())
    if counted != n:
        raise ValueError(f"{n - counted} of {n} monitor rows belong to no (configuration, monitor) group of this "
                         f"{K} x {M} result: their monitor or configuration index is out of range")
    return s, per_row


def monitor_stats(monitors, out: dict, engine=None) -> dict:
    """`DeviceMonitor(monitors[m], out, m).stats()` of every monitor of a `trace_bundle` result in one device call:
    the same keys as arrays shaped [M] (hist_y [M, 30])."""
    s, _ = grouped_stats(out, [list(monitors)], 0, engine)
    return {k: v[0] for k, v in s.items()}


class DeviceMonitor:
    def __init__(self, monitor, out: dict, index: int, engine=None):
        import torch

        from .backend import Engine

        self.monitor, self.torch = monitor, torch
        self.engine = engine or Engine.get(out["hit_px"].device.index or 0)
        # one grouped call with monitors 0..index, each in this monitor's frame: rows of higher monitors fall in no
        # group, and group `index` holds this monitor's rows (the Engine is called directly because grouped_slots
        # refuses rows outside every group)
        frames = (A.MonitorFrame * (index + 1))(*[_frame(monitor)] * (index + 1))
        stats, cols = self.engine.monitor_stats_grouped(out, frames, 1, index + 1)
        self._slots = stats[index]
        mon = out["hit_monitor"] if out.get("hit_monitor") is not None else (out["hit_key"] >> 24) & 0xFF
        sel = torch.nonzero(mon == index).squeeze(1)
        col = lambda k: out[k][sel] if out.get(k) is not None else None
        has_d, has_q = out.get("hit_dx") is not None, out.get("hit_q_re") is not None
        self._y, self._z = cols[0][sel], cols[1][sel]
        self._ty = cols[2][sel] if has_d else None
        self._tz = cols[3][sel] if has_d else None
        self._wd = cols[4][sel] if has_d and has_q else None
        if out.get("hit_key") is not None and out.get("hit_root") is None:
            key = out["hit_key"][sel]
            self.root, self.pop = (key >> 32) & 0xFFFFFFFF, key & 0xFFFFFF
        else:
            self.root, self.pop = col("hit_root"), col("hit_pop")
        self.P = torch.stack([col("hit_px"), col("hit_py"), col("hit_pz")], 1)
        self.I, self.t = col("hit_intensity"), col("hit_t")
        d = [col("hit_dx"), col("hit_dy"), col("hit_dz")]
        self.direction = torch.stack(d, 1) if d[0] is not None else None
        qr, qi = col("hit_q_re"), col("hit_q_im")
        self.q = torch.complex(qr, qi) if qr is not None and qi is not None else None
        self.hist_y = out["hist_y"][index] if out.get("hist_y") is not None else None
        self._orders = {}
        self._stats = None

    def stats(self) -> dict:
        """Order-free summaries of this monitor's rows, the keys of `stats_arrays` (one small device-to-host read):
        `count` an int, `hist_y` an int64 array, every other key a float."""
        if self._stats is None:
            s = stats_arrays(self._slots.cpu().numpy(), float(self.monitor.width))
            self._stats = {k: v if k == "hist_y" else int(v) if k == "count" else float(v) for k, v in s.items()}
        return self._stats

    @property
    def ndata(self) -> int:
        return int(self.I.numel())

    def order(self, sort="YZ"):
        """Row permutation (int64 tensor) for a sort key of the reference's accessors."""
        torch = self.torch
        if sort not in self._orders:
            if sort == "YZ":       # np.lexsort((z, y)): y primary, z secondary = stable sort by z, then by y
                by_z = torch.sort(self.P[:, 2], stable=True).indices
                idx = by_z[torch.sort(self.P[by_z, 1], stable=True).indices]
            elif sort == "ID":
                key = (self.root.to(torch.int64) & 0xFFFFFFFF) << 32 | (self.pop.to(torch.int64) & 0xFFFFFFFF)
                idx = torch.sort(key, stable=True).indices
            else:
                idx = torch.arange(self.ndata, device=self.P.device)
            self._orders[sort] = idx
        return self._orders[sort]

    # -- the accessors (tensors on the device) --------------------------------------------------------
    def get_PList(self, sort="YZ"):
        return self.P[self.order(sort)]

    def get_yList(self, sort="YZ"):
        return self._y[self.order(sort)]   # monitor-LOCAL point . LAB tangent: the reference's quirk, kept (kernel)

    def get_zList(self, sort="YZ"):
        return self._z[self.order(sort)]

    def get_IList(self, sort="YZ"):
        return self.I[self.order(sort)]

    def get_tList(self, sort="YZ"):
        return self.t[self.order(sort)]

    def get_directionList(self, sort="YZ"):
        return self.direction[self.order(sort)]

    def get_tYList(self, sort="YZ"):
        return self._ty[self.order(sort)]

    def get_tZList(self, sort="YZ"):
        return self._tz[self.order(sort)]

    @property
    def sum_intensity(self):
        return self.stats()["sum_intensity"]

    @property
    def avg_intensity(self):
        return self.stats()["avg_intensity"]

    def get_waist_distance(self, sort="YZ"):
        """Distance from every hit to its beam waist, signed along the monitor normal (monitor.py:202-216)."""
        return self._wd[self.order(sort)]

    def get_delta_pos(self):
        y, z = self.get_yList(), self.get_zList()
        if y.numel() == 0:
            zero = self.torch.zeros(1, dtype=self.torch.float64, device=self.P.device)
            return zero, zero.clone()
        idx = self.torch.sort(y, stable=True).indices
        return self.torch.diff(y[idx]), self.torch.diff(z[idx])

    def _get_hist_y(self):
        """(counts, bin edges) of the 30-bin histogram of yList over +-width/2 (monitor.py:195-200), accumulated by
        the statistics kernels with np.histogram's binning."""
        w = float(self.monitor.width)
        return self.stats()["hist_y"], np.linspace(-w / 2, w / 2, 31)

    @property
    def std_histy(self):
        return self.stats()["std_histy"]

    def export_rays_npz(self, filename: str):
        """Same arrays as Monitor.export_rays_npz (monitor.py:255-269); this is the one place rows leave the device."""
        print(f"Exporting {self.ndata} rays to {filename} ...")
        host = lambda x: x.cpu().numpy()
        np.savez(filename, xList=host(self.get_yList()), yList=host(self.get_zList()), tXList=host(self.get_tYList()),
                 tYList=host(self.get_tZList()), IList=host(self.get_IList()))
