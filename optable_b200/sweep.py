"""Scene sweeps: one ray bundle traced through K configurations of a scene in one device call.

The reference's heaviest callers re-trace one small scene many times with a parameter or two changed in between: the
GUI's `scan` over a grid of two script variables and its `optimize` (optable/interact.py:465-630), the Nelder-Mead
steps of `calibrate_symmetric_4f`, tolerance and Monte Carlo studies. One call per configuration leaves the GPU
nearly idle (a few hundred rays occupy a few SMs, and every call pays an upload and a host synchronisation). A sweep
uploads the K configurations as one sweep scene (include/optb.h `optb_scene_upload_sweep`) and traces K x N roots in
one call: root k * N + r is ray r of the bundle in configuration k.
"""
from __future__ import annotations

import numpy as np

from . import _abi as A

# what each node_i column means, for the topology-mismatch message
_NI_NAMES = {A.NI_GEOM: "geometry kind", A.NI_INTER: "interaction kind", A.NI_SKIP: "skip pointer",
             A.NI_AABB: "box-test flag", A.NI_MAT1: "material (x > 0 side)", A.NI_MAT2: "material (x < 0 side)",
             A.NI_CAPSLOT: "interact-cap slot", A.NI_AUX: "aux offset / asphere form", A.NI_ROCKIND: "ROC kind",
             A.NI_LEAF: "leaf index"}


def check_topology(flats):
    """Raise ValueError naming the first FlatScene that does not have the topology of flats[0]: the same table sizes,
    node_i rows identical except OPTB_NI_ORTHO, identical material kinds (what optb_scene_upload_sweep requires)."""
    f0 = flats[0]
    for k, f in enumerate(flats[1:], 1):
        what = None
        for name in ("n_nodes", "n_leaves", "n_materials", "n_monitors", "n_capslots"):
            if getattr(f, name) != getattr(f0, name):
                what = f"{name} {getattr(f, name)} != {getattr(f0, name)}"
                break
        if what is None and f.aux.size != f0.aux.size:
            what = f"aux pool of {f.aux.size} values != {f0.aux.size}"
        if what is None:
            cols = [c for c in range(A.NI_STRIDE) if c != A.NI_ORTHO]
            bad = np.argwhere(f.node_i[:, cols] != f0.node_i[:, cols])
            if bad.size:
                i, c = int(bad[0][0]), cols[int(bad[0][1])]
                what = f"node {i}: {_NI_NAMES.get(c, f'node_i column {c}')} {f.node_i[i, c]} != {f0.node_i[i, c]}"
        if what is None and not np.array_equal(f.mat_kind, f0.mat_kind):
            m = int(np.argmax(f.mat_kind != f0.mat_kind))
            what = f"material {m}: kind {f.mat_kind[m]} != {f0.mat_kind[m]}"
        if what is not None:
            raise ValueError(f"trace_sweep: table {k} does not have the topology of table 0 ({what})")


def _rays(rays):
    """(n, wavelength column, unit, packed host arrays or None) of a RayBundle or a list of Ray."""
    from .bundle import RayBundle
    from .flatten import pack_rays

    if isinstance(rays, RayBundle):
        return rays.n, rays.columns.get("wavelength"), None, None
    arrs, _, unit = pack_rays(list(rays))
    return len(arrs["ox"]), arrs["wavelength"], unit, arrs


def _device_sweep(flats, rays, limit, record_hits=True, record_hist=False, engine=None, unit=None, arrs=None):
    """The CUDA sweep: one sweep scene, one optb_trace over K x N roots, hit rows sorted into key order on the device."""
    from .backend import Engine
    from .bundle import DeviceTrace, run_to_fit

    engine = engine or Engine.get()
    K, M = len(flats), flats[0].n_monitors
    if limit > (1 << 24) or M > 256:
        raise ValueError("trace_sweep sorts rows by a packed key: max_trace_num <= 2^24 and at most 256 monitors")
    if arrs is None:
        n, rays_t = rays.n, rays.to_torch(device=f"cuda:{engine.device}")
    else:
        n = len(arrs["ox"])
        rays_t = engine.rays_to_device(arrs)
        del rays_t["family"]   # every root is its own family (rays.family must be NULL on a sweep scene)
    n_roots = K * n
    cap = n_roots * max(M, 1) * 2 if record_hits else 0
    dt, cnt = run_to_fit(lambda c: DeviceTrace(engine, flats[0], n, c, max_trace_num=limit, record_hist=record_hist,
                                               configs=flats, **({} if unit is None else {"unit": unit})),
                         rays_t, n_roots, limit, cap)
    nh = int(cnt[A.C_HITS]) if record_hits else 0
    engine._sort_rows_on_device(dt.res, 0, nh, limit, M)
    out = {k: dt.t[k][:nh] for k in dt.hit_columns} if record_hits else {}
    out["hist_y"], out["hist_yz"], out["counters"] = dt.t["hist_y"], dt.t["hist_yz"], cnt
    dt.scene.close()
    return out


class SweepResult:
    """Result of `trace_sweep`. `hits`: the monitor-row columns of all configurations (CUDA tensors in (root, monitor,
    pop) key order, so configuration-major; `hit_root` is the global root k * N + r); `hist_y` [K, M, 30],
    `hist_yz` [K, M, 30, 30]; `counters`: OPTB_C_* totals over all configurations (numpy)."""

    def __init__(self, tables, n, out, engine=None):
        import torch

        self.tables, self.n, self.n_configs, self.engine = list(tables), int(n), len(tables), engine
        K, M = self.n_configs, len(self.tables[0].monitors)
        self.counters = out["counters"]
        self.hist_y = out["hist_y"].reshape(K, -1, A.HIST_BINS)[:, :M]
        self.hist_yz = out["hist_yz"].reshape(K, -1, A.HIST_BINS, A.HIST_BINS)[:, :M]
        self.hits = {k: v for k, v in out.items() if k.startswith("hit_")}
        root = self.hits.get("hit_root")
        if root is not None:   # rows are sorted by root: configuration k owns the roots [k N, (k + 1) N)
            starts = torch.arange(K + 1, dtype=torch.int64, device=root.device) * self.n
            self._bounds = torch.searchsorted(root.long() & 0xFFFFFFFF, starts).tolist()
        else:
            self._bounds = [0] * (K + 1)
        self._grouped = None

    def _grouped_stats(self):
        from .analytics import grouped_stats

        if "hit_px" not in self.hits:
            raise ValueError("SweepResult.stats / row_values: this sweep was traced with record_hits=False, so it kept no "
                             "monitor rows to summarise")
        if self._grouped is None:
            M = len(self.tables[0].monitors)
            monitors = [[t.monitors[m] for m in range(M)] for t in self.tables]
            self._grouped = grouped_stats(self.hits, monitors, self.n, self.engine)
        return self._grouped

    def stats(self) -> dict:
        """Summaries of every configuration k and monitor m from one device call over all monitor rows
        (`optb_monitor_stats_grouped`; each in the frame of tables[k].monitors[m]) and one copy back: the keys of
        `DeviceMonitor.stats()` as numpy arrays [K, M] (hist_y [K, M, 30]), plus `std_tY` and `std_histy`. The same
        sweep gives the same bits on every call, so a ranking of configurations does not change between calls."""
        return self._grouped_stats()[0]

    def row_values(self) -> dict:
        """Per-row y, z, tY, tZ and waist_distance, each row evaluated in its own configuration's monitor frame: CUDA
        tensors aligned with `hits`, from the same device call as `stats()`."""
        v = self._grouped_stats()[1]
        return dict(zip(("y", "z", "tY", "tZ", "waist_distance"), v))

    def rows(self, k: int) -> dict:
        """Configuration k's monitor rows (views of the sorted columns) with `hit_root` (and `hit_key`) rebased to the
        bundle index r, plus its `hist_y` [M, 30] / `hist_yz` [M, 30, 30]: the shape of a `trace_bundle` result."""
        if not 0 <= k < self.n_configs:
            raise IndexError(f"configuration {k} of {self.n_configs}")
        lo, hi = self._bounds[k], self._bounds[k + 1]
        out = {c: v[lo:hi] for c, v in self.hits.items()}
        if "hit_root" in out:
            r = (out["hit_root"].long() & 0xFFFFFFFF) - k * self.n
            out["hit_root"] = (r - ((r >> 31) << 32)).to(out["hit_root"].dtype)   # uint32 bit pattern in int32
        if "hit_key" in out:
            out["hit_key"] = out["hit_key"] - ((k * self.n) << 32)
        out["hist_y"], out["hist_yz"] = self.hist_y[k], self.hist_yz[k]
        return out

    def monitor(self, k: int, m: int):
        """`DeviceMonitor` of monitor m in configuration k: every accessor of the reference's Monitor, on the device."""
        from .analytics import DeviceMonitor

        return DeviceMonitor(self.tables[k].monitors[m], self.rows(k), m, engine=self.engine)


def trace_sweep(tables, rays, perfomance_limit=None, record_hits=True, record_hist=False, engine=None, tracer=None):
    """Trace one bundle through every table of `tables` (K configurations of one scene, e.g. one builder function over
    a parameter grid) in one device call; returns a SweepResult.

    `tables`: OpticalTable-shaped objects (`.components`, `.monitors`; the reference's classes work too). Each is
    flattened with the bundle's wavelength set; tables whose topology differs from tables[0] (node count, component
    kinds, material kinds, ...) raise ValueError naming the first such table and what differs. Poses, apertures,
    reflectivities, glass coefficients and monitor placement may differ.
    `rays`: a RayBundle or a list of Ray (packed with pack_rays; every ray is its own interact-cap family).
    Interact caps follow `trace_bundle`: every capped component needs max_interact_count >= max_trace_num in every
    configuration, else NotImplementedError.

    Like `trace_bundle`, a sweep is a tensor entry point: it does not fill `table.rays`, `Monitor._data_raw` or the
    components' `_interact_count`. `tracer(flats, rays, max_trace_num, record_hits=, record_hist=, engine=, unit=,
    arrs=)` defaults to the CUDA sweep; the CPU tests pass a stand-in."""
    from .flatten import FlatScene, batch_wavelengths_m, trace_cap

    tables = list(tables)
    if not tables:
        raise ValueError("trace_sweep: no tables")
    n, wl, unit, arrs = _rays(rays)
    wl_unit = unit if unit is not None else getattr(tables[0], "unit", 1e-2)
    wls = None if wl is None else batch_wavelengths_m(wl, wl_unit)
    flats = [FlatScene(t.components, t.monitors, wavelengths_m=wls) for t in tables]
    check_topology(flats)
    tracer = tracer or _device_sweep
    out = tracer(flats, rays, trace_cap(perfomance_limit), record_hits=record_hits, record_hist=record_hist,
                 engine=engine, unit=unit, arrs=arrs)
    return SweepResult(tables, n, out, engine)
