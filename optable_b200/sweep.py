"""Scene sweeps: one ray bundle traced through K configurations of a scene in one device call.

The reference's heaviest callers re-trace one small scene many times with a parameter or two changed in between: the
GUI's `scan` over a grid of two script variables and its `optimize` (optable/interact.py:465-630), the Nelder-Mead
steps of `calibrate_symmetric_4f`, tolerance and Monte Carlo studies. One call per configuration leaves the GPU
nearly idle (a few hundred rays occupy a few SMs, and every call pays an upload and a host synchronisation). A sweep
uploads the K configurations as one sweep scene (include/optb.h `optb_scene_upload_sweep`) and traces K x N roots in
one call: root k * N + r is ray r of the bundle in configuration k.

`trace_sweep(tables)` flattens K whole tables. A study that moves one or two components of a large scene keeps a
`SweepScene` instead: the table is flattened once, each configuration re-reads only the varied components and monitors
(`FlatScene.refresh`), and the device builds the K configuration blobs from the base and those rows
(`optb_scene_upload_sweep_rows`).
"""
from __future__ import annotations

import numpy as np

from . import _abi as A

# what each node_i column means, for the topology-mismatch message
_NI_NAMES = {A.NI_GEOM: "geometry kind", A.NI_INTER: "interaction kind", A.NI_SKIP: "skip pointer",
             A.NI_AABB: "box-test flag", A.NI_MAT1: "material (x > 0 side)", A.NI_MAT2: "material (x < 0 side)",
             A.NI_CAPSLOT: "interact-cap slot", A.NI_AUX: "aux offset / asphere form", A.NI_ROCKIND: "ROC kind",
             A.NI_LEAF: "leaf index"}


def topology_mismatch(flats):
    """(k, what) of the first FlatScene of `flats` that does not have the topology of flats[0], or None: the same
    table sizes, node_i rows identical except OPTB_NI_ORTHO, identical material kinds (what optb_scene_upload_sweep
    requires)."""
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
            return k, what
    return None


def check_topology(flats):
    """Raise ValueError naming the first FlatScene that does not have the topology of flats[0] (`topology_mismatch`)."""
    bad = topology_mismatch(flats)
    if bad is not None:
        raise ValueError(f"trace_sweep: table {bad[0]} does not have the topology of table 0 ({bad[1]})")


def topology_key(flat) -> bytes:
    """Digest of what `topology_mismatch` compares: equal digests, equal topology. Ranks of a sharded sweep compare
    these instead of their tables."""
    import hashlib

    h = hashlib.sha256()
    h.update(np.array([flat.n_nodes, flat.n_leaves, flat.n_materials, flat.n_monitors, flat.n_capslots, flat.aux.size],
                      dtype=np.int64).tobytes())
    cols = [c for c in range(A.NI_STRIDE) if c != A.NI_ORTHO]
    h.update(np.ascontiguousarray(flat.node_i[:, cols], dtype=np.int32).tobytes())
    h.update(np.ascontiguousarray(flat.mat_kind, dtype=np.int32).tobytes())
    return h.digest()


def _rays(rays):
    """(n, wavelength column, unit, packed host arrays or None, family ids or None) of a RayBundle or a list of Ray."""
    from .bundle import RayBundle
    from .flatten import pack_rays

    if isinstance(rays, RayBundle):
        return rays.n, rays.columns.get("wavelength"), None, None, None
    arrs, fam_ids, unit = pack_rays(list(rays))
    return len(arrs["ox"]), arrs["wavelength"], unit, arrs, fam_ids


def initial_counts(cap_components, fam_ids):
    """The starting interact counts of a sweep of Ray objects, [n_capslots, K * F] int32: column k * F + f holds
    `cap_components[k][s]._interact_count` of ray id fam_ids[f] (F = len(fam_ids)). None for a bundle (fam_ids None)
    or a scene without caps."""
    if fam_ids is None or not cap_components or not len(cap_components[0]):
        return None
    F = len(fam_ids)
    out = np.zeros((len(cap_components[0]), len(cap_components) * F), np.int32)
    for k, comps in enumerate(cap_components):
        for s, c in enumerate(comps):
            out[s, k * F:(k + 1) * F] = [c._interact_count.get(rid, 0) for rid in fam_ids]
    return out


def largest_family(arrs) -> int:
    """Initial rays of the largest `_id` family of a packed batch (0 when empty)."""
    return int(np.bincount(arrs["family"]).max()) if len(arrs["family"]) else 0


def caps_bind(caps0, arrs, cap_min, limit) -> bool:
    """Whether a sweep of the packed Ray batch `arrs` from the initial counts `caps0` needs the family-serial path:
    the rule of `Engine._arrays_params` over all its configurations (`cap_min`: their smallest cap)."""
    from .backend import caps_can_bind

    return caps_can_bind(caps0.max(initial=0), largest_family(arrs), cap_min, limit)


def _family_counts(table, caps0, family, K, n, serial):
    """`SweepResult.interact_counts` [K, S, F] from the device's cap table: the family-serial table itself
    ([S, K * F]), or, where no cap can bind (every root its own family, counted from zero: [S, >= K * n]), the initial
    counts plus the counts of each family's roots."""
    S, F = caps0.shape[0], caps0.shape[1] // K
    if serial:
        c = np.asarray(table[:, :K * F]).reshape(S, K, F)
    else:
        c = caps0.reshape(S, K, F).astype(np.int64)
        np.add.at(c, (slice(None), slice(None), np.asarray(family)), np.asarray(table[:, :K * n]).reshape(S, K, n))
    return np.ascontiguousarray(c.transpose(1, 0, 2), dtype=np.int32)


def _device_sweep(configs, rays, limit, record_hits=True, record_hist=False, engine=None, unit=None, arrs=None,
                  chain_len=0, caps0=None, serial=False):
    """The CUDA sweep: one sweep scene, one optb_trace over K x N roots, hit rows sorted into key order on the device.
    `configs`: the FlatScenes of the K configurations, or a SweepRows. `chain_len` > 0 runs the wavefront kernels
    (a shard of a sharded sweep whose own configurations do not split, when others do). `caps0` (Ray objects on a
    capped scene: `initial_counts`) adds `interact_counts` [K, S, F] to the result; with `serial` (`caps_bind`) the
    sweep runs family-serially from these counts."""
    from .backend import Engine
    from .bundle import DeviceTrace, run_to_fit

    engine = engine or Engine.get()
    rows = configs if isinstance(configs, SweepRows) else None
    flat0, K = (rows.flat, rows.n_configs) if rows is not None else (configs[0], len(configs))
    M = flat0.n_monitors
    if limit > (1 << 24) or M > 256:
        raise ValueError("trace_sweep sorts rows by a packed key: max_trace_num <= 2^24 and at most 256 monitors")
    if arrs is None:
        n, rays_t = rays.n, rays.to_torch(device=f"cuda:{engine.device}")
    else:
        n = len(arrs["ox"])
        rays_t = engine.rays_to_device(arrs)
        if not serial:
            del rays_t["family"]   # every root is its own family (rays.family must be NULL on a parallel sweep)
    n_roots = K * n
    cap = n_roots * max(M, 1) * 2 if record_hits else 0
    serial_kw = {"cap_counts": caps0, "n_families": caps0.shape[1] // K} if serial else {}
    dt, cnt = run_to_fit(lambda c: DeviceTrace(engine, flat0, n, c, max_trace_num=limit, record_hist=record_hist,
                                               chain_len=chain_len, configs=configs, **serial_kw,
                                               **({} if unit is None else {"unit": unit})),
                         rays_t, n_roots, limit, cap)
    nh = int(cnt[A.C_HITS]) if record_hits else 0
    engine._sort_rows_on_device(dt.res, 0, nh, limit, M)
    out = {k: dt.t[k][:nh] for k in dt.hit_columns} if record_hits else {}
    out["hist_y"], out["hist_yz"], out["counters"] = dt.t["hist_y"], dt.t["hist_yz"], cnt
    if caps0 is not None:
        out["interact_counts"] = _family_counts(dt.t["cap_counts"].cpu().numpy(), caps0, arrs["family"], K, n, serial)
    dt.scene.close()
    return out


class SweepResult:
    """Result of `trace_sweep` or `SweepScene.trace`. `hits`: the monitor-row columns of all configurations (CUDA
    tensors in (root, monitor, pop) key order, so configuration-major; `hit_root` is the global root k * N + r);
    `hist_y` [K, M, 30], `hist_yz` [K, M, 30, 30]; `counters`: OPTB_C_* totals over all configurations (numpy).
    `monitors[k][m]`: monitor m as configuration k placed it (default: tables[k].monitors[m]), the frame `stats`,
    `row_values` and `monitor` evaluate its rows in.

    Of a sharded call (`group=`): `shard` = (k0, k1), the configurations this rank traced, and `counters_local` its own
    counters; `counters`, the histograms, `monitors` and `stats()` cover all K configurations on every rank. `hits`
    holds this rank's rows with global roots, or every rank's rows with `gather=True`; `rows(k)` and `monitor(k, m)`
    of a configuration whose rows this rank does not hold raise IndexError. `chain_len` > 0 when this rank ran the
    wavefront kernels with that chain length to match the kernel variant of the one-GPU sweep (0 otherwise).

    Of a sweep of Ray objects: `family_ids`, the ray id of each interact-cap family (`pack_rays` order);
    `cap_components` [K][S], the capped components of each configuration (FlatScene cap-slot order); and
    `interact_counts`, int32 [K, S, F]: interact_counts[k, s, f] is what cap_components[k][s]._interact_count[
    family_ids[f]] would hold after tables[k].ray_tracing(rays). A sweep does not write these counts back. A RayBundle
    sweep has none of the three (None)."""

    def __init__(self, tables, n, out, engine=None, monitors=None, family_ids=None, cap_components=None):
        import torch

        self.tables, self.n, self.n_configs, self.engine = list(tables), int(n), len(tables), engine
        self.monitors = [list(t.monitors) for t in self.tables] if monitors is None else monitors
        K, M = self.n_configs, len(self.monitors[0])
        self.counters = out["counters"]
        self.hist_y = out["hist_y"].reshape(K, -1, A.HIST_BINS)[:, :M]
        self.hist_yz = out["hist_yz"].reshape(K, -1, A.HIST_BINS, A.HIST_BINS)[:, :M]
        self.hits = {k: v for k, v in out.items() if k.startswith("hit_")}
        self.shard, self.counters_local, self.chain_len = out.get("shard"), out.get("counters_local"), out.get("chain_len", 0)
        self._world = out.get("world", 1)
        self.family_ids = None if family_ids is None else list(family_ids)
        self.interact_counts = out.get("interact_counts")
        if self.interact_counts is None and family_ids is not None:    # a scene without caps
            self.interact_counts = np.zeros((K, 0, len(family_ids)), np.int32)
        self._cap_components = cap_components
        self._holds = out.get("holds", (0, K))      # the configurations whose rows `hits` holds
        root = self.hits.get("hit_root")
        if root is not None:   # rows are sorted by root: configuration k owns the roots [k N, (k + 1) N)
            starts = torch.arange(K + 1, dtype=torch.int64, device=root.device) * self.n
            self._bounds = torch.searchsorted(root.long() & 0xFFFFFFFF, starts).tolist()
        else:
            self._bounds = [0] * (K + 1)
        self._grouped = None
        # a sharded call summarises every configuration on the rank that holds its rows and gathers the slots, so
        # stats() is never a collective (a script in which one rank asks must not hang)
        self._stats = None
        if out.get("stats_slots") is not None:
            from .analytics import monitor_widths, stats_arrays

            self._stats = stats_arrays(out["stats_slots"], monitor_widths(self.monitors))

    @property
    def cap_components(self):
        if callable(self._cap_components):
            self._cap_components = self._cap_components()
        return self._cap_components

    def _grouped_stats(self):
        from .analytics import grouped_stats

        if "hit_px" not in self.hits:
            raise ValueError("SweepResult.stats / row_values: this sweep was traced with record_hits=False, so it kept no "
                             "monitor rows to summarise")
        if self._grouped is None:
            self._grouped = grouped_stats(self.hits, self.monitors, self.n, self.engine)
        return self._grouped

    def stats(self) -> dict:
        """Summaries of every configuration k and monitor m from one device call over all monitor rows
        (`optb_monitor_stats_grouped`; each in the frame of monitors[k][m]) and one copy back: the keys of
        `DeviceMonitor.stats()` as numpy arrays [K, M] (hist_y [K, M, 30]). The same sweep gives the same bits on
        every call, so a ranking of configurations does not change between calls; a sharded sweep gives the bits of
        the one-GPU sweep."""
        return self._stats if self._stats is not None else self._grouped_stats()[0]

    def row_values(self) -> dict:
        """Per-row y, z, tY, tZ and waist_distance, each row evaluated in its own configuration's monitor frame: CUDA
        tensors aligned with `hits` (after a sharded call: the rows this rank holds)."""
        v = self._grouped_stats()[1]
        return dict(zip(("y", "z", "tY", "tZ", "waist_distance"), v))

    def rows(self, k: int) -> dict:
        """Configuration k's monitor rows (views of the sorted columns) with `hit_root` (and `hit_key`) rebased to the
        bundle index r, plus its `hist_y` [M, 30] / `hist_yz` [M, 30, 30]: the shape of a `trace_bundle` result."""
        if not 0 <= k < self.n_configs:
            raise IndexError(f"configuration {k} of {self.n_configs}")
        if not self._holds[0] <= k < self._holds[1]:
            from .dist import shard_bounds

            owner = next(r for r in range(self._world) if k < shard_bounds(self.n_configs, r, self._world)[1])
            raise IndexError(f"configuration {k}: its rows are on rank {owner} of this sharded sweep (this rank holds "
                             f"configurations [{self._holds[0]}, {self._holds[1]})); trace with gather=True to hold "
                             "every configuration's rows on every rank")
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

        return DeviceMonitor(self.monitors[k][m], self.rows(k), m, engine=self.engine)


def _sharded(group):
    """Whether `group=` asks for a sharded sweep: True (the default process group) or a ProcessGroup, under an
    initialised torch.distributed; None / False, or no process group, is the one-GPU call."""
    if group is None or group is False:
        return False
    import torch.distributed as dist

    return dist.is_available() and dist.is_initialized()


def trace_sweep(tables, rays, perfomance_limit=None, record_hits=True, record_hist=False, engine=None, tracer=None,
                group=None, gather=False):
    """Trace one bundle through every table of `tables` (K configurations of one scene, e.g. one builder function over
    a parameter grid) in one device call; returns a SweepResult.

    `tables`: OpticalTable-shaped objects (`.components`, `.monitors`; the reference's classes work too). Each is
    flattened with the bundle's wavelength set; tables whose topology differs from tables[0] (node count, component
    kinds, material kinds, ...) raise ValueError naming the first such table and what differs. Poses, apertures,
    reflectivities, glass coefficients and monitor placement may differ.
    `rays`: a RayBundle or a list of Ray (packed with pack_rays).
    Interact caps: a list of Ray is traced as `tables[k].ray_tracing(rays)` would trace it, with the rays' `_id`
    families and the components' current `_interact_count` as starting counts. Where a cap can bind (the rule of
    `Engine.trace_arrays`, over all configurations), every family runs serially in the reference's order (the
    family-serial sweep kernel); the final counts are `SweepResult.interact_counts`. A RayBundle follows
    `trace_bundle`: every ray is its own family counted from zero, and every capped component needs
    max_interact_count >= max_trace_num in every configuration, else NotImplementedError.

    `group=True` (the default process group) or a ProcessGroup shards the configurations over its ranks, one GPU
    each (`optable_b200.dist.trace_sweep_sharded`): rank r flattens and traces only the contiguous configurations
    `shard_bounds(K, r, world)`, and every rank gets the histograms, counters, monitor frames and `stats()` of all K;
    `gather=True` also gives every rank every row. Each configuration's rows, histograms and statistics are the bits
    of the one-GPU call.

    Like `trace_bundle`, a sweep is a tensor entry point: it does not fill `table.rays`, `Monitor._data_raw` or the
    components' `_interact_count`. `tracer(flats, rays, max_trace_num, record_hits=, record_hist=, engine=, unit=,
    arrs=)` (plus `chain_len=` when sharded, and `caps0=`, `serial=` for Ray objects on a capped scene) defaults to
    the CUDA sweep; the CPU tests pass a stand-in."""
    from .flatten import FlatScene, batch_wavelengths_m, trace_cap

    tables = list(tables)
    if not tables:
        raise ValueError("trace_sweep: no tables")
    n, wl, unit, arrs, fam_ids = _rays(rays)
    wl_unit = unit if unit is not None else getattr(tables[0], "unit", 1e-2)
    wls = None if wl is None else batch_wavelengths_m(wl, wl_unit)
    flatten = lambda ts: [FlatScene(t.components, t.monitors, wavelengths_m=wls) for t in ts]
    tracer = tracer or _device_sweep
    if _sharded(group):
        from .dist import trace_sweep_sharded

        def prepare(k0, k1):
            flats = flatten(tables[k0:k1])
            return flats, None, initial_counts([f.capslots for f in flats], fam_ids)

        out, _ = trace_sweep_sharded(len(tables), n, rays, trace_cap(perfomance_limit), prepare,
                                     [list(t.monitors) for t in tables], "trace_sweep: table", tracer,
                                     group=None if group is True else group, gather=gather, record_hits=record_hits,
                                     record_hist=record_hist, engine=engine, unit=unit, arrs=arrs, fam_ids=fam_ids)
        comps = None if fam_ids is None else (lambda: [list(f.capslots) for f in flatten(tables)])
        return SweepResult(tables, n, out, engine, family_ids=fam_ids, cap_components=comps)
    flats = flatten(tables)
    check_topology(flats)
    limit = trace_cap(perfomance_limit)
    caps0 = initial_counts([f.capslots for f in flats], fam_ids)
    kw = {} if caps0 is None else {"caps0": caps0, "serial": caps_bind(caps0, arrs, min(f.cap_min for f in flats), limit)}
    out = tracer(flats, rays, limit, record_hits=record_hits, record_hist=record_hist, engine=engine, unit=unit,
                 arrs=arrs, **kw)
    return SweepResult(tables, n, out, engine, family_ids=fam_ids,
                       cap_components=None if fam_ids is None else [list(f.capslots) for f in flats])


def _children(ni, nf):
    """Most rays one interaction of each row can emit (FlatScene._physics's count, from the rows)."""
    inter, refl, trans = ni[..., A.NI_INTER], nf[..., A.NF_REFL] > 0, nf[..., A.NF_TRANS] > 0
    return np.select([inter == A.I_MIRROR, inter == A.I_REFRACT, (inter == A.I_THINLENS) | (inter == A.I_PASS)],
                     [refl.astype(np.int64) + trans, 1 + refl.astype(np.int64), 1], 0)


class SweepRows:
    """K configurations of one scene as its base FlatScene plus the rows that differ (include/optb.h
    `optb_scene_upload_sweep_rows`): configuration k is `flat` with node rows `nodes[v]` replaced by node_i[k, v] /
    node_f[k, v] and monitor records `monitors[w]` by mon_f[k, w]. It stands for all K configurations wherever a sweep
    needs a property of them (Scene, DeviceTrace, backend.runs_wavefront), without K FlatScenes on the host."""

    def __init__(self, flat, n_configs, nodes, node_i, node_f, monitors, mon_f):
        self.flat, self.n_configs = flat, int(n_configs)
        self.nodes = np.ascontiguousarray(nodes, dtype=np.int32)
        self.monitors = np.ascontiguousarray(monitors, dtype=np.int32)
        self.node_i = np.ascontiguousarray(node_i, dtype=np.int32).reshape(self.n_configs, self.nodes.size, A.NI_STRIDE)
        self.node_f = np.ascontiguousarray(node_f, dtype=np.float64).reshape(self.n_configs, self.nodes.size, A.NF_STRIDE)
        self.mon_f = np.ascontiguousarray(mon_f, dtype=np.float64).reshape(self.n_configs, self.monitors.size, A.MON_STRIDE)
        self.n_monitors, self.n_capslots, self.has_pass = flat.n_monitors, flat.n_capslots, flat.has_pass
        fixed = np.ones(flat.n_nodes, dtype=bool)
        fixed[self.nodes] = False
        self.max_children = int(max(_children(flat.node_i[fixed], flat.node_f[fixed]).max(initial=0),
                                     _children(self.node_i, self.node_f).max(initial=0)))
        capped, capped_v = flat.node_i[fixed, A.NI_CAPSLOT] >= 0, self.node_i[..., A.NI_CAPSLOT] >= 0
        self.cap_min = float(min(flat.node_f[fixed][capped, A.NF_CAPMAX].min(initial=np.inf),
                                 self.node_f[capped_v][:, A.NF_CAPMAX].min(initial=np.inf)))

    def materialise(self, k):
        """Configuration k as a FlatScene of its own (tables only, like FlatScene.from_arrays)."""
        d = self.flat.to_arrays()
        d["node_i"], d["node_f"], d["mon_f"] = d["node_i"].copy(), d["node_f"].copy(), d["mon_f"].copy()
        d["node_i"][self.nodes], d["node_f"][self.nodes], d["mon_f"][self.monitors] = self.node_i[k], self.node_f[k], self.mon_f[k]
        d["counts"][4] = int(_children(d["node_i"], d["node_f"]).max(initial=0))
        return type(self.flat).from_arrays(d)


class _MonitorPose:
    """A monitor's frame and size as one configuration left them: what SweepResult's statistics and monitor(k, m) read,
    copied because the pose methods move the live object in place."""

    def __init__(self, m):
        self.origin = np.array(m.origin, dtype=np.float64)
        self.transform_matrix = np.array(m.transform_matrix, dtype=np.float64)
        self.tangent_Y, self.tangent_Z, self.normal = (np.array(getattr(m, a), dtype=np.float64)
                                                       for a in ("tangent_Y", "tangent_Z", "normal"))
        self.width, self.height = m.width, m.height


class SweepScene:
    """A sweep over configurations of one table that differ only in the components and monitors listed in `vary`
    (tolerance and Monte Carlo studies, optimizer steps): the table is flattened once per distinct wavelength set and
    kept, so repeated sweeps do not re-flatten a large scene.

        sw = SweepScene(table, vary=[lens2, mon1])
        res = sw.trace(rays, configure, n_configs)      # a SweepResult

    `vary` holds objects of the table: components (leaves or groups, at any depth) and monitors of `table.monitors`.
    What can vary is what `FlatScene.refresh` can rewrite in place: poses, apertures, reflectivity, transmission, focal
    lengths, interact caps, monitor placement and size. A change of topology, of a material, of a polygon or
    composite-aperture record or of the cap slots raises ValueError; so does a varied component inside a lattice group
    (its lattice descriptor would have to be recomputed) and an object that is not in the table. Such sweeps go through
    `trace_sweep(tables)`, which flattens every configuration."""

    def __init__(self, table, vary):
        self.table, self.vary = table, list(vary)
        self._bases = {}   # wavelength set -> (FlatScene, varied components, node rows V, varied monitor indices, node_i[V])

    def _what(self, j):
        return f"vary[{j}] ({type(self.vary[j]).__name__})"

    def _base(self, wls):
        from .flatten import FlatScene

        key = None if wls is None else tuple(wls)
        if key in self._bases:
            return self._bases[key]
        flat = FlatScene(self.table.components, self.table.monitors, wavelengths_m=wls)
        mon_index = {id(m): i for i, m in enumerate(flat.monitors)}
        parents = flat._parents()
        comps, rows, mons = [], set(), []
        for j, obj in enumerate(self.vary):
            first = flat._node_of.get(id(obj))
            if first is None and id(obj) not in mon_index:
                raise ValueError(f"SweepScene: {self._what(j)} is not a component or monitor of the table")
            if id(obj) in mon_index:
                mons.append(mon_index[id(obj)])
            if first is None:
                continue
            up, p = [], parents.get(first, -1)
            while p >= 0:
                up.append(p)
                p = parents.get(p, -1)
            if any(flat.node_i[p, A.NI_GEOM] == A.G_GRID for p in up):
                raise ValueError(f"SweepScene: {self._what(j)} lies in a lattice group, whose lattice descriptor a move "
                                 "would change: trace such configurations with trace_sweep(tables)")
            if flat.refresh(obj) is None:
                raise ValueError(f"SweepScene: {self._what(j)} cannot be rewritten in place (it holds a lattice, a box "
                                 "hierarchy, a polygon or composite-aperture record): trace such configurations with "
                                 "trace_sweep(tables)")
            comps.append((j, obj))
            rows.update(range(first, int(flat.node_i[first, A.NI_SKIP])), up)
        V = np.array(sorted(rows), dtype=np.int32)
        base = self._bases[key] = (flat, comps, V, np.array(mons, dtype=np.int32), flat.node_i[V].copy())
        return base

    def trace(self, rays, configure, n_configs, perfomance_limit=None, record_hits=True, record_hist=False, engine=None,
              tracer=None, group=None, gather=False):
        """Trace `rays` (a RayBundle or a list of Ray) through `n_configs` configurations in one device call; returns a
        SweepResult whose `rows(k)`, `monitor(k, m)`, `stats()` and `row_values()` see configuration k's monitor
        placement.

        `configure(k)` puts the objects of `vary` into configuration k, with absolute values (the same configuration
        whatever ran before it); it runs for k = 0 .. n_configs - 1 in order, and after the call the table stands in
        configuration n_configs - 1. Limits, interact caps and record flags follow `trace_sweep`. `tracer(rows, rays,
        max_trace_num, ...)` defaults to the CUDA sweep, where `rows` is the SweepRows of the configurations; the CPU
        tests pass a stand-in. The starting interact counts of a list of Ray are the table's, read after each
        `configure(k)`.

        `group=` / `gather=` shard the configurations as in `trace_sweep`: rank r calls `configure(k)` only for its own
        configurations `shard_bounds(K, r, world)`, in order (and `configure(n_configs - 1)` once more at the end when
        another rank owns that one), and the frames of the varied monitors are exchanged so that `monitors[k][m]`
        holds every configuration's placement on every rank."""
        from .flatten import batch_wavelengths_m, trace_cap

        K = int(n_configs)
        if K < 1:
            raise ValueError("SweepScene.trace: n_configs must be >= 1")
        n, wl, unit, arrs, fam_ids = _rays(rays)
        wl_unit = unit if unit is not None else getattr(self.table, "unit", 1e-2)
        wls = None if wl is None else batch_wavelengths_m(wl, wl_unit)
        tracer = tracer or _device_sweep
        comps = None if fam_ids is None else (lambda: [list(self._base(wls)[0].capslots)] * K)
        if _sharded(group):
            from .dist import trace_sweep_sharded

            def prepare(k0, k1):
                rows, frames, caps0 = self._configurations(wls, configure, k0, k1, fam_ids)
                return rows, [{m: f for m, f in enumerate(fr) if isinstance(f, _MonitorPose)} for fr in frames], caps0

            live = list(self.table.monitors)
            out, frames = trace_sweep_sharded(K, n, rays, trace_cap(perfomance_limit), prepare,
                                              lambda poses: [[p.get(m, mon) for m, mon in enumerate(live)] for p in poses],
                                              "SweepScene.trace: configuration", tracer,
                                              group=None if group is True else group, gather=gather,
                                              record_hits=record_hits, record_hist=record_hist, engine=engine, unit=unit,
                                              arrs=arrs, fam_ids=fam_ids)
            if not out["shard"][0] <= K - 1 < out["shard"][1]:
                configure(K - 1)     # the documented end state: the table stands in the last configuration
            return SweepResult([self.table] * K, n, out, engine, monitors=frames, family_ids=fam_ids, cap_components=comps)
        rows, frames, caps0 = self._configurations(wls, configure, 0, K, fam_ids)
        limit = trace_cap(perfomance_limit)
        kw = {} if caps0 is None else {"caps0": caps0, "serial": caps_bind(caps0, arrs, rows.cap_min, limit)}
        out = tracer(rows, rays, limit, record_hits=record_hits, record_hist=record_hist, engine=engine, unit=unit,
                     arrs=arrs, **kw)
        return SweepResult([self.table] * K, n, out, engine, monitors=frames, family_ids=fam_ids, cap_components=comps)

    def abcd_matrix(self, m0, m1, rays, configure, n_configs, disp=1e-5, rot=1e-5, perfomance_limit=None, engine=None,
                    group=None):
        """`OpticalTable.calculate_abcd_matrix(mon0, mon1, rays)` of every configuration from two sweep traces; returns
        a SweepABCD (see `sweep_abcd_matrix`, whose preconditions and refusals hold here too).

        `m0`, `m1`: monitor indices or monitors of the table. `configure(k)` runs once for every k = 0 .. n_configs - 1,
        in order, as for `trace`; both bundles are traced through the configurations this builds. A configuration that
        moves mon0 raises ValueError before anything is traced."""
        from .flatten import batch_wavelengths_m, pack_rays, trace_cap

        what = "SweepScene.abcd_matrix"
        work, ids = _abcd_work(rays, group)
        K = int(n_configs)
        if K < 1:
            raise ValueError(f"{what}: n_configs must be >= 1")
        live = list(self.table.monitors)
        m0, m1 = _monitor_index(live, m0, what), _monitor_index(live, m1, what)
        arrs, _, unit = pack_rays(work)     # (both bundles have these wavelengths)
        wls = batch_wavelengths_m(arrs["wavelength"], unit)
        if self._base(wls)[0].n_capslots:
            raise NotImplementedError(f"{what}: interact-capped components are not supported (the table method's three "
                                      "traces carry their interact counts over from one to the next)")
        rows, frames, _ = self._configurations(wls, configure, 0, K)
        _check_mon0(frames, m0, what)
        return _abcd(rows, K, [self.table] * K, frames, m0, m1, work, ids, disp, rot, trace_cap(perfomance_limit),
                     engine, what)

    def _configurations(self, wls, configure, k0, k1, fam_ids=None):
        """configure(k) for k = k0 .. k1 - 1 in order: the SweepRows of those configurations, their monitor frames
        (a _MonitorPose snapshot for a varied monitor, the live monitor otherwise) and the `initial_counts` of the
        families `fam_ids`, read after each configure(k) (None without fam_ids or caps)."""
        from .flatten import monitor_record

        flat, comps, V, mons, ni0 = self._base(wls)
        K = k1 - k0
        node_i = np.empty((K, V.size, A.NI_STRIDE), dtype=np.int32)
        node_f = np.empty((K, V.size, A.NF_STRIDE), dtype=np.float64)
        mon_f = np.zeros((K, mons.size, A.MON_STRIDE), dtype=np.float64)
        cols = [c for c in range(A.NI_STRIDE) if c != A.NI_ORTHO]
        owner = {}
        for j, obj in comps:
            first = flat._node_of[id(obj)]
            owner.update({i: j for i in range(first, int(flat.node_i[first, A.NI_SKIP]))})
        frames, varied_mons, counts = [], set(mons.tolist()), []
        for c, k in enumerate(range(k0, k1)):
            configure(k)
            counts.append(initial_counts([flat.capslots], fam_ids))
            for j, obj in comps:
                if flat.refresh(obj) is None:
                    raise ValueError(f"SweepScene: configuration {k} changes {self._what(j)} in a way the scene cannot "
                                     "take in place (topology, a material, a polygon or composite-aperture record or its "
                                     "cap slots): trace such configurations with trace_sweep(tables)")
            node_i[c], node_f[c] = flat.node_i[V], flat.node_f[V]
            bad = np.argwhere(node_i[c][:, cols] != ni0[:, cols])
            if bad.size:
                i, col = int(V[bad[0][0]]), cols[int(bad[0][1])]
                raise ValueError(f"SweepScene: configuration {k} changes the {_NI_NAMES.get(col, f'node_i column {col}')} "
                                 f"of {self._what(owner[i]) if i in owner else f'node {i}'}: trace such configurations "
                                 "with trace_sweep(tables)")
            for w, m in enumerate(mons.tolist()):
                monitor_record(flat.monitors[m], mon_f[c, w])
            live = list(flat.monitors)
            frames.append([_MonitorPose(live[m]) if m in varied_mons else live[m] for m in range(len(live))])
        caps0 = np.concatenate(counts, axis=1) if counts and counts[0] is not None else None
        return SweepRows(flat, K, V, node_i, node_f, mons, mon_f), frames, caps0


class SweepABCD:
    """ABCD matrices of every configuration of a sweep (`sweep_abcd_matrix`, `SweepScene.abcd_matrix`).

    `M` [K, N, 2, 2]: M[k, r] is what `OpticalTable.calculate_abcd_matrix(mon0, mon1, rays)` returns for ray r on
    configuration k, rays in order of their ids `ids`; NaN where it is not defined. `row_counts` [K, N, 3]: the mon1 rows
    of ray r in the nominal, the shifted and the turned trace. `defined` [K, N]: exactly one row in each trace. `valid`
    [K]: every ray defined, the configurations for which the table method returns instead of raising. `traces`: the
    SweepResults of the two sweeps (the nominal and shifted bundle, 2N rays; the turned bundle, N rays), so that
    `traces[0].stats()` summarises the nominal trace at hand."""

    def __init__(self, M, row_counts, ids, traces):
        self.M, self.row_counts, self.ids, self.traces = M, row_counts, list(ids), tuple(traces)
        self.defined = (row_counts == 1).all(-1)
        self.valid = self.defined.all(-1)


def _abcd_work(rays, group):
    """calculate_abcd_matrix's `work` (copies of the rays, sorted by id) and the sorted ids, with its refusals."""
    if group is not None and group is not False:
        raise NotImplementedError("ABCD matrices of a sharded sweep (group=) are not supported: trace on one GPU")
    rays = list(rays)
    if not rays:
        raise ValueError("No rays to trace in ABCD calculation.")
    ids = [r._id for r in rays]
    if len(set(ids)) != len(rays):
        raise ValueError("Redundant ray ids in ABCD calculation.")
    order = np.argsort(ids)
    return [rays[i].copy() for i in order], [ids[i] for i in order]


def _abcd_bundle_a(work, mon0, disp):
    """The nominal rays and the same rays shifted by disp along mon0's tangent_Y: the one batch of
    `OpticalTable._abcd_first_two_traces`."""
    shift = mon0.tangent_Y * disp
    return work + [r.copy()._Translate(shift) for r in work]


def _abcd_bundle_b(work, mon0, pivots, disp, rot):
    """The shifted rays turned by rot about mon0's tangent_Z through their pivots (the third trace of
    calculate_abcd_matrix: the shift is not undone first)."""
    shift, axis = mon0.tangent_Y * disp, mon0.tangent_Z
    return [r.copy()._Translate(shift)._RotAround(axis, pivots[k], rot) for k, r in enumerate(work)]


def _monitor_index(monitors, m, what):
    if isinstance(m, (int, np.integer)):
        if not 0 <= int(m) < len(monitors):
            raise IndexError(f"{what}: monitor {int(m)} of {len(monitors)}")
        return int(m)
    for i, mon in enumerate(monitors):
        if mon is m:
            return i
    raise ValueError(f"{what}: {type(m).__name__} is not a monitor of the table")


def _check_mon0(monitors, m0, what):
    """Every configuration must place mon0 (origin, tangents, size) exactly as configuration 0 does: then the three
    bundles are the same in every configuration."""
    ref = monitors[0][m0]
    for k in range(1, len(monitors)):
        mon = monitors[k][m0]
        for a in ("origin", "tangent_Y", "tangent_Z", "width", "height"):
            if not np.array_equal(np.asarray(getattr(mon, a), np.float64), np.asarray(getattr(ref, a), np.float64)):
                raise ValueError(f"{what}: configuration {k} changes the {a} of mon0 (monitor {m0}): its ABCD bundles "
                                 "would differ from configuration 0's, and sweeps that need a bundle per configuration "
                                 "are not supported")


def _abcd(configs, K, tables, monitors, m0, m1, work, ids, disp, rot, limit, engine, what):
    """The device part of sweep_abcd_matrix / SweepScene.abcd_matrix: sweep A, the pivots, sweep B, the matrices."""
    from .analytics import _frame
    from .backend import Engine
    from .flatten import pack_rays

    engine = engine or Engine.get()
    N, mon0 = len(work), monitors[0][m0]
    arrs, _, unit = pack_rays(_abcd_bundle_a(work, mon0, disp))
    res_a = SweepResult(tables, 2 * N, _device_sweep(configs, None, limit, engine=engine, unit=unit, arrs=arrs), engine,
                        monitors=monitors)
    pivots, first_bad = engine.sweep_abcd_pivots(res_a.hits, N, K, m0)
    bad = int(first_bad.item())
    if bad >= 0:
        k, r = divmod(bad, N)
        if k == 0:
            raise ValueError(f"Rays at mon0 do not match the input rays. ({what}: ray id {ids[r]} has not exactly one "
                             "row at mon0 in configuration 0)")
        raise ValueError(f"{what}: in configuration {k}, ray id {ids[r]} does not cross mon0 exactly once at the point "
                         "it crosses it in configuration 0: its ABCD bundles would differ from configuration 0's, and "
                         "sweeps that need a bundle per configuration are not supported")
    arrs, _, unit = pack_rays(_abcd_bundle_b(work, mon0, pivots.cpu().numpy(), disp, rot))
    res_b = SweepResult(tables, N, _device_sweep(configs, None, limit, engine=engine, unit=unit, arrs=arrs), engine,
                        monitors=monitors)
    frames = (A.MonitorFrame * K)(*[_frame(monitors[k][m1]) for k in range(K)])
    abcd, counts = engine.sweep_abcd(res_a.hits, res_b.hits, N, K, m1, frames, disp, rot)
    return SweepABCD(abcd.cpu().numpy().reshape(K, N, 2, 2), counts.cpu().numpy(), ids, (res_a, res_b))


def sweep_abcd_matrix(tables, m0, m1, rays, disp=1e-5, rot=1e-5, perfomance_limit=None, engine=None, group=None):
    """`OpticalTable.calculate_abcd_matrix(mon0, mon1, rays)` of every table of `tables` (K configurations of one
    scene, as for `trace_sweep`) from two sweep traces; returns a SweepABCD.

    `m0`, `m1`: monitor indices, or monitors of tables[0]. The three bundles of the finite differences depend on the
    scene only through mon0 and what lies in front of it, so every configuration must place mon0 exactly as
    configuration 0 does and give every ray exactly one nominal mon0 hit point, bit-identical to configuration 0's
    (then the bundles are the same for all K): otherwise ValueError, naming the configuration (and ray). Like the table
    method: repeated ray ids raise ValueError; the pivots are configuration 0's mon0 hit points in monitor-local
    coordinates. Interact-capped components raise NotImplementedError (the table method's three traces share their
    counts), as does `group=`."""
    from .flatten import FlatScene, batch_wavelengths_m, pack_rays, trace_cap

    what = "sweep_abcd_matrix"
    work, ids = _abcd_work(rays, group)
    tables = list(tables)
    if not tables:
        raise ValueError(f"{what}: no tables")
    monitors = [list(t.monitors) for t in tables]
    m0, m1 = _monitor_index(monitors[0], m0, what), _monitor_index(monitors[0], m1, what)
    _check_mon0(monitors, m0, what)
    arrs, _, unit = pack_rays(work)     # (both bundles have these wavelengths)
    wls = batch_wavelengths_m(arrs["wavelength"], unit)
    flats = [FlatScene(t.components, t.monitors, wavelengths_m=wls) for t in tables]
    check_topology(flats)
    if flats[0].n_capslots:
        raise NotImplementedError(f"{what}: interact-capped components are not supported (the table method's three "
                                  "traces carry their interact counts over from one to the next)")
    return _abcd(flats, len(tables), tables, monitors, m0, m1, work, ids, disp, rot, trace_cap(perfomance_limit), engine,
                 what)
