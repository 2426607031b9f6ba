"""RayBundle: SoA ray batches that never become Python objects, and the tensor trace entry point.

A bundle is a dict of fp64 columns in the order of include/optb.h `optb_rays` (ox oy oz dx dy dz intensity
wavelength q_re q_im pathlength n_medium length). A column of length 1 is broadcast to every ray (ABI
`broadcast` mask), so a collimated monochromatic bundle is two real columns. Columns are numpy arrays or torch
tensors (pinned host or CUDA).

Synthetic bundles for the benchmarks are generated from the ray index with splitmix64, so any shard of any batch
can be produced independently and identically on every rank (SURVEY 8(d)).
"""
from __future__ import annotations

import math

import numpy as np

from . import _abi as A

SEED = 20261018
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x: np.ndarray) -> np.ndarray:
    """Counter-based hash: uint64 array -> uint64 array."""
    with np.errstate(over="ignore"):
        z = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
        return z ^ (z >> np.uint64(31))


def uniform01(index: np.ndarray, stream: int, seed: int = SEED) -> np.ndarray:
    """U[0,1) doubles from (seed, stream, index)."""
    with np.errstate(over="ignore"):
        key = splitmix64(index.astype(np.uint64) * np.uint64(4) + np.uint64(stream)) ^ splitmix64(np.uint64(seed) + np.zeros(1, np.uint64))
    return (splitmix64(key) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def gaussian_q(w0: float, wavelength: float, n: float = 1.0) -> complex:
    return (1j * n * math.pi * w0 ** 2) / wavelength


class RayBundle:
    def __init__(self, columns: dict, n: int):
        self.columns, self.n = columns, int(n)

    @classmethod
    def collimated_disc(cls, n, start=0, x0=-10.0, radius=3.0, direction=(1.0, 0.0, 0.0), wavelength=780e-7, w0=61e-4,
                        seed=SEED):
        """Rays start..start+n of an (in principle endless) collimated bundle filling a disc uniformly."""
        idx = np.arange(start, start + n, dtype=np.uint64)
        rr = radius * np.sqrt(uniform01(idx, 0, seed))
        th = 2.0 * math.pi * uniform01(idx, 1, seed)
        q = gaussian_q(w0, wavelength) if w0 else 0j
        d = np.asarray(direction, float) / np.linalg.norm(direction)
        one = lambda v: np.array([v], dtype=np.float64)
        cols = {"ox": one(x0), "oy": rr * np.cos(th), "oz": rr * np.sin(th), "dx": one(d[0]), "dy": one(d[1]),
                "dz": one(d[2]), "intensity": one(1.0), "wavelength": one(wavelength), "q_re": one(q.real),
                "q_im": one(q.imag), "pathlength": one(0.0), "n_medium": one(1.0), "length": None}
        b = cls(cols, n)
        b.has_q = bool(w0)
        return b

    def slice(self, lo: int, hi: int) -> "RayBundle":
        """Rays [lo, hi) as a bundle of their own (broadcast columns stay single values; views, no copies)."""
        cols = {k: (c if c is None or np.asarray(c).size == 1 else c[lo:hi]) for k, c in self.columns.items()}
        b = RayBundle(cols, hi - lo)
        if hasattr(self, "has_q"):
            b.has_q = self.has_q
        return b

    def materialise(self) -> dict:
        """Full-length numpy columns (+ flags / family) for the oracle or for object-level comparisons."""
        out = {}
        for k in A.RAY_F64:
            c = self.columns.get(k)
            if c is None:
                out[k] = np.full(self.n, np.inf)
            else:
                c = np.asarray(c, dtype=np.float64)
                out[k] = np.ascontiguousarray(np.broadcast_to(c, (self.n,)) if c.size == 1 else c)
        flags = A.RF_ALIVE | (A.RF_HASQ if getattr(self, "has_q", True) else 0)
        out["flags"] = np.full(self.n, flags, dtype=np.uint32)
        out["family"] = np.arange(self.n, dtype=np.int32)
        return out

    def to_torch(self, device=None, pin=False):
        """Columns as torch tensors: on `device` (CUDA) or in pinned host memory."""
        import torch

        t = {}
        for k, c in self.columns.items():
            if c is None:
                continue
            x = torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64))
            if device is not None:
                x = x.to(device)
            elif pin:
                x = x.pin_memory()
            t[k] = x
        if not getattr(self, "has_q", True):
            f = torch.full((self.n,), A.RF_ALIVE, dtype=torch.int32)
            t["flags"] = f.to(device) if device is not None else (f.pin_memory() if pin else f)
        return t


HIT_COLUMNS_ALL = A.HIT_I32 + A.HIT_U32 + A.HIT_F64


class DeviceTrace:
    """Reusable device-side state for repeated traces of same-shaped bundles through one scene: scene tables,
    result buffers and workspace are allocated once; `run` only enqueues kernels. With `configs` (the FlatScenes of a
    sweep, `flat` = configs[0], or a SweepRows, `flat` = its base) the scene is a sweep scene and one run traces the
    bundle through every configuration.

    `cap_counts` (a sweep of Ray objects whose interact caps can bind: [n_capslots, n_configs * n_families], column
    k * n_families + f = family f in configuration k) runs the family-serial sweep: every run starts from these counts,
    and the rays must carry a `family` column (< n_families)."""

    def __init__(self, engine, flat, n_rays, hit_capacity, seg_capacity=0, hit_columns=HIT_COLUMNS_ALL,
                 max_trace_num=2000, unit=1e-2, record_hist=False, chain_len=0, flag_ambiguity=False, configs=None,
                 cap_counts=None, n_families=None):
        import torch

        self.engine, self.flat, self.torch = engine, flat, torch
        self.scene = engine.upload(flat) if configs is None else engine.upload_sweep(configs)
        n_roots = n_rays * self.scene.n_configs
        serial = cap_counts is not None and flat.n_capslots > 0
        self.res, self.t = engine.alloc_result(self.scene, seg_capacity, hit_capacity,
                                               self.scene.n_configs * n_families if serial else n_roots,
                                               hit_columns=tuple(hit_columns) + (() if "hit_key" in hit_columns else ("hit_monitor",)))
        self._caps0 = torch.from_numpy(np.ascontiguousarray(cap_counts, dtype=np.int32)).to(self.t["cap_counts"].device) if serial else None
        if flag_ambiguity:
            self.t["root_flags"] = torch.zeros(max(int(n_rays), 1), dtype=torch.int32, device=f"cuda:{engine.device}")
            self.res.root_flags = self.t["root_flags"].data_ptr()
        slack = 0
        if flat.n_capslots and not serial:
            # a bundle ray is its own `_id` family starting from zero counts: a cap can only bind if it is
            # smaller than the pop budget. Binding caps need Ray objects (OpticalTable.ray_tracing, trace_sweep).
            if min(f.cap_min for f in self.scene.configs) < max_trace_num:
                raise NotImplementedError("bundle traces need max_interact_count >= max_trace_num on every capped "
                                          "component (a sweep of Ray objects with ids lifts this)")
            slack = 1
        self.prm = engine.make_params(max_trace_num, unit, seg_capacity > 0, hit_capacity > 0, record_hist, chain_len,
                                      n_families if serial else n_roots, slack, flag_ambiguity)
        self.hit_columns = tuple(k for k in HIT_COLUMNS_ALL + ("hit_key",) if k in self.t)

    def run(self, rays_t, max_live=None):
        if self._caps0 is not None:
            self.t["cap_counts"].copy_(self._caps0)   # every attempt starts from the initial counts
        elif self.flat.n_capslots:
            self.t["cap_counts"].zero_()  # a bundle is a fresh set of ray ids every time
        self.engine.trace_device(self.scene, rays_t, self.prm, self.res, max_live)

    def capture(self, rays_t, max_live=None):
        """Capture one `run` on `rays_t` into a CUDA graph (scenes that cannot split rays: their whole bounce loop
        is a fixed sequence of launches). `replay()` then re-issues it with one driver call; the ray columns, the
        result buffers and the scene blob are read at replay time, so the caller may overwrite the rays in place
        and move components with `scene.update_nodes(flat.refresh(component))` between replays (SURVEY 8f item 3)."""
        from .backend import runs_wavefront

        torch = self.torch
        if runs_wavefront(self.scene.configs, self.prm):
            raise NotImplementedError("CUDA-graph replay needs a trace without host round trips (backend.runs_wavefront)")
        self.run(rays_t, max_live)          # warm-up: workspace and kernel attributes exist before the capture
        torch.cuda.synchronize()
        self._graph_rays = rays_t
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self.run(rays_t, max_live)
        return self

    def replay(self):
        self._graph.replay()

    def close(self):
        self.torch.cuda.synchronize()
        self._graph = None
        self.scene.close()

    def counters(self):
        return self.t["counters"].cpu().numpy()

    def hit_row_bytes(self):
        return sum(self.t[k].element_size() for k in self.hit_columns)


def trace_bundle(table, bundle: RayBundle, perfomance_limit=None, record_hits=True, record_hist=False,
                 hit_capacity=None, engine=None, max_live=None, hit_columns=HIT_COLUMNS_ALL):
    """Trace a RayBundle through `table` entirely on the device; returns a dict of CUDA tensors (hit columns
    trimmed to the rows produced, histograms, counters as numpy). Rows are in device append order and carry
    their (root, pop) key."""
    from .backend import Engine
    from .flatten import FlatScene, batch_wavelengths_m, trace_cap

    engine = engine or Engine.get()
    wl = bundle.columns.get("wavelength")
    flat = FlatScene(table.components, table.monitors,
                     wavelengths_m=None if wl is None else batch_wavelengths_m(wl, getattr(table, "unit", 1e-2)))
    cap = int(hit_capacity if hit_capacity is not None else bundle.n * max(flat.n_monitors, 1) * 2) if record_hits else 0
    limit = trace_cap(perfomance_limit)
    rays_t = bundle.to_torch(device=f"cuda:{engine.device}")
    dt, cnt = run_to_fit(lambda c: DeviceTrace(engine, flat, bundle.n, c, max_trace_num=limit, record_hist=record_hist,
                                               hit_columns=hit_columns),
                         rays_t, bundle.n, limit, cap, hit_capacity is not None, max_live)
    nh = int(cnt[A.C_HITS]) if record_hits else 0
    out = {k: dt.t[k][:nh] for k in dt.hit_columns}
    out["hist_y"], out["hist_yz"], out["counters"] = dt.t["hist_y"], dt.t["hist_yz"], cnt
    return out


def run_to_fit(make, rays_t, n_roots, limit, cap, fixed_cap=False, max_live=None):
    """Trace with `make(hit_capacity)` (a DeviceTrace) until the run fits; returns (DeviceTrace, counters).

    Live-ray budget of a splitting scene: grow on overflow towards the bound 2 n max_trace_num (a root pops at most
    max_trace_num rays and each pop queues at most two); row capacity (unless `fixed_cap`): the counters keep counting
    past it, so an overflowing attempt is repeated once with the exact size."""
    live, bound = max_live, max(2 * n_roots * max(limit, 1), 1024)
    resized = False
    while True:
        dt = make(cap)
        dt.run(rays_t, live)
        cnt = dt.counters()
        st = int(cnt[A.C_STATUS])
        cur = live if live is not None else max(4 * n_roots, 1024)
        if st & A.ST_WORK_OVERFLOW and cur < bound:
            live = min(4 * cur, bound)
        elif st & A.ST_HIT_OVERFLOW and not resized and not fixed_cap:
            cap, resized = int(cnt[A.C_HITS]), True
        else:
            break
        dt.scene.close()
    dt.engine._raise_status(cnt)
    return dt, cnt
