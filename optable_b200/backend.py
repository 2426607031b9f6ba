"""ctypes binding of the C-ABI CUDA library (include/optb.h) + the device-side trace driver.

PyTorch is plumbing here: it owns device memory (tensors whose data_ptr() goes through the ABI) and the
CUDA stream. All arithmetic of the bounce loop is in optable_b200/liboptb.so. There is no CPU fallback:
if the extension is missing or no CUDA device is present, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _abi as A
from .flatten import FlatScene

_SO = os.environ.get("OPTB_LIB_PATH") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "liboptb.so")
_lib = None


class BackendError(RuntimeError):
    pass


def lib():
    """Load liboptb.so (built in-tree by optable_b200.build). Fails loudly when absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise BackendError(f"{_SO} not found: build it with `python -m optable_b200.build` (no CPU fallback exists)")
        L = C.CDLL(_SO)
        L.optb_abi_version.restype = C.c_int
        L.optb_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.optb_ctx_destroy.argtypes = [C.c_void_p]
        L.optb_last_error.restype = C.c_char_p
        L.optb_last_error.argtypes = [C.c_void_p]
        L.optb_scene_upload.argtypes = [C.c_void_p, C.POINTER(A.SceneDesc), C.POINTER(C.c_void_p)]
        L.optb_scene_upload_sweep.argtypes = [C.c_void_p, C.POINTER(A.SceneDesc), C.c_int32, C.POINTER(C.c_void_p)]
        L.optb_scene_upload_sweep_rows.argtypes = [C.c_void_p, C.POINTER(A.SceneDesc), C.c_int32, C.c_void_p, C.c_int32,
                                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                                   C.POINTER(C.c_void_p)]
        L.optb_scene_destroy.argtypes = [C.c_void_p, C.c_void_p]
        L.optb_workspace_bytes.restype = C.c_int64
        L.optb_workspace_bytes.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
        L.optb_trace.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(A.Rays), C.POINTER(A.Params), C.POINTER(A.Result),
                                 C.c_void_p, C.c_int64, C.c_void_p]
        L.optb_trace_host.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(A.Rays), C.POINTER(A.Params), C.POINTER(A.Result)]
        if hasattr(L, "optb_trace_plan"):   # (a library built before the entry point still traces)
            L.optb_trace_plan.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(A.Rays), C.POINTER(A.Params), C.POINTER(C.c_int64)]
        L.optb_measure_fp64_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.optb_sort_workspace_bytes.restype = C.c_int64
        L.optb_sort_workspace_bytes.argtypes = [C.c_int64]
        L.optb_sort_rows.argtypes = [C.c_void_p, C.POINTER(A.Result), C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
        L.optb_monitor_stats_grouped_workspace_bytes.restype = C.c_int64
        L.optb_monitor_stats_grouped_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
        L.optb_monitor_stats_grouped.argtypes = [C.c_void_p, C.POINTER(A.Result), C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                                 C.c_int32, C.c_void_p, C.c_void_p] + [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]
        L.optb_sweep_abcd_workspace_bytes.restype = C.c_int64
        L.optb_sweep_abcd_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
        L.optb_sweep_abcd_pivots.argtypes = [C.c_void_p, C.POINTER(A.Result), C.c_int64, C.c_int64, C.c_int32, C.c_int32,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.optb_sweep_abcd.argtypes = [C.c_void_p, C.POINTER(A.Result), C.c_int64, C.POINTER(A.Result), C.c_int64, C.c_int64,
                                      C.c_int32, C.c_int32, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int64, C.c_void_p]
        if L.optb_abi_version() != A.ABI_VERSION:
            raise BackendError("liboptb.so ABI version does not match optable_b200._abi")
        _lib = L
    return _lib


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise BackendError("no CUDA device: optable_b200 has no CPU fallback")
    return torch


_RESULT_DTYPES = None


def _result_fields(torch):
    global _RESULT_DTYPES
    if _RESULT_DTYPES is None:
        d = {}
        for k in A.SEG_F64 + A.HIT_F64:
            d[k] = torch.float64
        for k in A.SEG_U32 + A.HIT_U32:
            d[k] = torch.int32  # bit pattern of uint32; viewed as uint32 on the host
        for k in A.SEG_I32 + A.HIT_I32:
            d[k] = torch.int32
        _RESULT_DTYPES = d
    return _RESULT_DTYPES


def runs_wavefront(flats, params: A.Params) -> bool:
    """Whether a trace of the scene made of `flats` (its configurations) with `params` can run the wavefront path (or
    the family-serial one): it then needs workspace for the live rays of every generation and synchronises with the
    host once per generation, so it cannot be captured into a CUDA graph. Splitting scenes, capped scenes, pass-through
    leaves, chain_len > 0 and the two diagnostics modes do."""
    return bool(params.chain_len > 0 or params.flag_ambiguity or params.reference_roots
                or any(f.max_children > 1 or f.n_capslots > 0 or f.has_pass for f in flats))


def caps_can_bind(count_max, fam_size, cap_min, max_trace_num) -> bool:
    """Whether an interact cap can bind in a trace: a family's count grows by at most one per pop of each of its initial
    rays, so a cap binds only if the largest initial count plus max_trace_num pops of the largest family can exceed the
    smallest cap. Traces where it can run family-serially (params.caps_slack = 0)."""
    return not int(count_max) + int(max_trace_num) * int(fam_size) <= cap_min


class Scene:
    """Device-resident scene tables (optb_scene handle). With `configs` it is a sweep scene, and every trace runs its
    bundle through all `n_configs` configurations: `configs` is a list of FlatScene of one topology
    (optb_scene_upload_sweep; `flat` is then configs[0]) or a sweep.SweepRows, a base scene plus the rows that differ
    (optb_scene_upload_sweep_rows; `flat` is then its base). `self.configs` holds what runs_wavefront and the cap check
    read: the FlatScenes, or the one SweepRows, whose properties cover all its configurations."""

    def __init__(self, engine, flat: FlatScene, configs=None):
        from .sweep import SweepRows

        self.engine, self.flat = engine, flat
        rows = configs if isinstance(configs, SweepRows) else None
        self.configs = [rows] if rows is not None else list(configs) if configs is not None else [flat]
        self.n_configs = rows.n_configs if rows is not None else len(self.configs)
        self.sweep = configs is not None
        self.max_children = max(f.max_children for f in self.configs)
        h = C.c_void_p()
        if rows is not None:
            desc = flat.desc()
            engine._check(lib().optb_scene_upload_sweep_rows(
                engine._ctx, C.byref(desc), rows.n_configs, rows.nodes.ctypes.data, rows.nodes.size, rows.node_f.ctypes.data,
                rows.node_i.ctypes.data, rows.monitors.ctypes.data, rows.monitors.size, rows.mon_f.ctypes.data, C.byref(h)))
        elif self.sweep:
            descs = (A.SceneDesc * self.n_configs)(*[f.desc() for f in self.configs])   # (the arrays stay alive in configs)
            engine._check(lib().optb_scene_upload_sweep(engine._ctx, descs, self.n_configs, C.byref(h)))
        else:
            desc = flat.desc()
            engine._check(lib().optb_scene_upload(engine._ctx, C.byref(desc), C.byref(h)))
        self._h = h

    def update_nodes(self, nodes, stream=None):
        """Send the rows of `nodes` (FlatScene.refresh's return value) of the already updated `self.flat` tables to
        the device copy of the scene (optb_scene_update_nodes): the handle, and CUDA graphs captured over it, stay valid."""
        L = lib()
        L.optb_scene_update_nodes.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(A.SceneDesc), C.c_void_p, C.c_int32, C.c_void_p]
        idx = np.ascontiguousarray(nodes, dtype=np.int32)
        desc = self.flat.desc()
        st = self.engine.torch.cuda.current_stream(self.engine.device).cuda_stream if stream is None else stream
        self.engine._check(L.optb_scene_update_nodes(self.engine._ctx, self._h, C.byref(desc), idx.ctypes.data, len(idx), C.c_void_p(st)))

    def close(self):
        if self._h:
            lib().optb_scene_destroy(self.engine._ctx, self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    """One context per CUDA device (optb_ctx)."""

    _cache = {}

    @classmethod
    def get(cls, device=None):
        torch = _torch()
        dev = torch.cuda.current_device() if device is None else int(device)
        if dev not in cls._cache:
            cls._cache[dev] = cls(dev)
        return cls._cache[dev]

    def __init__(self, device=0):
        self.torch = _torch()
        self.device = int(device)
        self._ctx = C.c_void_p()
        rc = lib().optb_ctx_create(self.device, C.byref(self._ctx))
        if rc != 0:
            raise BackendError(f"optb_ctx_create({device}) failed: {rc}")
        self._workspace = None

    def _check(self, rc):
        if rc != 0:
            raise BackendError(f"liboptb error {rc}: {lib().optb_last_error(self._ctx).decode()}")

    def upload(self, flat: FlatScene) -> Scene:
        return Scene(self, flat)

    def upload_sweep(self, configs) -> Scene:
        """One sweep scene from the FlatScenes of K configurations with the same topology (optb_scene_upload_sweep), or
        from a sweep.SweepRows (optb_scene_upload_sweep_rows)."""
        from .sweep import SweepRows

        return Scene(self, configs.flat if isinstance(configs, SweepRows) else configs[0], configs=configs)

    def fp64_peak_tflops(self) -> float:
        v = C.c_double(0)
        self._check(lib().optb_measure_fp64_peak(self._ctx, C.byref(v)))
        return v.value

    # -- device buffers --------------------------------------------------------------------------
    def _ws(self, nbytes):
        torch = self.torch
        if self._workspace is None or self._workspace.numel() < nbytes:
            self._workspace = None
            self._workspace = torch.empty(int(nbytes), dtype=torch.uint8, device=f"cuda:{self.device}")
        return self._workspace

    def rays_to_device(self, arrs):
        """dict of numpy arrays (flatten.pack_rays) -> dict of CUDA tensors (two transfers: the fp64 columns as
        one block, flags + family as another)."""
        torch = self.torch
        dev = f"cuda:{self.device}"
        n = len(arrs["ox"])
        f = np.empty((len(A.RAY_F64), n), dtype=np.float64)
        for j, k in enumerate(A.RAY_F64):
            f[j] = arrs[k]
        i = np.empty((2, n), dtype=np.int32)
        i[0] = np.ascontiguousarray(arrs["flags"]).view(np.int32)
        i[1] = arrs["family"]
        fd, idev = torch.from_numpy(f).to(dev), torch.from_numpy(i).to(dev)
        out = {k: fd[j] for j, k in enumerate(A.RAY_F64)}
        out["flags"], out["family"] = idev[0], idev[1]
        return out

    @staticmethod
    def _rays_struct(t, n=None):
        s = A.Rays()
        s.n = int(max(t[k].numel() for k in A.RAY_F64 if t.get(k) is not None) if n is None else n)
        s.broadcast = 0
        for bit, k in enumerate(A.RAY_F64):
            v = t.get(k)
            setattr(s, k, None if v is None else v.data_ptr())
            if v is not None and v.numel() == 1 and s.n != 1:
                s.broadcast |= 1 << bit
        for k in ("flags", "family"):
            v = t.get(k)
            setattr(s, k, None if v is None else v.data_ptr())
        return s

    SLAB_LIMIT = 4 << 20

    def alloc_result(self, scene: Scene, seg_capacity, hit_capacity, n_families, cap_counts=None, slab=False,
                     hit_columns=None):
        """Device buffers for one trace + the optb_result that points at them. With `slab`, small results are
        carved out of ONE zeroed buffer (returned as `result._slab`, layout in `result._layout`) so that the
        whole result comes back with a single device-to-host copy."""
        torch = self.torch
        dev = f"cuda:{self.device}"
        dt = _result_fields(torch)
        nm = max(scene.flat.n_monitors, 1) * scene.n_configs   # a sweep: [n_configs][n_monitors] histograms
        spec = [(k, dt[k], (int(seg_capacity),)) for k in A.SEG_F64 + A.SEG_U32 + A.SEG_I32]
        # `hit_columns`: the monitor-row columns the caller wants (default: all but the packed key); the others stay
        # NULL in the result struct: neither allocated nor written
        want = set(A.HIT_I32 + A.HIT_U32 + A.HIT_F64) if hit_columns is None else set(hit_columns)
        spec += [(k, dt[k], (int(hit_capacity),)) for k in A.HIT_I32 + A.HIT_U32 + A.HIT_F64 if k in want]
        if "hit_key" in want:
            spec += [("hit_key", torch.int64, (int(hit_capacity),))]
        spec += [("hist_y", torch.int64, (nm, A.HIST_BINS)), ("hist_yz", torch.int64, (nm, A.HIST_BINS, A.HIST_BINS)),
                 ("cap_counts", torch.int32, (max(scene.flat.n_capslots, 1), max(int(n_families), 1))),
                 ("counters", torch.int64, (A.C_COUNT,))]
        size = {torch.float64: 8, torch.int64: 8, torch.int32: 4}
        layout, total = {}, 0
        for k, d, shape in spec:
            nbytes = size[d] * int(np.prod(shape))
            layout[k] = (total, nbytes, d, shape)
            total += (nbytes + 15) & ~15
        t = {}
        r = A.Result()
        if slab and total <= self.SLAB_LIMIT:
            buf = torch.zeros(total, dtype=torch.uint8, device=dev)
            base = buf.data_ptr()
            for k, (off, nbytes, d, shape) in layout.items():
                setattr(r, k, base + off)
            off, nbytes, d, shape = layout["cap_counts"]
            t["cap_counts"] = buf[off:off + nbytes].view(d).view(shape)
            r._slab, r._layout = buf, layout
        else:
            for k, d, shape in spec:
                zero = k in ("hist_y", "hist_yz", "cap_counts", "counters")
                t[k] = (torch.zeros if zero else torch.empty)(shape, dtype=d, device=dev)
            r._slab = None
        if cap_counts is not None:
            t["cap_counts"].copy_(torch.from_numpy(np.ascontiguousarray(cap_counts, dtype=np.int32)))
        r.seg_capacity, r.hit_capacity = int(seg_capacity), int(hit_capacity)
        if r._slab is None:
            for k, v in t.items():
                setattr(r, k, v.data_ptr())
        return r, t

    @staticmethod
    def make_params(max_trace_num=2000, unit=1e-2, record_segments=True, record_hits=True, record_hist=False,
                    chain_len=0, n_families=1, caps_slack=0, flag_ambiguity=False, reference_roots=False):
        p = A.Params()
        p.max_trace_num, p.unit = int(max_trace_num), float(unit)
        p.record_segments, p.record_hits, p.record_hist = int(record_segments), int(record_hits), int(record_hist)
        p.chain_len, p.n_families, p.caps_slack = int(chain_len), int(n_families), int(caps_slack)
        p.flag_ambiguity = int(bool(flag_ambiguity))
        p.reference_roots = int(bool(reference_roots))
        return p

    def trace_device(self, scene: Scene, rays_t, params: A.Params, result: A.Result, max_live=None, stream=None):
        """Enqueue optb_trace on tensors already resident on the device. Asynchronous for scenes that cannot
        split rays; returns after the last generation otherwise."""
        torch = self.torch
        rs = self._rays_struct(rays_t)
        n = int(rs.n) * scene.n_configs   # roots
        live = 0 if not runs_wavefront(scene.configs, params) else int(max_live if max_live is not None else max(4 * n, 1024))
        if scene.flat.n_capslots and not params.caps_slack:  # family-serial mode: total FIFO entries over all families
            live = max(live, min(64 * max(n, 16), n * (int(params.max_trace_num) + 2)))
        nbytes = lib().optb_workspace_bytes(scene._h, int(rs.n), live)
        ws = self._ws(nbytes)
        st = torch.cuda.current_stream(self.device).cuda_stream if stream is None else stream
        self._check(lib().optb_trace(self._ctx, scene._h, C.byref(rs), C.byref(params), C.byref(result),
                                     ws.data_ptr(), int(ws.numel()), C.c_void_p(st)))

    def trace_host(self, scene: Scene, rays_struct: A.Rays, params: A.Params, result: A.Result):
        """optb_trace_host: host buffers in, host buffers out (copies inside the call)."""
        self._check(lib().optb_trace_host(self._ctx, scene._h, C.byref(rays_struct), C.byref(params), C.byref(result)))

    def _arrays_params(self, scene: Scene, arrs, max_trace_num=2000, unit=1e-2, record_segments=True, record_hits=True,
                       record_hist=False, n_families=None, cap_counts=None, chain_len=0, flag_ambiguity=False,
                       reference_roots=False):
        """optb_params of trace_arrays for a packed batch, and the initial interact-count table (None without caps)."""
        n = len(arrs["ox"])
        if n_families is None:
            n_families = int(arrs["family"].max()) + 1 if n else 1
        flat = scene.flat
        caps0, slack = None, 0
        if flat.n_capslots:
            caps0 = np.zeros((flat.n_capslots, n_families), np.int32) if cap_counts is None else np.array(cap_counts, np.int32)
            fam_size = np.bincount(arrs["family"], minlength=n_families).max() if n else 0
            capmax = flat.node_f[flat.node_i[:, A.NI_CAPSLOT] >= 0, A.NF_CAPMAX].min()
            slack = int(not caps_can_bind(caps0.max(), fam_size, capmax, max_trace_num))
        prm = self.make_params(max_trace_num, unit, record_segments, record_hits, record_hist, chain_len, n_families, slack,
                               flag_ambiguity, reference_roots)
        return prm, caps0

    def trace_plan(self, scene: Scene, arrs, **params):
        """The launch plan (optb_trace_plan) of `trace_arrays(scene, arrs, **params)`: a dict of the variant bits
        (`bits`, OPTB_PLAN_*), `blob` bytes, `dynamic` and `static` shared memory of the kernel, and the device's
        `optin` limit. Nothing is traced."""
        prm, _ = self._arrays_params(scene, arrs, **params)
        rs = A.Rays()
        rs.n = len(arrs["ox"])
        family = np.ascontiguousarray(arrs["family"], dtype=np.int32)
        # (trace_arrays always passes the family column; the plan only tests it is set). A sweep's roots are their own
        # families unless its caps can bind: that sweep runs family-serially, with the family column.
        if not scene.sweep or (scene.flat.n_capslots and not prm.caps_slack):
            rs.family = family.ctypes.data
        out = (C.c_int64 * 5)()
        self._check(lib().optb_trace_plan(self._ctx, scene._h, C.byref(rs), C.byref(prm), out))
        return dict(zip(("bits", "blob", "dynamic", "static", "optin"), (int(v) for v in out)))

    # -- convenience: exact-size traced result on the host, in reference order -------------------------
    def trace_arrays(self, scene: Scene, arrs, max_trace_num=2000, unit=1e-2, record_segments=True, record_hits=True,
                     record_hist=False, n_families=None, cap_counts=None, chain_len=0, max_live=None, flag_ambiguity=False,
                     reference_roots=False):
        """Trace a packed ray batch and return numpy result arrays trimmed and sorted to reference order
        (segments by (root, pop); monitor rows by (root, monitor, pop))."""
        torch = self.torch
        n = len(arrs["ox"])
        prm, caps0 = self._arrays_params(scene, arrs, max_trace_num, unit, record_segments, record_hits, record_hist,
                                         n_families, cap_counts, chain_len, flag_ambiguity, reference_roots)
        n_families = prm.n_families
        rays_t = self.rays_to_device(arrs)
        flat = scene.flat
        # Row counts are only known after the trace. First try with capacities guessed from the batch; the
        # counters keep counting past the capacity, so an overflowing attempt is repeated once with exact sizes
        # (interact counts restart from caps0: every attempt gets a fresh table).
        pops_max = n * int(max_trace_num)
        nseg = min(pops_max, 8 * n + 1024) if record_segments else 0
        nhit = min(pops_max * flat.n_monitors, 8 * n + 1024) if record_hits else 0
        root_flags = torch.zeros(max(n, 1), dtype=torch.int32, device=f"cuda:{self.device}") if flag_ambiguity else None
        np_dt = {torch.float64: np.float64, torch.int64: np.int64, torch.int32: np.int32}
        # The live ray set of a splitting scene is not known in advance either: a root pops at most max_trace_num rays
        # and every pop queues at most two, so 2 n max_trace_num live rays always suffice; grow towards that bound.
        live_bound = max(2 * n * max(int(max_trace_num), 1), 1024)
        live = max_live
        retried_rows = False
        while True:
            res, t = self.alloc_result(scene, nseg, nhit, n_families, caps0, slab=True)
            if root_flags is not None:
                res.root_flags = root_flags.data_ptr()
            self.trace_device(scene, rays_t, prm, res, live)
            host = None
            if res._slab is not None:  # everything in one copy (synchronises)
                raw = res._slab.cpu().numpy()
                host = {k: raw[off:off + nb].view(np_dt[d]).reshape(shape) for k, (off, nb, d, shape) in res._layout.items()}
                cnt = host["counters"]
            else:
                cnt = t["counters"].cpu().numpy()
            st = int(cnt[A.C_STATUS])
            if st & A.ST_WORK_OVERFLOW:
                cur = live if live is not None else max(4 * n, 1024)
                if cur >= live_bound:
                    self._raise_status(cnt)
                live = min(4 * cur, live_bound)
                continue
            if not st & (A.ST_SEG_OVERFLOW | A.ST_HIT_OVERFLOW) or retried_rows:
                break
            retried_rows = True
            nseg = int(cnt[A.C_SEGMENTS]) if record_segments else 0
            nhit = int(cnt[A.C_HITS]) if record_hits else 0
        self._raise_status(cnt)
        nseg = int(cnt[A.C_SEGMENTS]) if record_segments else 0
        nhit = int(cnt[A.C_HITS]) if record_hits else 0
        trim = {k: nseg for k in A.SEG_F64 + A.SEG_U32 + A.SEG_I32}
        trim.update({k: nhit for k in A.HIT_I32 + A.HIT_U32 + A.HIT_F64})
        if host is not None:
            out = {k: (v[:trim[k]] if k in trim else v) for k, v in host.items()}
            presorted = False
        else:
            # large results: put the rows into reference order on the device (one 64-bit key per row), then copy
            presorted = self._sort_rows_on_device(res, nseg, nhit, int(max_trace_num), flat.n_monitors)
            out = {k: (v[:trim[k]] if k in trim else v).cpu().numpy() for k, v in t.items()}
        for k in A.SEG_U32 + A.HIT_U32:
            out[k] = out[k].view(np.uint32)
        if root_flags is not None:  # OPTB_AMB_* bits per initial ray (SURVEY A.9), evaluated in-kernel
            out["root_flags"] = root_flags.cpu().numpy().view(np.uint32)[:n]
        self._raise_status(out["counters"])
        if presorted:
            return out
        if record_segments and nseg:
            order = np.lexsort((out["seg_pop"], out["seg_root"]))
            for k in A.SEG_F64 + A.SEG_U32 + A.SEG_I32:
                out[k] = out[k][order]
        if record_hits and nhit:
            order = np.lexsort((out["hit_pop"], out["hit_monitor"], out["hit_root"]))
            for k in A.HIT_I32 + A.HIT_U32 + A.HIT_F64:
                out[k] = out[k][order]
        return out

    def _sort_rows_on_device(self, res, nseg, nhit, max_trace_num, n_monitors):
        """Reorder the row columns of `res` (device buffers) to (root, pop) / (root, monitor, pop) with the library's
        own sort (optb_sort_rows: one packed 64-bit key per row + a gather per column). Returns False when the key
        would not fit (pop >= 2^24 or > 256 monitors): the caller then sorts on the host."""
        if int(max_trace_num) > (1 << 24) or int(n_monitors) > 256:
            return False
        n = max(int(nseg), int(nhit))
        if n <= 1:
            return True
        nbytes = lib().optb_sort_workspace_bytes(n)
        ws = self._ws(nbytes)
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(lib().optb_sort_rows(self._ctx, C.byref(res), int(nseg), int(nhit), ws.data_ptr(), int(ws.numel()), C.c_void_p(st)))
        return True

    def monitor_stats_grouped(self, cols, frames, n_configs, n_monitors, rays_per_config=0):
        """optb_monitor_stats_grouped over every row of `cols` (the CUDA hit columns of one result) on the current
        stream. `frames`: a ctypes array of n_configs * n_monitors MonitorFrame, group k * n_monitors + m at its place.
        Returns the device tensors stats [n_configs * n_monitors, OPTB_MS_STRIDE] and per-row values [5, n] (y, z, tY,
        tZ, waist distance in each row's own frame; the last three rows are unwritten without hit_dx..dz / hit_q_re)."""
        torch = self.torch
        dev = f"cuda:{self.device}"
        n, G = int(cols["hit_px"].numel()), int(n_configs) * int(n_monitors)
        res = self._hit_result(cols)
        frames_dev = torch.frombuffer(bytearray(frames), dtype=torch.uint8).to(dev)
        stats = torch.empty((G, A.MS_STRIDE), dtype=torch.float64, device=dev)
        per_row = torch.empty((5, max(n, 1)), dtype=torch.float64, device=dev)
        has_d, has_q = cols.get("hit_dx") is not None, cols.get("hit_q_re") is not None
        ptr = lambda r, ok=True: C.c_void_p(per_row[r].data_ptr()) if ok else None
        L = lib()
        # a group count the library refuses gets no workspace size (-1): the call then reports why
        ws = self._ws(max(int(L.optb_monitor_stats_grouped_workspace_bytes(n, G)), 1))
        st = torch.cuda.current_stream(self.device).cuda_stream
        self._check(L.optb_monitor_stats_grouped(self._ctx, C.byref(res), 0, n, int(rays_per_config), int(n_configs),
                                                 int(n_monitors), C.c_void_p(frames_dev.data_ptr()), C.c_void_p(stats.data_ptr()),
                                                 ptr(0), ptr(1), ptr(2, has_d), ptr(3, has_d), ptr(4, has_d and has_q),
                                                 C.c_void_p(ws.data_ptr()), int(ws.numel()), C.c_void_p(st)))
        return stats, per_row[:, :n]

    @staticmethod
    def _hit_result(cols):
        """optb_result whose hit columns point at the CUDA tensors of `cols` (absent columns stay NULL)."""
        res = A.Result()
        for k in A.HIT_I32 + A.HIT_U32 + A.HIT_F64 + ("hit_key",):
            if cols.get(k) is not None:
                setattr(res, k, cols[k].data_ptr())
        return res

    def sweep_abcd_pivots(self, cols, n_rays, n_configs, mon0):
        """optb_sweep_abcd_pivots over the rows `cols` of sweep A (2 n_rays rays per configuration) on the current
        stream. Returns the device tensors pivots [n_rays, 3] and first_bad [1] (int64; -1: every configuration shares
        configuration 0's mon0 hit points)."""
        torch = self.torch
        dev = f"cuda:{self.device}"
        res = self._hit_result(cols)
        pivots = torch.empty((int(n_rays), 3), dtype=torch.float64, device=dev)
        first_bad = torch.empty(1, dtype=torch.int64, device=dev)
        L = lib()
        ws = self._ws(max(int(L.optb_sweep_abcd_workspace_bytes(int(n_rays), int(n_configs))), 1))
        st = torch.cuda.current_stream(self.device).cuda_stream
        self._check(L.optb_sweep_abcd_pivots(self._ctx, C.byref(res), int(cols["hit_px"].numel()), int(n_rays),
                                             int(n_configs), int(mon0), C.c_void_p(pivots.data_ptr()),
                                             C.c_void_p(first_bad.data_ptr()), C.c_void_p(ws.data_ptr()), int(ws.numel()),
                                             C.c_void_p(st)))
        return pivots, first_bad

    def sweep_abcd(self, cols_a, cols_b, n_rays, n_configs, mon1, frames, disp, rot):
        """optb_sweep_abcd over the rows of sweep A (`cols_a`, 2 n_rays rays per configuration) and sweep B (`cols_b`,
        n_rays) on the current stream; `frames`: a ctypes array of n_configs MonitorFrame (mon1 in each
        configuration). Returns the device tensors abcd [n_configs, n_rays, 4] and counts [n_configs, n_rays, 3]."""
        torch = self.torch
        dev = f"cuda:{self.device}"
        ra, rb = self._hit_result(cols_a), self._hit_result(cols_b)
        frames_dev = torch.frombuffer(bytearray(frames), dtype=torch.uint8).to(dev)
        abcd = torch.empty((int(n_configs), int(n_rays), 4), dtype=torch.float64, device=dev)
        counts = torch.empty((int(n_configs), int(n_rays), 3), dtype=torch.int32, device=dev)
        L = lib()
        ws = self._ws(max(int(L.optb_sweep_abcd_workspace_bytes(int(n_rays), int(n_configs))), 1))
        st = torch.cuda.current_stream(self.device).cuda_stream
        self._check(L.optb_sweep_abcd(self._ctx, C.byref(ra), int(cols_a["hit_px"].numel()), C.byref(rb),
                                      int(cols_b["hit_px"].numel()), int(n_rays), int(n_configs), int(mon1),
                                      C.c_void_p(frames_dev.data_ptr()), float(disp), float(rot),
                                      C.c_void_p(abcd.data_ptr()), C.c_void_p(counts.data_ptr()),
                                      C.c_void_p(ws.data_ptr()), int(ws.numel()), C.c_void_p(st)))
        return abcd, counts

    @staticmethod
    def _raise_status(counters):
        st = int(counters[A.C_STATUS])
        if st & A.ST_WORK_OVERFLOW:
            raise BackendError("wavefront workspace overflow: pass a larger max_live")
        if st & (A.ST_SEG_OVERFLOW | A.ST_HIT_OVERFLOW):
            raise BackendError("result capacity overflow")
