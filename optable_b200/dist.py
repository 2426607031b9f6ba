"""Multi-GPU plumbing for the ray_tracing path: shard the initial rays, merge the monitors.

The path shards without any data-path collective (SURVEY 8e): every rank traces a contiguous block of the
initial rays against its own replica of the scene tables. The only exchange is the monitor merge at the end:
all-reduce of the histograms, all-gather of the row counts and, when one rank wants every row, a gather-v of
the row columns. torch.distributed is the transport (NCCL over NVLink on the GPU box, gloo in the CPU tests).
"""
from __future__ import annotations

import numpy as np


def shard_bounds(n: int, rank: int, world: int, family=None):
    """Contiguous block [lo, hi) of initial-ray indices for `rank`. Concatenating the blocks in rank order
    keeps the reference's (initial ray, pop) output order. When `family` (dense Ray._id index per ray) is
    given, boundaries move forward to the next family change so that rays sharing an `_id` (interact-cap
    state, optical_component.py:136-149) stay on one rank; `family` must then be grouped contiguously."""
    lo, hi = n * rank // world, n * (rank + 1) // world
    if family is not None and n:
        fam = np.asarray(family)

        def snap(i):
            while 0 < i < n and fam[i] == fam[i - 1]:
                i += 1
            return i

        lo, hi = snap(lo), snap(hi)
    return lo, hi


def merge_histograms(hist_y, hist_yz, group=None):
    """In-place sum over ranks of the per-monitor histograms (int64 tensors)."""
    import torch.distributed as dist

    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(hist_y, group=group)
        dist.all_reduce(hist_yz, group=group)
    return hist_y, hist_yz


def gather_row_counts(n_rows: int, device="cpu", group=None):
    """Number of monitor rows every rank holds (list of ints, rank order)."""
    import torch
    import torch.distributed as dist

    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return [int(n_rows)]
    mine = torch.tensor([int(n_rows)], dtype=torch.int64, device=device)
    out = [torch.zeros_like(mine) for _ in range(dist.get_world_size(group))]
    dist.all_gather(out, mine, group=group)
    return [int(t.item()) for t in out]


def gather_rows(columns: dict, n_rows: int, root_offset: int = 0, group=None):
    """Gather-v of monitor row columns: every rank receives the rows of all ranks, concatenated in rank order
    (= initial-ray block order). `hit_root` is shifted by `root_offset` (the rank's first global ray index) so
    that row keys stay global. Columns are 1-D tensors with at least n_rows valid leading entries."""
    import torch
    import torch.distributed as dist

    cols = {k: v[:n_rows] for k, v in columns.items()}
    if "hit_root" in cols and root_offset:
        cols["hit_root"] = cols["hit_root"] + int(root_offset)
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return cols
    any_col = next(iter(cols.values()))
    counts = gather_row_counts(n_rows, any_col.device, group)
    width = max(counts)
    out = {}
    for k, v in cols.items():
        padded = torch.zeros(width, dtype=v.dtype, device=v.device)
        padded[:n_rows] = v
        parts = [torch.zeros_like(padded) for _ in counts]
        dist.all_gather(parts, padded, group=group)
        out[k] = torch.cat([p[:c] for p, c in zip(parts, counts)])
    return out


def merge_counters(counters, group=None):
    """Sum over ranks of the OPTB_C_* counters of one sharded trace (numpy int64 array or tensor); the status word is
    a bit mask and is OR-ed. Returns a numpy array."""
    import torch
    import torch.distributed as dist

    from . import _abi as A

    c = torch.as_tensor(np.asarray(counters, dtype=np.int64)).clone()
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return c.numpy()
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    bits = torch.tensor([(int(c[A.C_STATUS]) >> k) & 1 for k in range(16)], dtype=torch.int64)
    c[A.C_STATUS] = 0
    gens = c[A.C_GENERATIONS].clone()
    both = torch.cat([c, bits, gens.reshape(1)]).to(dev)
    dist.all_reduce(both, group=group)
    mx = gens.reshape(1).to(dev)
    dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    both = both.cpu()
    out = both[:len(c)].clone()
    out[A.C_STATUS] = sum((1 << k) for k in range(16) if int(both[len(c) + k]) > 0)
    out[A.C_GENERATIONS] = int(mx.item())  # generations run side by side on the ranks: the longest shard counts
    return out.numpy()


def trace_sharded(table, bundle, perfomance_limit=None, group=None, gather=False, record_hits=True, record_hist=True,
                  engine=None, tracer=None, **kw):
    """Multi-GPU form of `OpticalTable.trace_bundle` (SURVEY 8e): rank r of `group` traces the contiguous block
    [lo, hi) = shard_bounds(bundle.n, r, world) of the initial rays on its own GPU against its own replica of the
    scene tables; no data-path collective. The only exchange is the monitor merge at the end: all-reduce of the
    histograms and of the counters and, with `gather=True`, a gather-v of the monitor row columns so that every
    rank holds all rows (concatenated in rank order = initial-ray block order). Row keys are global (`hit_root` /
    `hit_key` count from ray 0 of the whole bundle).

    Returns the dict of `trace_bundle` with merged `hist_y` / `hist_yz` / `counters`, plus `counters_local` and
    `shard` = (lo, hi). Without an initialised process group it is `trace_bundle` on the whole bundle.
    `tracer(table, bundle, perfomance_limit, record_hits=, record_hist=, engine=, **kw)` defaults to the CUDA
    `bundle.trace_bundle`; the CPU tests of this module pass a stand-in."""
    import torch.distributed as dist

    from . import _abi as A

    on = dist.is_initialized()
    rank, world = (dist.get_rank(group), dist.get_world_size(group)) if on else (0, 1)
    lo, hi = shard_bounds(bundle.n, rank, world)
    if tracer is None:
        from .bundle import trace_bundle as tracer
    res = tracer(table, bundle.slice(lo, hi), perfomance_limit, record_hits=record_hits, record_hist=record_hist,
                 engine=engine, **kw)
    rows = {k: v for k, v in res.items() if k.startswith("hit_")}
    n_rows = int(res["counters"][A.C_HITS]) if record_hits else 0
    if lo:
        if "hit_root" in rows:
            rows["hit_root"] = rows["hit_root"] + int(lo)     # uint32 bit pattern in int32: wraps like unsigned
        if "hit_key" in rows:
            rows["hit_key"] = rows["hit_key"] + (int(lo) << 32)
    out = dict(res)
    out["counters_local"] = np.asarray(res["counters"]).copy()
    out["shard"] = (lo, hi)
    if on and world > 1:
        if record_hist:
            merge_histograms(res["hist_y"], res["hist_yz"], group)
        out["counters"] = merge_counters(res["counters"], group)
        if gather and record_hits:
            rows = gather_rows(rows, n_rows, 0, group)
    out.update(rows)
    return out


def _collective_device(group=None):
    """Where tensors of a collective live: the current CUDA device under NCCL, the host under gloo."""
    import torch.distributed as dist

    return "cuda" if dist.get_backend(group) == "nccl" else "cpu"


def _gather_configs(t, counts, group=None):
    """All-gather of per-rank slices [K_r, ...] of a per-configuration array (uneven K_r = `counts`, rank order):
    padded to the largest slice, returns the concatenation [sum K_r, ...] on every rank, on t's device. Not a sum:
    each slice lands at its own configurations."""
    import torch
    import torch.distributed as dist

    padded = torch.zeros((max(counts),) + tuple(t.shape[1:]), dtype=t.dtype, device=_collective_device(group))
    padded[:t.shape[0]] = t
    parts = [torch.empty_like(padded) for _ in counts]
    dist.all_gather(parts, padded, group=group)
    return torch.cat([p[:c] for p, c in zip(parts, counts)]).to(t.device)


def trace_sweep_sharded(n_configs, n_rays, rays, limit, prepare, monitors, label, tracer, group=None, gather=False,
                        record_hits=True, record_hist=False, engine=None, unit=None, arrs=None, fam_ids=None):
    """Multi-GPU form of a sweep (`trace_sweep` / `SweepScene.trace` with `group=`): the K configurations are sharded
    over the ranks of `group`, rank r owning the contiguous configurations [k0, k1) = shard_bounds(K, r, world) (equal
    counts, no balancing by cost; K < world leaves ranks without configurations, which still take part in every
    collective). Every group (k, m) of the monitor statistics is reduced on its own rows in a fixed order, so a
    configuration that stays on one rank gets the bits of the one-GPU sweep: rows, histograms and statistics.

    `prepare(k0, k1)` runs this rank's host side and returns (configs, shares, caps0): the FlatScenes or SweepRows of
    its configurations (None when k0 == k1), a list with one picklable item per configuration that every rank receives
    (SweepScene: the frames of the varied monitors, else None) and the starting interact counts of its configurations
    (`sweep.initial_counts` of the families `fam_ids` of a list of Ray, or None). `monitors`: the [K][M] monitor frames, or a function of the
    gathered shares (configuration order) that returns them. A rank without configurations does not call `prepare`.

    Before any trace, one exchange checks on every rank (so that no rank waits in a collective while another raised):
    what `prepare` raised on any rank, the topology of the ranks' configurations (`sweep.topology_key`; ValueError
    naming the first differing global configuration), interact caps, and the largest `max_children`. A rank whose
    own configurations do not split while others do runs the wavefront kernels with chain_len = limit + 1, which
    selects the variant the one-GPU sweep runs and never cuts a chain (a root pops at most `limit` times). For a list
    of Ray on a capped scene, every rank also sends its largest starting count and its smallest cap, so that all ranks
    decide as the one-GPU sweep does, over all K configurations, whether to trace family-serially (`sweep.caps_bind`;
    chain_len is then 0); the [K, S, F] `interact_counts` are all-gathered. The global
    K * N < 2^32 bound is checked up front, since row keys are global.

    After the trace: statistics of the rank's own rows (`optb_monitor_stats_grouped`, configurations numbered from
    k0), all-gather of their slots and of the [K_r, M, ...] histograms, `merge_counters`, roots rebased to k * N + r
    and, with `gather`, `gather_rows`. Returns (out, monitors): the result dict SweepResult reads (`shard`, `world`,
    `holds`, `counters_local`, `chain_len`, `stats_slots`) and the [K][M] frames."""
    import builtins

    import torch
    import torch.distributed as dist

    from . import _abi as A
    from .analytics import grouped_slots
    from .backend import caps_can_bind
    from .sweep import SweepRows, largest_family, topology_key, topology_mismatch

    K, n = int(n_configs), int(n_rays)
    who, what = label.split(": ")
    if K * n >= 1 << 32:
        raise ValueError(f"{who}: n_configs * rays ({K} x {n}) must stay below 2^32: row keys count roots over all "
                         "configurations")
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    bounds = [shard_bounds(K, r, world) for r in range(world)]
    counts = [hi - lo for lo, hi in bounds]
    k0, k1 = bounds[rank]
    mismatch = lambda k, why: f"{label} {k} does not have the topology of {what} 0 ({why})"

    # ---- this rank's host side, and one exchange of what every rank must know before any trace
    mine = {"error": None, "key": None, "max_children": 0, "shares": [], "caps": (0, float("inf"), 0)}
    configs, err, caps0 = None, None, None
    try:
        if k1 > k0:
            configs, shares, caps0 = prepare(k0, k1)
            mine["shares"] = shares or []
        if configs is not None:
            rows = configs if isinstance(configs, SweepRows) else None
            flats = [rows] if rows is not None else configs
            flat0 = rows.flat if rows is not None else configs[0]
            mine["key"] = topology_key(flat0)     # (sent even when a later configuration of this rank differs)
            bad = topology_mismatch(configs) if rows is None else None
            if bad is not None:
                raise ValueError(mismatch(k0 + bad[0], bad[1]))
            cap_min = min(f.cap_min for f in flats)
            if flat0.n_capslots and arrs is None and cap_min < limit:
                raise NotImplementedError("bundle traces need max_interact_count >= max_trace_num on every capped "
                                          "component (a sweep of Ray objects with ids lifts this)")
            mine["max_children"] = max(f.max_children for f in flats)
            mine["caps"] = (int(caps0.max(initial=0)) if caps0 is not None else 0, cap_min, flat0.n_capslots)
    except Exception as e:   # raised on every rank below
        err, mine["error"] = e, (k0, type(e).__name__, str(e))
    states = [None] * world
    dist.all_gather_object(states, mine, group=group)
    # (first configuration, exception name, message, rank that raised it or None): the earliest one is raised everywhere
    found = [s["error"] + (r,) for r, s in enumerate(states) if s["error"] is not None]
    ref = next((s["key"] for s in states if s["key"] is not None), None)
    found += [(bounds[r][0], "ValueError", mismatch(bounds[r][0], f"its sizes, node kinds or material kinds differ; "
                                                    f"rank {r} traces it"), None)
              for r, s in enumerate(states) if s["key"] not in (None, ref)]
    if found:
        k, name, msg, r = min(found, key=lambda f: (f[0], f[3] is not None))
        if r == rank:
            raise err
        cls = getattr(builtins, name, None)
        cls = cls if isinstance(cls, type) and issubclass(cls, Exception) else RuntimeError
        raise cls(msg if r is None else f"{msg} (raised on rank {r} of the sharded sweep)")
    if callable(monitors):
        monitors = monitors([x for s in states for x in s["shares"]])
    M = len(monitors[0])
    Mh = max(M, 1)       # the device keeps one histogram row per monitor, at least one per configuration
    wide = max(s["max_children"] for s in states)
    n_caps = max(s["caps"][2] for s in states)
    counted = fam_ids is not None and n_caps > 0     # a list of Ray on a capped scene: interact_counts are returned
    serial = counted and caps_can_bind(max(s["caps"][0] for s in states), largest_family(arrs),
                                       min(s["caps"][1] for s in states), limit)
    chain_len = int(limit) + 1 if configs is not None and wide > 1 >= mine["max_children"] and not serial else 0

    # ---- this rank's trace
    dev = _collective_device(group)
    cols = A.HIT_I32 + A.HIT_U32 + A.HIT_F64
    if configs is not None:
        res = tracer(configs, rays, limit, record_hits=record_hits, record_hist=record_hist, engine=engine, unit=unit,
                     arrs=arrs, chain_len=chain_len, **({"caps0": caps0, "serial": serial} if counted else {}))
        counters = np.asarray(res["counters"])
    else:
        dt = {k: torch.int32 for k in A.HIT_I32 + A.HIT_U32}
        res = {k: torch.empty(0, dtype=dt.get(k, torch.float64), device=dev) for k in cols} if record_hits else {}
        res["hist_y"] = torch.zeros((0, Mh, A.HIST_BINS), dtype=torch.int64, device=dev)
        res["hist_yz"] = torch.zeros((0, Mh, A.HIST_BINS, A.HIST_BINS), dtype=torch.int64, device=dev)
        counters = np.zeros(A.C_COUNT, dtype=np.int64)
    rows = {k: res[k] for k in cols + ("hit_key",) if k in res}
    n_rows = int(rows["hit_px"].numel()) if record_hits else 0

    # ---- statistics of the own rows, before their roots are made global
    out = {"shard": (k0, k1), "world": world, "holds": (0, K) if gather and record_hits else (k0, k1),
           "counters_local": counters.copy(), "chain_len": chain_len, "stats_slots": None}
    if record_hits:
        slots = (torch.from_numpy(grouped_slots(rows, monitors[k0:k1], n, engine)[0]) if configs is not None
                 else torch.zeros((0, M, A.MS_STRIDE), dtype=torch.float64))
        out["stats_slots"] = _gather_configs(slots, counts, group).numpy()
    if k0 and "hit_root" in rows:
        r = (rows["hit_root"].long() & 0xFFFFFFFF) + k0 * n
        rows["hit_root"] = (r - ((r >> 31) << 32)).to(rows["hit_root"].dtype)   # uint32 bit pattern in int32
    if k0 and "hit_key" in rows:
        rows["hit_key"] = rows["hit_key"] + ((k0 * n) << 32)

    # ---- what every rank receives
    hy = res["hist_y"].reshape(k1 - k0, Mh, A.HIST_BINS)
    hyz = res["hist_yz"].reshape(k1 - k0, Mh, A.HIST_BINS, A.HIST_BINS)
    if record_hist:
        out["hist_y"], out["hist_yz"] = _gather_configs(hy, counts, group), _gather_configs(hyz, counts, group)
    else:
        out["hist_y"] = torch.zeros((K,) + tuple(hy.shape[1:]), dtype=hy.dtype, device=hy.device)
        out["hist_yz"] = torch.zeros((K,) + tuple(hyz.shape[1:]), dtype=hyz.dtype, device=hyz.device)
    out["counters"] = merge_counters(counters, group)
    if counted:
        mine_counts = (torch.from_numpy(np.asarray(res["interact_counts"])) if configs is not None
                       else torch.zeros((0, n_caps, len(fam_ids)), dtype=torch.int32))
        out["interact_counts"] = _gather_configs(mine_counts, counts, group).numpy()
    if gather and record_hits:
        where = rows["hit_px"].device
        rows = {k: v.to(where) for k, v in gather_rows({k: v.to(dev) for k, v in rows.items()}, n_rows, 0, group).items()}
    out.update(rows)
    return out, monitors
