"""CPU, gloo: sweeps sharded over ranks by configuration (`trace_sweep` / `SweepScene.trace` with `group=`). The C
oracle stands in for the device trace and a host model of `optb_monitor_stats_grouped` for the statistics; the
sharded call must give every rank what the one-process call gives: rows with global roots, `rows(k)`, the [K, M, ...]
histograms, counters, statistics and monitor frames. Errors that one rank sees are raised on every rank."""
import datetime
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import optable_b200 as ob
from optable_b200 import _abi as A
from optable_b200 import dist as D
from optable_b200.bundle import RayBundle
from optable_b200.sweep import SweepRows, SweepScene, trace_sweep
from optable_b200.workloads import telescope_4f_grid
from tests import scenes

HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64
SAME_COUNTERS = [c for c in range(A.C_COUNT) if c not in (A.C_LAUNCHES, A.C_GENERATIONS)]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _oracle(configs, rays, limit, record_hits=True, record_hist=False, engine=None, unit=None, arrs=None, chain_len=0):
    """Stand-in for the CUDA sweep (FlatScenes or a SweepRows): K oracle traces, roots renumbered k * N + r, rows and
    histograms concatenated in configuration order. Records the chain_len it was handed in `_oracle.chain_lens`."""
    from oracle import oracle as O

    _oracle.chain_lens.append(chain_len)
    flats = [configs.materialise(k) for k in range(configs.n_configs)] if isinstance(configs, SweepRows) else configs
    arrs = rays.materialise() if arrs is None else arrs
    n = len(arrs["ox"])
    parts = [O.trace(f, arrs, max_trace_num=limit, record_segments=False, record_hits=record_hits, record_hist=True)
             for f in flats]
    out = {}
    if record_hits:
        for k in HIT_COLS:
            v = np.concatenate([p[k].astype(np.int64) + c * n if k == "hit_root" else p[k] for c, p in enumerate(parts)])
            out[k] = torch.from_numpy(v.astype(np.uint32).view(np.int32) if k == "hit_root" else
                                      (v.view(np.int32) if v.dtype == np.uint32 else v))
    out["hist_y"] = torch.from_numpy(np.concatenate([p["hist_y"] for p in parts]))
    out["hist_yz"] = torch.from_numpy(np.concatenate([p["hist_yz"] for p in parts]))
    out["counters"] = np.sum([p["counters"] for p in parts], axis=0)
    return out


_oracle.chain_lens = []


class _HostStats:
    """Host model of Engine.monitor_stats_grouped: each (configuration, monitor) group summarised from its own rows in
    row order, in the frame it is given (y, z = the hit point along the frame's tangents). Like the device, a group's
    slots depend on its rows and frame only."""

    def monitor_stats_grouped(self, cols, frames, n_configs, n_monitors, rays_per_config=0):
        P = np.stack([cols[k].numpy() for k in ("hit_px", "hit_py", "hit_pz")], 1)
        root = cols["hit_root"].numpy().view(np.uint32).astype(np.int64)
        g = (root // rays_per_config if rays_per_config else 0) * n_monitors + cols["hit_monitor"].numpy()
        I = cols["hit_intensity"].numpy()
        y, z = np.empty(len(P)), np.empty(len(P))
        s = np.zeros((n_configs * n_monitors, A.MS_STRIDE))
        for i, fr in enumerate(frames):
            sel = g == i
            y[sel], z[sel] = P[sel] @ np.array(fr.tangent_y[:]), P[sel] @ np.array(fr.tangent_z[:])
            ys, zs = y[sel], z[sel]
            s[i, A.MS_COUNT], s[i, A.MS_SUM_I], s[i, A.MS_SUM_Y], s[i, A.MS_SUM_Z] = sel.sum(), I[sel].sum(), ys.sum(), zs.sum()
            s[i, A.MS_MIN_Y], s[i, A.MS_MAX_Y] = ys.min(initial=np.inf), ys.max(initial=-np.inf)
            s[i, A.MS_MIN_Z], s[i, A.MS_MAX_Z] = zs.min(initial=np.inf), zs.max(initial=-np.inf)
            s[i, A.MS_M2_Y] = ((ys - ys.mean()) ** 2).sum() if ys.size else 0.0
            w = fr.half_width
            s[i, A.MS_HIST:A.MS_HIST + A.HIST_BINS] = np.histogram(ys, A.HIST_BINS, (-w, w))[0]
        per_row = torch.from_numpy(np.stack([y, z, np.zeros_like(y), np.zeros_like(y), np.zeros_like(y)]))
        return torch.from_numpy(s), per_row


def _grid(K):
    return [telescope_4f_grid(ob, 43.17 + 0.4 * k - 1.0, 43.17 - 0.3 * k + 0.5) for k in range(K)]


def _four_f_scene(calls):
    """The 4f grid with lens 2 and monitor 1 varied; configure(k) appends k to `calls`."""
    t = telescope_4f_grid(ob, 43.17, 43.17)
    lens, mon = t.components[1], t.monitors[1]
    saved = []

    def walk(o):
        saved.append((o, o.origin.copy(), np.array(o.transform_matrix, dtype=np.float64), o._bbox))
        for c in getattr(o, "components", []):
            walk(c)

    walk(lens)
    walk(mon)

    def configure(k):
        calls.append(k)
        for o, org, T, box in saved:
            o.origin, o.transform_matrix, o._bbox = org.copy(), T.copy(), box
        lens.TX(0.3 * k - 0.4)
        mon.TX(0.5 * k - 0.2)

    return t, [lens, mon], configure


def _bundle():
    return RayBundle.collimated_disc(37, radius=2.5)   # not a multiple of 32


def _run(kind, K, gather, group=True):
    """One sweep of `kind` ("tables" or "scene") with the stand-ins; returns (result, configure calls, table)."""
    calls = []
    if kind == "tables":
        return trace_sweep(_grid(K), _bundle(), record_hist=True, tracer=_oracle, engine=_HostStats(), group=group,
                           gather=gather), calls, None
    t, vary, configure = _four_f_scene(calls)
    res = SweepScene(t, vary).trace(_bundle(), configure, K, record_hist=True, tracer=_oracle, engine=_HostStats(),
                                    group=group, gather=gather)
    return res, calls, t


def _dump(res, calls, t):
    """What a rank's result holds, as numpy arrays."""
    d = {"shard": np.array(res.shard), "calls": np.array(calls, dtype=np.int64), "counters": res.counters,
         "counters_local": res.counters_local, "hist_y": res.hist_y.numpy(), "hist_yz": res.hist_yz.numpy(),
         "chain_len": np.array(res.chain_len)}
    d.update({f"hits/{c}": v.numpy() for c, v in res.hits.items()})
    d.update({f"stats/{q}": v for q, v in res.stats().items()})
    d.update({f"frame/{k}/{m}": np.concatenate([f.origin, np.ravel(f.tangent_Y), np.ravel(f.tangent_Z), [f.width]])
              for k, row in enumerate(res.monitors) for m, f in enumerate(row)})
    held = range(*res._holds)
    for k in held:
        d.update({f"rows/{k}/{c}": v.numpy() for c, v in res.rows(k).items()})
    d["row_values"] = res.row_values()["y"].numpy()
    if t is not None:
        d["end"] = np.concatenate([t.components[1].origin, t.monitors[1].origin])
    others = [k for k in range(res.n_configs) if k not in held]
    if others:
        with pytest.raises(IndexError, match=r"rank \d+ of this sharded sweep.*gather=True"):
            res.rows(others[0])
        with pytest.raises(IndexError, match="gather=True"):
            res.monitor(others[0], 0)
    return d


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))


def _sweep_worker(rank, world, port, kind, K, gather, path):
    _init(rank, world, port)
    try:
        np.savez(f"{path}_{rank}.npz", **_dump(*_run(kind, K, gather)))
    finally:
        dist.destroy_process_group()


def _same(a, b, label):
    assert a.shape == b.shape, label
    if a.dtype.kind == "f":
        bits = lambda x: np.ascontiguousarray(x).view(np.uint8)
        assert np.array_equal(bits(a), bits(b)) or np.array_equal(a, b, equal_nan=True), label
    else:
        assert np.array_equal(a, b), label


@pytest.mark.parametrize("kind,world,K,gather", [("tables", 2, 5, False), ("tables", 3, 5, False), ("tables", 2, 5, True),
                                                 ("tables", 3, 2, False), ("scene", 2, 5, False), ("scene", 3, 5, True),
                                                 ("scene", 3, 2, False)])
def test_sharded_sweep_equals_one_process(tmp_path, kind, world, K, gather):
    path = str(tmp_path / "rank")
    mp.spawn(_sweep_worker, args=(world, _free_port(), kind, K, gather, path), nprocs=world, join=True)
    one, calls_one, t_one = _run(kind, K, False, group=None)
    want = _dump(one, calls_one, t_one)
    lo_rows = 0
    for r in range(world):
        got = dict(np.load(f"{path}_{r}.npz"))
        k0, k1 = D.shard_bounds(K, r, world)
        assert tuple(got["shard"]) == (k0, k1)
        for q in ("hist_y", "hist_yz") + tuple(k for k in want if k.startswith(("stats/", "frame/"))):
            _same(got[q], want[q], f"rank {r} {q}")
        np.testing.assert_array_equal(got["counters"][SAME_COUNTERS], want["counters"][SAME_COUNTERS])
        # rows: this rank's configurations with global roots (all of them after gather=True)
        a, b = (0, K) if gather else (k0, k1)
        lo, hi = one._bounds[a], one._bounds[b]
        for c in HIT_COLS:
            _same(got[f"hits/{c}"], want[f"hits/{c}"][lo:hi], f"rank {r} {c}")
        _same(got["row_values"], want["row_values"][lo:hi], f"rank {r} row_values")
        for k in range(a, b):
            for c in HIT_COLS + ("hist_y", "hist_yz"):
                _same(got[f"rows/{k}/{c}"], want[f"rows/{k}/{c}"], f"rank {r} rows({k}) {c}")
        if k0 == k1:   # a rank without configurations: no rows, but every histogram and statistic
            assert got["hits/hit_px"].size == 0 and got["counters_local"].sum() == 0
        lo_rows += int(got["counters_local"][A.C_HITS])
        assert int(got["chain_len"]) == 0       # the 4f grid never splits
        if kind == "scene":
            owned = list(range(k0, k1))
            assert list(got["calls"]) == owned + ([] if K - 1 in owned else [K - 1])
            _same(got["end"], want["end"], f"rank {r}: the table stands in configuration K - 1")
    assert lo_rows == int(want["counters"][A.C_HITS])


def _slab_tables(K):
    """Splitting slab between two mirrors whose faces reflect nothing in configuration 0: that configuration alone
    would run a non-splitting kernel."""
    def one(k):
        slab = ob.GlassSlab([0, 0, 0], width=2, height=2, thickness=0.5, n1=1, n2=1.5, reflectivity=0.05 * k)
        return scenes.Scene([ob.Mirror([-2, 0, 0], radius=3, reflectivity=0.9, transmission=0.0), slab,
                             ob.Mirror([2, 0, 0], radius=3, reflectivity=0.9, transmission=0.0).RotZ(np.pi)],
                            [], [ob.Monitor([1, 0, 0], 6, 6), ob.Monitor([-3, 0, 0], 6, 6)])
    return [one(k) for k in range(K)]


def _slab_worker(rank, world, port, path):
    _init(rank, world, port)
    try:
        bundle = RayBundle.collimated_disc(9, x0=-1.5, radius=0.6, direction=(1.0, 0.01, 0.0))
        res = trace_sweep(_slab_tables(3), bundle, {"max_trace_num": 12}, record_hist=True, tracer=_oracle,
                          engine=_HostStats(), group=True, gather=True)
        np.savez(f"{path}_{rank}.npz", chain_len=np.array(_oracle.chain_lens), res_chain_len=np.array(res.chain_len),
                 hist_y=res.hist_y.numpy(), **{c: v.numpy() for c, v in res.hits.items()})
    finally:
        dist.destroy_process_group()


def test_shard_without_splitting_configurations_runs_the_wavefront_kernels(tmp_path):
    """World 2, K = 3: rank 0 owns configuration 0 alone, whose faces reflect nothing, so it is handed chain_len =
    max_trace_num + 1 (the wavefront kernels the one-GPU sweep runs); rank 1's configurations split and need no
    forcing. Rows and histograms stay those of the one-process sweep."""
    path = str(tmp_path / "slab")
    mp.spawn(_slab_worker, args=(2, _free_port(), path), nprocs=2, join=True)
    r0, r1 = dict(np.load(f"{path}_0.npz")), dict(np.load(f"{path}_1.npz"))
    assert D.shard_bounds(3, 0, 2) == (0, 1)
    assert list(r0["chain_len"]) == [13] and int(r0["res_chain_len"]) == 13
    assert list(r1["chain_len"]) == [0] and int(r1["res_chain_len"]) == 0
    bundle = RayBundle.collimated_disc(9, x0=-1.5, radius=0.6, direction=(1.0, 0.01, 0.0))
    want = trace_sweep(_slab_tables(3), bundle, {"max_trace_num": 12}, record_hist=True, tracer=_oracle)
    for got in (r0, r1):
        np.testing.assert_array_equal(got["hist_y"], want.hist_y.numpy())
        for c in HIT_COLS:
            _same(got[c], want.hits[c].numpy(), c)


def _error_worker(rank, world, port, case, path):
    _init(rank, world, port)
    try:
        a = scenes.Scene([ob.Mirror([0, 0, 0])], [], [ob.Monitor([2, 0, 0], 4, 4)])
        b = scenes.Scene([ob.Mirror([0, 0, 0]), ob.Mirror([5, 0, 0])], [], [ob.Monitor([2, 0, 0], 4, 4)])
        kw = dict(tracer=_oracle, engine=_HostStats(), group=True)
        try:
            if case == "local":       # only rank 1 holds the odd table, behind one of its own
                trace_sweep([a, a, a, b], RayBundle.collimated_disc(4), **kw)
            elif case == "across":    # rank 1's tables agree with each other, not with rank 0's
                trace_sweep([a, a, b, b], RayBundle.collimated_disc(4), **kw)
            elif case == "roots":     # 2^16 + 1 configurations of 2^16 rays: global keys would not fit
                trace_sweep([a] * ((1 << 16) + 1), RayBundle.collimated_disc(1 << 16), **kw)
            elif case == "configure":  # configure fails on rank 1 only
                t = telescope_4f_grid(ob, 43.17, 43.17)

                def configure(k):
                    if k == 3:
                        raise RuntimeError("configuration 3 cannot be built")

                SweepScene(t, [t.components[1]]).trace(_bundle(), configure, 4, **kw)
            got = "no error"
        except Exception as e:
            got = f"{type(e).__name__}: {e}"
        dist.barrier()   # every rank got here: none waits in a collective of the sweep
        with open(f"{path}_{rank}.txt", "w") as f:
            f.write(got)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("case,pattern", [
    ("local", r"ValueError: trace_sweep: table 3 does not have the topology of table 0 \(n_nodes 2 != 1\)"),
    ("across", r"ValueError: trace_sweep: table 2 does not have the topology of table 0 \(.*rank 1 traces it\)"),
    ("roots", r"ValueError: trace_sweep: n_configs \* rays \(65537 x 65536\) must stay below 2\^32"),
    ("configure", r"RuntimeError: configuration 3 cannot be built"),
])
def test_errors_are_raised_on_every_rank(tmp_path, case, pattern):
    import re

    path = str(tmp_path / "err")
    mp.spawn(_error_worker, args=(2, _free_port(), case, path), nprocs=2, join=True)
    for r in range(2):
        msg = open(f"{path}_{r}.txt").read()
        assert re.match(pattern, msg), (r, msg)
