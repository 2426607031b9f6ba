"""CPU: sweeps of Ray objects through scenes whose interact caps bind (the family-serial sweep). The C oracle stands in
for the device and traces each configuration on its own from that configuration's starting counts; the sweep must give
per configuration its rows, histograms and final `interact_counts`, decide family-serial or parallel with the rule of
`Engine.trace_arrays` over all configurations, and give the same under gloo with 2 and 3 ranks."""
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
from optable_b200.bundle import RayBundle
from optable_b200.flatten import FlatScene, pack_rays
from optable_b200.sweep import SweepRows, SweepScene, _family_counts, sweep_abcd_matrix, trace_sweep
from tests import scenes

HIT_COLS = A.HIT_I32 + A.HIT_U32 + A.HIT_F64


def _oracle(configs, rays, limit, record_hits=True, record_hist=False, engine=None, unit=None, arrs=None, chain_len=0,
            caps0=None, serial=None):
    """Stand-in for the CUDA sweep: configuration k traced alone by the oracle from columns [k F, (k + 1) F) of `caps0`,
    roots renumbered k * N + r. Records what it was handed in `_oracle.calls`."""
    from oracle import oracle as O

    _oracle.calls.append({"caps0": caps0, "serial": serial, "chain_len": chain_len})
    flats = [configs.materialise(k) for k in range(configs.n_configs)] if isinstance(configs, SweepRows) else configs
    arrs = rays.materialise() if arrs is None else arrs
    n, K = len(arrs["ox"]), len(flats)
    F = None if caps0 is None else caps0.shape[1] // K
    parts = [O.trace(f, arrs, max_trace_num=limit, unit=unit or 1e-2, record_segments=False, record_hits=record_hits,
                     record_hist=True, **({} if F is None else {"n_families": F, "cap_counts": caps0[:, k * F:(k + 1) * F]}))
             for k, f in enumerate(flats)]
    out = {}
    for k in HIT_COLS:
        v = np.concatenate([p[k].astype(np.int64) + c * n if k == "hit_root" else p[k] for c, p in enumerate(parts)])
        out[k] = torch.from_numpy(v.astype(np.uint32).view(np.int32) if k == "hit_root" else
                                  (v.view(np.int32) if v.dtype == np.uint32 else v))
    out["hist_y"] = torch.from_numpy(np.concatenate([p["hist_y"] for p in parts]))
    out["hist_yz"] = torch.from_numpy(np.concatenate([p["hist_yz"] for p in parts]))
    out["counters"] = np.sum([p["counters"] for p in parts], axis=0)
    if caps0 is not None:
        out["interact_counts"] = np.stack([p["cap_counts"] for p in parts]).astype(np.int32)
    return out


_oracle.calls = []


def _prism_table(refl, tilt, cap=3):
    """tests.scenes.caps_binding with its reflectivities and tilt varied and caps of `cap` on faces 2 and 3."""
    sc = scenes.caps_binding(ob)
    L = 6
    ps = ob.TriangularPrism(origin=[0, 0, 0], width=L, height=L, n1=1, n2=ob.Glass_NBK7(), alpha=np.pi / 4,
                            beta=np.pi / 2, reflectivity_1=refl, reflectivity_2=0.5, reflectivity_3=0.4,
                            max_interact_count_2=cap, max_interact_count_3=cap).RotZ(tilt)
    return scenes.Scene([ps], sc.rays, sc.monitors, limit=sc.limit)


def _seed_counts(table, fam_ids, k):
    """Non-zero starting counts that differ per configuration."""
    for s, comp in enumerate(FlatScene(table.components, table.monitors).capslots):
        comp._interact_count = {rid: (f + s + k) % 3 for f, rid in enumerate(fam_ids) if (f + k) % 2 == 0}


def _check(res, tables, rays, limit):
    """Every configuration equals its own oracle trace from the components' counts."""
    from oracle import oracle as O

    arrs, fam_ids, unit = pack_rays(rays)
    assert res.family_ids == fam_ids
    assert res.interact_counts.shape == (len(tables), res.interact_counts.shape[1], len(fam_ids))
    for k, t in enumerate(tables):
        flat = FlatScene(t.components, t.monitors)
        caps0 = np.array([[c._interact_count.get(rid, 0) for rid in fam_ids] for c in flat.capslots], np.int32)
        assert [id(c) for c in res.cap_components[k]] == [id(c) for c in flat.capslots]
        want = O.trace(flat, arrs, max_trace_num=limit, unit=unit, record_segments=False, record_hist=True,
                       n_families=len(fam_ids), cap_counts=caps0.copy())   # (the oracle counts in place)
        got = res.rows(k)
        assert len(got["hit_root"]) == len(want["hit_root"]) > 0
        for c in HIT_COLS:
            g = got[c].numpy()
            np.testing.assert_array_equal(g.view(want[c].dtype) if want[c].dtype == np.uint32 else g, want[c], err_msg=f"{k} {c}")
        np.testing.assert_array_equal(got["hist_y"].numpy(), want["hist_y"][:1])
        np.testing.assert_array_equal(got["hist_yz"].numpy(), want["hist_yz"][:1])
        np.testing.assert_array_equal(res.interact_counts[k], want["cap_counts"])
        assert not np.array_equal(want["cap_counts"], caps0)


def test_trace_sweep_binding_caps_with_starting_counts():
    tables = [_prism_table(r, t) for r, t in ((0.3, 0.0), (0.2, 0.03), (0.45, -0.05))]
    rays = tables[0].rays
    _, fam_ids, _ = pack_rays(rays)
    for k, t in enumerate(tables):
        _seed_counts(t, fam_ids, k)
    _oracle.calls.clear()
    res = trace_sweep(tables, rays, tables[0].limit, record_hist=True, tracer=_oracle)
    assert _oracle.calls[-1]["serial"] is True
    _check(res, tables, rays, 80)
    # a sweep is a tensor entry point: the components' counts are not written back
    assert res.cap_components[0][0]._interact_count == {rid: (f + 0) % 3 for f, rid in enumerate(fam_ids) if f % 2 == 0}


def test_shared_ids_bind_where_every_root_alone_would_not():
    # caps of 100 against 80 pops: one root alone cannot reach them, but 6 wavelengths share each id, as in
    # ray_tracing; the sweep must run family-serially and count per id
    tables = [_prism_table(0.3, t, cap=100) for t in (0.0, 0.02)]
    rays = tables[0].rays
    _oracle.calls.clear()
    res = trace_sweep(tables, rays, {"max_trace_num": 80}, record_hist=True, tracer=_oracle)
    assert _oracle.calls[-1]["serial"] is True
    _check(res, tables, rays, 80)
    assert res.interact_counts.max() > 80


def test_caps_that_cannot_bind_keep_the_parallel_sweep():
    tables = [_prism_table(0.3, t, cap=10 ** 5) for t in (0.0, 0.02)]
    rays = tables[0].rays
    _oracle.calls.clear()
    res = trace_sweep(tables, rays, {"max_trace_num": 80}, record_hist=True, tracer=_oracle)
    assert _oracle.calls[-1]["serial"] is False
    _check(res, tables, rays, 80)


def test_family_counts_of_the_parallel_sweep():
    """Where no cap binds, the device counts every root from zero: per family, the starting counts plus its roots'."""
    from oracle import oracle as O

    tables = [_prism_table(0.3, t, cap=10 ** 5) for t in (0.0, 0.02)]
    arrs, fam_ids, unit = pack_rays(tables[0].rays)
    n, F, K = len(arrs["ox"]), len(fam_ids), 2
    flats = [FlatScene(t.components, t.monitors) for t in tables]
    caps0 = np.arange(2 * K * F, dtype=np.int32).reshape(2, K * F) % 5
    per_root = np.concatenate([O.trace(f, dict(arrs, family=np.arange(n, dtype=np.int32)), max_trace_num=80, unit=unit,
                                       record_segments=False, n_families=n)["cap_counts"] for f in flats], axis=1)
    got = _family_counts(per_root, caps0, arrs["family"], K, n, False)
    for k, f in enumerate(flats):
        want = O.trace(f, arrs, max_trace_num=80, unit=unit, record_segments=False, n_families=F,
                       cap_counts=caps0[:, k * F:(k + 1) * F])["cap_counts"]
        np.testing.assert_array_equal(got[k], want)


def _prism_scene():
    t = _prism_table(0.3, 0.0)
    prism = t.components[0]
    saved = []

    def walk(o):
        saved.append((o, o.origin.copy(), np.array(o.transform_matrix, dtype=np.float64), o._bbox))
        for c in getattr(o, "components", []):
            walk(c)

    walk(prism)
    _, fam_ids, _ = pack_rays(t.rays)

    def configure(k):
        for o, org, T, box in saved:
            o.origin, o.transform_matrix, o._bbox = org.copy(), T.copy(), box
        prism.RotZ(0.02 * k - 0.03)
        _seed_counts(t, fam_ids, k)

    return t, prism, configure


def test_sweep_scene_reads_counts_after_configure():
    from oracle import oracle as O

    t, prism, configure = _prism_scene()
    K = 3
    _oracle.calls.clear()
    res = SweepScene(t, [prism]).trace(t.rays, configure, K, t.limit, record_hist=True, tracer=_oracle)
    assert _oracle.calls[-1]["serial"] is True
    arrs, fam_ids, unit = pack_rays(t.rays)
    for k in range(K):
        configure(k)
        flat = FlatScene(t.components, t.monitors)
        caps0 = np.array([[c._interact_count.get(rid, 0) for rid in fam_ids] for c in flat.capslots], np.int32)
        want = O.trace(flat, arrs, max_trace_num=80, unit=unit, record_segments=False, n_families=len(fam_ids),
                       cap_counts=caps0)
        np.testing.assert_array_equal(res.interact_counts[k], want["cap_counts"])
        np.testing.assert_array_equal(res.rows(k)["hit_px"].numpy(), want["hit_px"])
        assert [id(c) for c in res.cap_components[k]] == [id(c) for c in flat.capslots]


def test_bundles_and_abcd_keep_their_refusals():
    tables = [_prism_table(0.3, t) for t in (0.0, 0.02)]
    _oracle.calls.clear()
    bundle = RayBundle.collimated_disc(8, x0=3, radius=0.5, direction=(-1.0, 0.0, 0.0))
    res = trace_sweep(tables, bundle, tracer=_oracle)
    assert _oracle.calls[-1]["caps0"] is None          # every root its own family from zero, as before
    assert res.interact_counts is None and res.family_ids is None
    rays = [ob.Ray([3, y, 0], [-1, 0, 0], wavelength=780e-7, w0=61e-4, id=i) for i, y in enumerate((2.5, 3.0, 3.5))]
    tables[0].monitors.append(ob.Monitor([-4, 0, 0], 12, 12))
    tables[1].monitors.append(ob.Monitor([-4, 0, 0], 12, 12))
    with pytest.raises(NotImplementedError, match="interact-capped"):
        sweep_abcd_matrix(tables, 0, 1, rays)


# ---- gloo: the sharded sweep decides as the one-process sweep and gathers the counts

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(kind, cap, group):
    from tests.test_dist_sweep_cpu import _HostStats

    if kind == "tables":
        tables = [_prism_table(r, t, cap) for r, t in ((0.3, 0.0), (0.2, 0.03), (0.45, -0.05), (0.35, 0.01))]
        _, fam_ids, _ = pack_rays(tables[0].rays)
        for k, t in enumerate(tables):
            _seed_counts(t, fam_ids, k)
        return trace_sweep(tables, tables[0].rays, {"max_trace_num": 80}, record_hist=True, tracer=_oracle, group=group,
                           gather=True, engine=_HostStats())
    t, prism, configure = _prism_scene()
    return SweepScene(t, [prism]).trace(t.rays, configure, 4, {"max_trace_num": 80}, record_hist=True, tracer=_oracle,
                                        group=group, gather=True, engine=_HostStats())


def _worker(rank, world, port, kind, cap, path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
    try:
        _oracle.calls.clear()
        res = _run(kind, cap, True)
        call = _oracle.calls[-1] if _oracle.calls else {"serial": None, "chain_len": -1}
        np.savez(f"{path}_{rank}.npz", counts=res.interact_counts, hist=res.hist_y.numpy(), px=res.hits["hit_px"].numpy(),
                 serial=np.array(-1 if call["serial"] is None else int(call["serial"])), chain=np.array(call["chain_len"]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("kind,world,cap", [("tables", 2, 3), ("tables", 3, 3), ("scene", 3, 3), ("tables", 2, 100)])
def test_sharded_caps_sweep_equals_one_process(tmp_path, kind, world, cap):
    path = str(tmp_path / "rank")
    mp.spawn(_worker, args=(world, _free_port(), kind, cap, path), nprocs=world, join=True)
    _oracle.calls.clear()
    one = _run(kind, cap, None)
    assert _oracle.calls[-1]["serial"] is True
    for r in range(world):
        got = np.load(f"{path}_{r}.npz")
        np.testing.assert_array_equal(got["counts"], one.interact_counts)
        np.testing.assert_array_equal(got["hist"], one.hist_y.numpy())
        np.testing.assert_array_equal(got["px"], one.hits["hit_px"].numpy())
        assert int(got["serial"]) == 1 and int(got["chain"]) == 0
