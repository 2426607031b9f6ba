"""Scene flattener: component tree -> the SoA tables of include/optb.h.

Duck-typed: it only reads attributes, so the same function serves optable_b200's own scene
classes and objects of the reference package (tests feed one scene to both back ends).
Flatten map = SURVEY.md Appendix D. What is read, and where the reference defines it:

  pose            comp.origin, comp.transform_matrix           optical_component.py:19-20
  inverse         np.linalg.inv(transform_matrix)              optical_component.py:108
  lab AABB        comp.bbox (the object's own cached value)    optical_component.py:62-97,
                                                               component_group.py:28-47
  group children  comp.components, DFS pre-order               component_group.py:104-115
  surface         comp.surface (+ class name)                  surfaces.py
  physics         reflectivity / transmission / focal_length / roc / _n1 / _n2
  caps            max_interact_count, _interact_count          optical_component.py:37-38,136-149
"""
from __future__ import annotations

import ctypes as C
import functools
import math
import os

import numpy as np

from . import _abi as A


class FlattenError(NotImplementedError):
    """The scene uses a construct the device tables cannot express (no CPU fallback exists)."""


def _orthonormal(M) -> bool:
    return bool(np.abs(M @ M.T - np.identity(3)).max() < 1e-14)


def _mro_names(obj):
    return {k.__name__ for k in type(obj).__mro__}


def _closure_map(fn):
    code = getattr(fn, "__code__", None)
    cells = getattr(fn, "__closure__", None)
    if code is None or not cells:
        return {}
    return {name: cell.cell_contents for name, cell in zip(code.co_freevars, cells)}


class _Materials:
    def __init__(self, wavelengths_m=None, aux=None):
        self.kind, self.f, self._index = [], [], {}
        self.wavelengths_m, self.aux = wavelengths_m, aux

    def add(self, m) -> int:
        key, kind, row = self._describe(m)
        if key in self._index:
            return self._index[key]
        self._index[key] = len(self.kind)
        self.kind.append(kind)
        self.f.append(row)
        return self._index[key]

    def _lut(self, m):
        """Material(name, n=<any callable>) (material.py:4-21): the device cannot run Python, so the host evaluates
        the callable once per DISTINCT wavelength of the batch (metres = ray.wavelength * ray.unit, the product the
        reference's RefractiveIndex descriptor forms, material.py:54-85) and ships (wavelength, n) pairs sorted by
        wavelength (SURVEY Appendix D). Same callable, same argument, same float: the index a ray sees is the
        reference's, bit for bit."""
        if self.wavelengths_m is None:
            raise FlattenError(f"material {m!r} is an arbitrary n(wavelength) callable: pass the batch's wavelengths "
                               "(FlatScene(..., wavelengths_m=...); OpticalTable.ray_tracing / trace_bundle do)")
        row = [0.0] * A.MF_STRIDE
        ws = sorted({float(w) for w in self.wavelengths_m})
        row[0], row[1] = float(len(self.aux)), float(len(ws))
        for w in ws:
            self.aux.extend([w, float(m.n(w))])
        return ("lut", id(m)), A.MAT_LUT, row

    def _describe(self, m):
        row = [0.0] * A.MF_STRIDE
        if isinstance(m, (int, float, np.integer, np.floating)):
            row[0] = float(m)
            return ("c", row[0]), A.MAT_CONST, row
        if hasattr(m, "Bs") and hasattr(m, "Cs"):
            Bs, Cs = [float(b) for b in m.Bs], [float(c) for c in m.Cs]
            if len(Bs) != 3 or len(Cs) != 3:
                raise FlattenError("Sellmeier materials need exactly 3 (B, C) pairs")
            row[0:3], row[3:6] = Bs, Cs
            return ("s", tuple(Bs), tuple(Cs)), A.MAT_SELLMEIER, row
        nc = getattr(m, "n_const", None)
        if nc is None:
            # reference Material(name, n=<number>) hides the number in a lambda closure (material.py:8-9)
            cm = _closure_map(getattr(m, "n_func", None))
            if set(cm) == {"n"} and isinstance(cm["n"], (int, float, np.integer, np.floating)):
                nc = cm["n"]
        if nc is None:
            return self._lut(m)
        row[0] = float(nc)
        return ("c", row[0]), A.MAT_CONST, row


def _asphere_spec(surface):
    spec = getattr(surface, "asphere_spec", None)
    if spec is None:
        cm = _closure_map(surface.f_asphere)
        if set(cm) == {"R", "kappa", "a4", "a6", "a8"}:
            spec = ("parametric", cm)
        elif set(cm) == {"EFL", "n"}:
            spec = ("exact_spherical", cm)
        else:
            raise FlattenError("ASphere.f_asphere: only the parametric and exact-spherical profiles are supported")
    form, p = spec
    if form == "parametric":
        return A.ASPH_PARAMETRIC, [float(p["R"]), float(p["kappa"]), float(p["a4"]), float(p["a6"]), float(p["a8"])]
    if form == "exact_spherical":
        return A.ASPH_EXACT_SPH, [float(p["EFL"]), float(p["n"]), 0.0, 0.0, 0.0]
    raise FlattenError(f"unknown asphere form {form!r}")


def _csg_spec(surface):
    spec = getattr(surface, "csg", None)
    if spec is not None:
        return spec
    fn = surface.__dict__.get("within_boundary")
    cm = _closure_map(fn)
    if fn is None or set(cm) != {"self", "other"}:
        raise FlattenError("bare Plane surface has no boundary (surfaces.py:29-33)")
    op = "subtract" if "subtract" in fn.__qualname__ else "union" if "union" in fn.__qualname__ else None
    if op is None:
        raise FlattenError("unrecognised composite plane")
    return op, cm["self"], cm["other"]


_BVH_PLANS = {}  # (fanout, n, box bytes) -> hierarchy plan, see FlatScene._wrap_runs


class FlatScene:
    """Numpy tables + bookkeeping for one OpticalTable."""

    def __init__(self, components, monitors=(), wavelengths_m=None):
        """`wavelengths_m`: the distinct wavelengths (metres) of the rays that will be traced; only needed when a
        material of the scene is an arbitrary Python callable (per-wavelength table, see _Materials._lut)."""
        self._ni, self._nf, self._aux = [], [], []
        self._mats = _Materials(wavelengths_m, self._aux)
        self.leaves = []       # leaf index -> component object
        self.capslots = []     # cap slot -> component object
        self.max_children = 0  # most rays one interaction can emit (<=1: no splitting anywhere)
        self._pending_inv = []
        self._row_owner = {}   # id(node_i row) -> the component object that produced it (refresh)
        self._node_of = {}     # id(component) -> node index
        self._grids = []       # (aux offset of the cell table, [child node_i rows in list order]) per lattice group
        for c in components:
            tree = self._visit(c, in_group=False)
            if tree is not None:
                self._emit(tree)
        for off, rows in self._grids:  # node indices are only known after emission
            self._aux[off:off + len(rows)] = [float(r[A.NI_SKIP] - 1) for r in rows]  # a leaf skips to index + 1
        del self._grids
        self._finish_inverses()
        self._owner_of_node = {i: self._row_owner[id(r)] for i, r in enumerate(self._ni) if id(r) in self._row_owner}
        del self._row_owner
        self.node_i = np.ascontiguousarray(np.array(self._ni, dtype=np.int32).reshape(-1, A.NI_STRIDE))
        self.node_f = np.ascontiguousarray(np.array(self._nf, dtype=np.float64).reshape(-1, A.NF_STRIDE))
        self.mat_kind = np.array(self._mats.kind or [0], dtype=np.int32)
        self.mat_f = np.array(self._mats.f or [[1.0] + [0.0] * (A.MF_STRIDE - 1)], dtype=np.float64)
        self.aux = np.array(self._aux or [0.0], dtype=np.float64)
        self.monitors = list(monitors)
        self.mon_f = np.zeros((max(len(self.monitors), 1), A.MON_STRIDE), dtype=np.float64)
        for k, m in enumerate(self.monitors):
            monitor_record(m, self.mon_f[k])
        self.n_nodes = self.node_i.shape[0]
        self.n_leaves = len(self.leaves)
        self.n_materials = int(self.mat_kind.shape[0])  # >= 1 (a dummy row when nothing refracts)
        self.n_monitors = len(self.monitors)
        self.n_capslots = len(self.capslots)

    @property
    def cap_min(self) -> float:
        """Smallest max_interact_count of a capped leaf (+inf without caps)."""
        caps = self.node_f[self.node_i[:, A.NI_CAPSLOT] >= 0, A.NF_CAPMAX]
        return float(caps.min()) if caps.size else float("inf")

    @functools.cached_property
    def has_pass(self) -> bool:
        """Some leaf hands every ray that reaches it back unchanged (A.I_PASS: a Monitor listed as a component)."""
        return bool((self.node_i[:, A.NI_INTER] == A.I_PASS).any())

    def _finish_inverses(self):
        if self._pending_inv:
            # np.linalg.inv on the stack runs the same per-matrix LAPACK solve as the reference's call per
            # component (optical_component.py:108): identical bits, ~30x less Python overhead
            Ts = np.array([nf[A.NF_T:A.NF_T + 9] for _, nf in self._pending_inv], dtype=np.float64).reshape(-1, 3, 3)
            Tinvs = np.linalg.inv(Ts)
            ortho = np.abs(Tinvs @ Tinvs.transpose(0, 2, 1) - np.identity(3)).max(axis=(1, 2)) < 1e-14
            for (ni, nf), Ti, flag in zip(self._pending_inv, Tinvs.reshape(-1, 9).tolist(), ortho.tolist()):
                nf[A.NF_TINV:A.NF_TINV + 9] = Ti
                ni[A.NI_ORTHO] = int(flag)
        self._pending_inv = []

    # -- incremental re-flatten (SURVEY 8f item 3: the GUI loop moves ONE component per slider event) ----------
    def refresh(self, component):
        """Re-read one component (leaf, or group without a synthetic box hierarchy) after its pose or parameters
        changed, rewrite its rows of the tables in place and re-read the cached boxes of its ancestor groups (the
        reference's groups keep their own, possibly stale, `.bbox`: SURVEY A.2 -- whatever the objects say is what
        gets flattened). Returns the list of node indices whose rows changed (for Scene.update_nodes), or None when
        the change cannot be expressed in place (topology, materials, polygons, lattice descriptors or cap slots would
        move): the caller then builds a new FlatScene."""
        first = self._node_of.get(id(component))
        if first is None:
            return None
        end = int(self.node_i[first, A.NI_SKIP])
        owners = self._owner_of_node
        if any(i not in owners for i in range(first, end)) or (self.node_i[first:end, A.NI_GEOM] == A.G_GRID).any():
            return None   # synthetic wrappers / lattice inside: rebuild
        in_group = bool(self.node_i[first, A.NI_AABB]) if self.node_i[first, A.NI_GEOM] not in (A.G_GROUP, A.G_GRID) else first in self._parents()
        # re-visit into scratch lists with the bookkeeping of this scene (materials, aux, leaves, caps must not grow)
        keep = (self._ni, self._nf, self.leaves, self.capslots, len(self._aux), len(self._mats.kind))
        self._ni, self._nf, self.leaves, self.capslots = [], [], list(self.leaves), list(self.capslots)
        self._row_owner, node_of_backup = {}, dict(self._node_of)
        n_leaves0, n_caps0 = len(self.leaves), len(self.capslots)
        try:
            tree = self._visit(component, in_group=in_group)
            if tree is None:
                return None
            self._emit(tree)
            self._finish_inverses()
            new_i = np.array(self._ni, dtype=np.int32).reshape(-1, A.NI_STRIDE)
            new_f = np.array(self._nf, dtype=np.float64).reshape(-1, A.NF_STRIDE)
            grew = len(self._aux) != keep[4] or len(self._mats.kind) != keep[5] or len(self.capslots) != n_caps0 + int((new_i[:, A.NI_CAPSLOT] >= 0).sum())
        finally:
            new_leaves = self.leaves[n_leaves0:]
            self._ni, self._nf, self.leaves, self.capslots = keep[0], keep[1], keep[2], keep[3]
            del self._aux[keep[4]:]
            self._node_of = node_of_backup
            self._row_owner = {}
        old_i = self.node_i[first:end]
        if grew or new_i.shape[0] != end - first or not np.array_equal(new_i[:, A.NI_GEOM], old_i[:, A.NI_GEOM]):
            return None
        # keep the global numbering of the old rows (skip pointers, dense leaf numbers, cap slots)
        new_i[:, A.NI_SKIP] += first
        new_i[:, A.NI_LEAF] = old_i[:, A.NI_LEAF]
        new_i[:, A.NI_CAPSLOT] = old_i[:, A.NI_CAPSLOT]
        if not np.array_equal(new_i[:, [A.NI_AUX, A.NI_MAT1, A.NI_MAT2]], old_i[:, [A.NI_AUX, A.NI_MAT1, A.NI_MAT2]]):
            return None
        self.node_i[first:end] = new_i
        self.node_f[first:end] = new_f
        for k, leaf in zip(old_i[:, A.NI_LEAF][old_i[:, A.NI_LEAF] >= 0].tolist(), new_leaves):
            self.leaves[k] = leaf
        changed = list(range(first, end))
        parents = self._parents()
        p = parents.get(first, -1)
        while p >= 0:  # ancestors: re-read the object's own box; synthetic wrappers take the union of their children
            owner = owners.get(p)
            if owner is not None:
                box = [float(v) for v in owner.bbox]
            else:
                kids, j = [], p + 1
                while j < self.node_i[p, A.NI_SKIP]:
                    kids.append(self.node_f[j, A.NF_AABB:A.NF_AABB + 6])
                    j = int(self.node_i[j, A.NI_SKIP])
                kids = np.array(kids)
                lo, hi = kids[:, 0::2].min(axis=0), kids[:, 1::2].max(axis=0)
                box = [lo[0], hi[0], lo[1], hi[1], lo[2], hi[2]]
            if not np.array_equal(self.node_f[p, A.NF_AABB:A.NF_AABB + 6], box):
                self.node_f[p, A.NF_AABB:A.NF_AABB + 6] = box
                changed.append(p)
            p = parents.get(p, -1)
        return changed

    def _parents(self):
        """node -> parent node (cached): from the skip pointers of the pre-order table."""
        cache = getattr(self, "_parent_cache", None)
        if cache is None:
            cache, open_ = {}, []
            for i in range(self.n_nodes):
                while open_ and self.node_i[open_[-1], A.NI_SKIP] <= i:
                    open_.pop()
                if open_:
                    cache[i] = open_[-1]
                if self.node_i[i, A.NI_GEOM] in (A.G_GROUP, A.G_GRID):
                    open_.append(i)
            self._parent_cache = cache
        return cache

    # -- tree walk ---------------------------------------------------------------------------
    # Large groups get synthetic sub-groups over contiguous runs of children (a BVH in list order). The box of a
    # synthetic group is the union of its members' own boxes, and the slab test is monotone under box inclusion
    # (bit for bit: subtraction and multiplication by a fixed reciprocal are monotone in floating point), so a
    # child whose box the ray hits is never culled by a wrapper: the set of leaves that get tested, and their
    # order, are exactly the reference's (component_group.py:104-115), only reached in O(log n) box tests.
    BVH_FANOUT = int(os.environ.get("OPTB_BVH_FANOUT", "4"))
    BVH_MIN_CHILDREN = int(os.environ.get("OPTB_BVH_MIN_CHILDREN", "9"))

    GRID_MIN_CHILDREN = int(os.environ.get("OPTB_GRID_MIN_CHILDREN", "32"))

    def _grid(self, ni, children):
        """Regular arrays (MMA / MLA / DMD, component_group.py:228-391): when the lab boxes of a group's leaf children
        sit on a 2-D lattice c00 + i U + j V (list order k = i * n_inner + j; up to 8 trailing children may be off the
        lattice, e.g. the back face of an MMA), write the lattice descriptor of include/optb.h (OPTB_GRID_*) into the
        aux pool and mark the group OPTB_G_GRID. Pure geometry of the children's own boxes: nothing here depends on
        the class of the group. The box hierarchy over the children is still emitted; it serves rays for which the
        lattice window would be large (in-plane rays) or the slab test takes its parallel-axis branch."""
        if any(c[0][A.NI_GEOM] in (A.G_GROUP, A.G_GRID) or c[0][A.NI_CAPSLOT] >= 0 for c in children):
            return
        B = np.array([c[1][A.NF_AABB:A.NF_AABB + 6] for c in children], dtype=np.float64)
        C, H = (B[:, 0::2] + B[:, 1::2]) / 2, (B[:, 1::2] - B[:, 0::2]) / 2
        n = len(children)
        V = C[1] - C[0]
        pitch = float(np.linalg.norm(V))
        if not pitch > 0:
            return
        tol = 0.02 * pitch
        step = np.linalg.norm(np.diff(C, axis=0) - V, axis=1)          # deviation of every first difference from V
        breaks = np.nonzero(step > tol)[0]
        n_inner = int(breaks[0]) + 1 if len(breaks) else n
        n_outer = 1
        if n_inner < n:
            U = C[n_inner] - C[0]
            n_outer = 1
            while (n_outer + 1) * n_inner <= n:
                k0 = n_outer * n_inner
                pred = C[0] + n_outer * U + np.arange(n_inner)[:, None] * V
                if np.linalg.norm(C[k0:k0 + n_inner] - pred, axis=1).max() > 4 * tol:
                    break
                n_outer += 1
        m = n_outer * n_inner
        if n - m > 8 or m < self.GRID_MIN_CHILDREN:
            return
        if n_inner > 1:
            V = (C[n_inner - 1] - C[0]) / (n_inner - 1)
        if n_outer > 1:
            U = (C[(n_outer - 1) * n_inner] - C[0]) / (n_outer - 1)
        else:  # one row: complete the plane with the direction in which the boxes are thinnest
            e = np.identity(3)[int(np.argmin(H[:m].max(axis=0)))]
            nh = e - (e @ V) * V / (V @ V)
            if np.linalg.norm(nh) < 1e-6:
                return
            nh /= np.linalg.norm(nh)
            U = np.cross(nh, V)
        nhat = np.cross(U, V)
        if np.linalg.norm(nhat) < 1e-12 * np.linalg.norm(U) * np.linalg.norm(V):
            return
        nhat /= np.linalg.norm(nhat)
        ii, jj = np.divmod(np.arange(m), n_inner)
        L = C[0] + ii[:, None] * U + jj[:, None] * V
        dev = np.linalg.norm(C[:m] - L, axis=1)
        R = float((np.linalg.norm(H[:m], axis=1) + dev).max()) * (1 + 1e-6) + 1e-9 * (1.0 + float(np.abs(C).max()))
        Ud = np.cross(V, nhat) / (U @ np.cross(V, nhat))
        Vd = np.cross(nhat, U) / (V @ np.cross(nhat, U))
        rho_a, rho_b = R * float(np.linalg.norm(Ud)), R * float(np.linalg.norm(Vd))
        if rho_a > 2.0 or rho_b > 2.0:
            return  # boxes much larger than the lattice spacing: the window would hold too many cells to pay off
        off = len(self._aux)
        self._aux.extend([float(n_outer), float(n_inner), float(n - m), R, *C[0].tolist(), *nhat.tolist(), *Ud.tolist(),
                          *Vd.tolist(), rho_a, rho_b])
        assert len(self._aux) - off == A.GRID_CELLS
        self._grids.append((len(self._aux), [c[0] for c in children]))
        self._aux.extend([0.0] * n)
        ni[A.NI_GEOM], ni[A.NI_AUX] = A.G_GRID, off

    @staticmethod
    def _blank():
        ni, nf = [0] * A.NI_STRIDE, [0.0] * A.NF_STRIDE
        ni[A.NI_CAPSLOT] = -1
        ni[A.NI_LEAF] = -1
        return ni, nf

    def _emit(self, tree):
        """Append a (sub)tree in pre-order; `skip` = index of the first node after the subtree."""
        ni, nf, children = tree
        comp = self._row_owner.get(id(ni))
        if comp is not None:
            self._node_of[id(comp)] = len(self._ni)
        self._ni.append(ni)
        self._nf.append(nf)
        for child in children:
            self._emit(child)
        ni[A.NI_SKIP] = len(self._ni)

    def _synthetic(self, members):
        """A box-only group node over `members` (list of trees); box = union of the members' own boxes."""
        ni, nf = self._blank()
        ni[A.NI_GEOM], ni[A.NI_AABB] = A.G_GROUP, 1
        boxes = np.array([m[1][A.NF_AABB:A.NF_AABB + 6] for m in members], dtype=np.float64)
        lo, hi = boxes[:, 0::2].min(axis=0), boxes[:, 1::2].max(axis=0)
        nf[A.NF_AABB:A.NF_AABB + 6] = [float(lo[0]), float(hi[0]), float(lo[1]), float(hi[1]), float(lo[2]), float(hi[2])]
        return ni, nf, members

    def _wrap_runs(self, children):
        """Hierarchy over a child list that keeps the list order: every node covers a contiguous run, runs are cut
        where the surface-area heuristic is cheapest (for a row-major array: first between rows, then inside a
        row), at most BVH_FANOUT runs per node."""
        boxes = np.array([c[1][A.NF_AABB:A.NF_AABB + 6] for c in children], dtype=np.float64)
        F = max(2, self.BVH_FANOUT)
        # the hierarchy is a pure function of the children's boxes: keep it across calls (a GUI loop or a parameter
        # sweep re-flattens the same arrays many times); plan = nested (box, members) tuples over child indices
        key = (F, boxes.shape[0], boxes.tobytes())
        plan = _BVH_PLANS.get(key)
        if plan is not None:
            return self._from_plan(plan, children)

        def area(lo, hi):
            d = np.maximum(hi - lo, 0.0)
            return 2.0 * (d[..., 0] * d[..., 1] + d[..., 1] * d[..., 2] + d[..., 2] * d[..., 0]) + 1e-300

        def best_cut(a, b):
            """Cheapest cut of [a, b) into [a, s) + [s, b); returns (cost, s)."""
            blo, bhi = boxes[a:b, 0::2], boxes[a:b, 1::2]
            pl, ph = np.minimum.accumulate(blo, 0), np.maximum.accumulate(bhi, 0)
            sl, sh = np.minimum.accumulate(blo[::-1], 0)[::-1], np.maximum.accumulate(bhi[::-1], 0)[::-1]
            k = np.arange(1, b - a)
            cost = area(pl[:-1], ph[:-1]) * k + area(sl[1:], sh[1:]) * (b - a - k)
            j = int(np.argmin(cost))
            return float(cost[j]), a + 1 + j

        def build(a, b):
            """Trees that stand for the run [a, b) inside its parent (at most F of them)."""
            if b - a <= F:
                return list(children[a:b])
            parts = [(a, b)]
            while len(parts) < F:
                # cut the part whose cut saves the most (largest part first is a good proxy and O(n log n))
                k = max(range(len(parts)), key=lambda i: parts[i][1] - parts[i][0])
                pa, pb = parts[k]
                if pb - pa < 2:
                    break
                _, s = best_cut(pa, pb)
                parts[k:k + 1] = [(pa, s), (s, pb)]
            out = []
            for pa, pb in parts:
                out.append(children[pa] if pb - pa == 1 else self._synthetic(build(pa, pb)))
            return out

        built = build(0, len(children))
        index = {id(c): k for k, c in enumerate(children)}

        def to_plan(tree):
            k = index.get(id(tree))
            return k if k is not None else (tuple(tree[1][A.NF_AABB:A.NF_AABB + 6]), tuple(to_plan(m) for m in tree[2]))

        if len(_BVH_PLANS) >= 64:
            _BVH_PLANS.clear()
        _BVH_PLANS[key] = tuple(to_plan(t) for t in built)
        return built

    def _from_plan(self, plan, children):
        out = []
        for item in plan:
            if isinstance(item, int):
                out.append(children[item])
            else:
                ni, nf = self._blank()
                ni[A.NI_GEOM], ni[A.NI_AABB] = A.G_GROUP, 1
                nf[A.NF_AABB:A.NF_AABB + 6] = item[0]
                out.append((ni, nf, self._from_plan(item[1], children)))
        return out

    def _visit(self, comp, in_group):
        """Component (sub)tree -> (node_i row, node_f row, children) or None when nothing can be hit."""
        if hasattr(comp, "components") and "ComponentGroup" in _mro_names(comp):
            if len(comp.components) == 0:
                return None  # nothing to hit (the reference would raise in merge_bboxs on first use)
            ni, nf = self._blank()
            self._row_owner[id(ni)] = comp
            ni[A.NI_GEOM] = A.G_GROUP
            ni[A.NI_AABB] = 1
            nf[A.NF_AABB:A.NF_AABB + 6] = [float(v) for v in comp.bbox]
            children = [t for t in (self._visit(child, in_group=True) for child in comp.components) if t is not None]
            if len(children) >= self.GRID_MIN_CHILDREN:
                self._grid(ni, children)
            if len(children) >= self.BVH_MIN_CHILDREN:
                children = self._wrap_runs(children)
            return ni, nf, children
        names = _mro_names(comp)
        sname = type(comp.surface).__name__
        if "PointObj" in names or sname == "Point":
            return None  # Point.f = |P| never changes sign -> never hit (surfaces.py:68-86)
        ni, nf = self._blank()
        self._row_owner[id(ni)] = comp
        ni[A.NI_AABB] = 1 if in_group else 0
        ni[A.NI_LEAF] = len(self.leaves)
        self.leaves.append(comp)
        T = np.asarray(comp.transform_matrix, dtype=np.float64)
        nf[A.NF_ORIGIN:A.NF_ORIGIN + 3] = [float(v) for v in comp.origin]
        nf[A.NF_T:A.NF_T + 9] = T.reshape(-1).tolist()
        self._pending_inv.append((ni, nf))  # Tinv / orthonormal flag: one batched LAPACK call at the end
        if in_group:
            nf[A.NF_AABB:A.NF_AABB + 6] = [float(v) for v in comp.bbox]
        self._geometry(comp.surface, sname, ni, nf)
        self._physics(comp, names, ni, nf)
        cap = getattr(comp, "max_interact_count", None)
        if cap is not None:
            ni[A.NI_CAPSLOT] = len(self.capslots)
            nf[A.NF_CAPMAX] = float(cap)
            self.capslots.append(comp)
        return ni, nf, []

    def _poly_record(self, s):
        off = len(self._aux)
        v2 = np.asarray(s._verts2d, dtype=np.float64)
        u, v = s._basis
        rec = [float(len(v2))] + [float(x) for x in s._normal] + [float(x) for x in s.vertices[0]]
        rec += [float(x) for x in u] + [float(x) for x in v] + [float(x) for x in s._bbox]
        assert len(rec) == A.POLY_HEADER
        self._aux.extend(rec + v2.reshape(-1).tolist())
        return off

    def _planar_shape(self, s):
        """(kind, p0, p1) of a simple planar shape (also used as CSG operand)."""
        n = type(s).__name__
        if n == "Circle":
            return A.G_CIRCLE, float(s.radius), 0.0
        if n == "Rectangle":
            return A.G_RECT, s.width / 2, s.height / 2
        if n == "Polygon" and s.planar:
            return A.G_POLY2D, float(self._poly_record(s)), 0.0
        raise FlattenError(f"surface {n} cannot be used as a planar aperture operand")

    def _csg_program(self, s, prog, depth):
        """Postfix tokens (code, a, b) of a composite plane; shapes push, operators pop two (include/optb.h)."""
        if depth > 64:
            raise FlattenError("composite plane nests too deep")
        if type(s).__name__ != "Plane":
            prog.extend(float(v) for v in self._planar_shape(s))
            return
        op, sa, sb = _csg_spec(s)
        self._csg_program(sa, prog, depth + 1)
        self._csg_program(sb, prog, depth + 1)
        prog.extend([float(A.CSG_SUBTRACT if op == "subtract" else A.CSG_UNION), 0.0, 0.0])

    def _geometry(self, s, sname, ni, nf):
        p = [0.0] * 8
        if sname == "Circle":
            ni[A.NI_GEOM], p[0] = A.G_CIRCLE, float(s.radius)
        elif sname == "Rectangle":
            ni[A.NI_GEOM] = A.G_RECT
            p[0], p[1] = s.width / 2, s.height / 2
        elif sname == "Sphere":
            ni[A.NI_GEOM] = A.G_SPHERE
            p[0], p[1] = float(s.radius), float(s.height)
            p[2:8] = [float(v) for v in s.get_bbox_local()]
        elif sname == "ASphere":
            ni[A.NI_GEOM] = A.G_ASPHERE
            form, coeffs = _asphere_spec(s)
            ni[A.NI_AUX] = form
            p[0] = float(s.radius)
            p[1:6] = coeffs
            p[6], p[7] = float(s.xmin), float(s.xmax)
        elif sname == "Cylinder":
            ni[A.NI_GEOM] = A.G_CYL
            p[0], p[1] = float(s.radius), float(s.height)
            p[2], p[3] = float(s.theta_range[0]), float(s.theta_range[1])
        elif sname == "Polygon":
            ni[A.NI_GEOM] = A.G_POLY2D if s.planar else A.G_POLY3D
            ni[A.NI_AUX] = self._poly_record(s)
        elif sname == "Plane":
            op, sa, sb = _csg_spec(s)
            ni[A.NI_GEOM] = A.G_CSG
            if type(sa).__name__ != "Plane" and type(sb).__name__ != "Plane":
                p[0] = 0.0 if op == "subtract" else 1.0
                p[1], p[2], p[3] = self._planar_shape(sa)
                p[4], p[5], p[6] = self._planar_shape(sb)
            else:
                # an operand is itself a union / subtract (surfaces.py:100-136 compose freely): postfix program
                prog = []
                self._csg_program(s, prog, 0)
                p[0] = 2.0
                ni[A.NI_AUX] = len(self._aux)
                self._aux.extend([float(len(prog) // 3)] + prog)
        else:
            raise FlattenError(f"unsupported surface class {sname}")
        nf[A.NF_P:A.NF_P + 8] = p

    def _physics(self, comp, names, ni, nf):
        if "BaseMirror" in names:
            ni[A.NI_INTER] = A.I_MIRROR
            nf[A.NF_REFL], nf[A.NF_TRANS] = float(comp.reflectivity), float(comp.transmission)
            nchild = int(comp.reflectivity > 0) + int(comp.transmission > 0)
        elif "BaseRefraciveSurface" in names:
            ni[A.NI_INTER] = A.I_REFRACT
            nf[A.NF_REFL], nf[A.NF_TRANS] = float(comp.reflectivity), float(comp.transmission)
            d = vars(comp)
            ni[A.NI_MAT1] = self._mats.add(d["_n1"])
            ni[A.NI_MAT2] = self._mats.add(d["_n2"])
            roc = getattr(comp, "roc", math.inf)
            if callable(roc):
                if ni[A.NI_GEOM] != A.G_ASPHERE:
                    raise FlattenError("callable roc is only supported for ASphere surfaces")
                ni[A.NI_ROCKIND] = A.ROC_ASPHERE_FD
            elif math.isinf(float(roc)) and float(roc) > 0:
                ni[A.NI_ROCKIND] = A.ROC_INF
                nf[A.NF_ROC] = math.inf
            else:
                ni[A.NI_ROCKIND] = A.ROC_CONST
                nf[A.NF_ROC] = float(roc)
            nchild = 2 if comp.reflectivity > 0 else 1
        elif "Lens" in names:
            ni[A.NI_INTER] = A.I_THINLENS
            nf[A.NF_FOCAL], nf[A.NF_TRANS] = float(comp.focal_length), float(comp.transmission)
            nchild = 1
        elif "Block" in names:
            ni[A.NI_INTER] = A.I_ABSORB
            nchild = 0
        elif "Monitor" in names:
            # Monitor.interact_local returns the ray itself (monitor.py:174-175): a monitor listed as a COMPONENT hands
            # every ray that reaches it back unchanged, to be hit again until the pop cap (SURVEY a18)
            ni[A.NI_INTER] = A.I_PASS
            nf[A.NF_FOCAL], nf[A.NF_TRANS] = math.inf, 1.0   # the device runs it as a thin lens of no power at t = 0
            nchild = 1
        else:
            raise FlattenError(f"component class {type(comp).__name__} has no device interaction")
        self.max_children = max(self.max_children, nchild)

    # -- (de)serialisation: the tables alone define the device scene ------------------------------
    TABLES = ("node_i", "node_f", "mat_kind", "mat_f", "mon_f", "aux")

    def to_arrays(self) -> dict:
        d = {k: getattr(self, k) for k in self.TABLES}
        d["counts"] = np.array([self.n_leaves, self.n_materials, self.n_monitors, self.n_capslots, self.max_children],
                               dtype=np.int64)
        return d

    @classmethod
    def from_arrays(cls, d) -> "FlatScene":
        self = cls.__new__(cls)
        self.node_i = np.ascontiguousarray(d["node_i"], dtype=np.int32).reshape(-1, A.NI_STRIDE)
        self.node_f = np.ascontiguousarray(d["node_f"], dtype=np.float64).reshape(-1, A.NF_STRIDE)
        self.mat_kind = np.ascontiguousarray(d["mat_kind"], dtype=np.int32)
        self.mat_f = np.ascontiguousarray(d["mat_f"], dtype=np.float64)
        self.mon_f = np.ascontiguousarray(d["mon_f"], dtype=np.float64)
        self.aux = np.ascontiguousarray(d["aux"], dtype=np.float64)
        c = [int(v) for v in d["counts"]]
        self.n_leaves, self.n_materials, self.n_monitors, self.n_capslots, self.max_children = c
        self.n_nodes = self.node_i.shape[0]
        self.n_materials = int(self.mat_kind.shape[0])
        self.leaves, self.capslots, self.monitors = [], [], []
        return self

    # -- ABI view ----------------------------------------------------------------------------
    def desc(self) -> A.SceneDesc:
        d = A.SceneDesc()
        d.abi_version = A.ABI_VERSION
        d.n_nodes, d.n_leaves = self.n_nodes, self.n_leaves
        d.n_materials, d.n_monitors, d.n_capslots = self.n_materials, self.n_monitors, self.n_capslots
        d.n_aux = self.aux.size
        d.node_i = self.node_i.ctypes.data
        d.node_f = self.node_f.ctypes.data
        d.mat_kind = self.mat_kind.ctypes.data
        d.mat_f = self.mat_f.ctypes.data
        d.mon_f = self.mon_f.ctypes.data
        d.aux = self.aux.ctypes.data
        d._keepalive = self  # arrays must outlive the struct
        return d


def monitor_record(m, row):
    """Write monitor m's OPTB_MON_* record (include/optb.h) into `row` (float64 [A.MON_STRIDE]) and return it."""
    T = np.asarray(m.transform_matrix, dtype=np.float64)
    row[A.MON_ORIGIN:A.MON_ORIGIN + 3] = np.asarray(m.origin, dtype=np.float64)
    row[A.MON_TINV:A.MON_TINV + 9] = np.linalg.inv(T).reshape(-1)
    row[A.MON_ORTHO] = float(_orthonormal(np.linalg.inv(T)))
    row[A.MON_HW] = m.width / 2
    row[A.MON_HH] = m.height / 2
    row[A.MON_TY:A.MON_TY + 3] = T @ np.array([0.0, 1.0, 0.0])
    row[A.MON_TZ:A.MON_TZ + 3] = T @ np.array([0.0, 0.0, 1.0])
    return row


def material_value(m, wavelength_m: float = 0.0) -> float:
    """Index of a Material-like object or a plain number at a wavelength in metres."""
    if isinstance(m, (int, float, np.integer, np.floating)):
        return float(m)
    return float(m.n(wavelength_m))


def pack_rays(rays):
    """list[Ray] -> dict of SoA numpy arrays (include/optb.h optb_rays), family table, unit.

    Reads the fields Ray.__init__ sets (ray.py:63-105): origin, _direction, intensity, wavelength,
    length (None -> +inf), alive, qo (None -> flag), _pathlength, n, _id, unit.
    """
    n = len(rays)
    f64 = lambda it: np.fromiter(it, dtype=np.float64, count=n)
    O = np.array([r.origin for r in rays], dtype=np.float64).reshape(n, 3)
    D = np.array([r._direction for r in rays], dtype=np.float64).reshape(n, 3)
    out = {"ox": O[:, 0].copy(), "oy": O[:, 1].copy(), "oz": O[:, 2].copy(),
           "dx": D[:, 0].copy(), "dy": D[:, 1].copy(), "dz": D[:, 2].copy(),
           "intensity": f64(r.intensity for r in rays),
           "wavelength": f64((r.wavelength if r.wavelength is not None else 0.0) for r in rays)}
    qs = [r.qo for r in rays]
    hasq = np.fromiter((q is not None for q in qs), dtype=bool, count=n)
    qc = np.fromiter((0j if q is None else q for q in qs), dtype=np.complex128, count=n)
    out["q_re"], out["q_im"] = qc.real.copy(), qc.imag.copy()
    out["pathlength"] = f64(r._pathlength for r in rays)
    out["n_medium"] = f64(r.n for r in rays)
    out["length"] = f64((math.inf if r.length is None else r.length) for r in rays)
    out = {k: out[k] for k in A.RAY_F64}
    alive = np.fromiter((bool(r.alive) for r in rays), dtype=bool, count=n)
    flags = (np.where(hasq, A.RF_HASQ, 0) | np.where(alive, A.RF_ALIVE, 0)).astype(np.uint32)
    fam_index, fam_ids = {}, []
    fam = [0] * n
    for i, r in enumerate(rays):
        rid = r._id
        j = fam_index.get(rid)
        if j is None:
            j = fam_index[rid] = len(fam_ids)
            fam_ids.append(rid)
        fam[i] = j
    family = np.array(fam, dtype=np.int32).reshape(n)
    units = {float(r.unit) for r in rays}
    if len(units) > 1:
        raise FlattenError("rays with different .unit in one batch are not supported")
    out["flags"], out["family"] = flags, family
    return out, fam_ids, (units.pop() if units else 1e-2)


def batch_wavelengths_m(wavelength_column, unit):
    """Distinct values of ray.wavelength * ray.unit of a batch (what Material.n is called with, optical_component.py:627-628)."""
    w = np.unique(np.asarray(wavelength_column, dtype=np.float64).reshape(-1))
    return (w * float(unit)).tolist()


def rays_struct(arrs, n=None) -> A.Rays:
    """ctypes view over a dict of numpy arrays (host pointers)."""
    s = A.Rays()
    s.n = int(n if n is not None else max(len(arrs[k]) for k in A.RAY_F64 if arrs.get(k) is not None))
    s.broadcast = 0
    for bit, k in enumerate(A.RAY_F64):
        a = arrs.get(k)
        setattr(s, k, None if a is None else a.ctypes.data)
        if a is not None and len(a) == 1 and s.n != 1:
            s.broadcast |= 1 << bit
    for k in ("flags", "family"):
        a = arrs.get(k)
        setattr(s, k, None if a is None else a.ctypes.data)
    s._keepalive = arrs
    return s


def trace_cap(perfomance_limit) -> int:
    """MAX_TRACE_NUM semantics (optical_table.py:86-97): loop runs while trace_num < MAX."""
    cap = 2000
    if perfomance_limit is not None and "max_trace_num" in perfomance_limit:
        cap = perfomance_limit["max_trace_num"]
    return max(0, int(math.ceil(cap)))
