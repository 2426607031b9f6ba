"""The benchmark workloads of the ray_tracing path (BASELINE.json configs[1..4], SURVEY 8(d) C2-C5): scene builders
and synthetic ray bundles. Shared by bench.py, __graft_entry__.smoke() and the parity tests (tests/scenes.py
re-exports the builders), so the benchmark of record does not depend on the test package.

Every builder takes a namespace `ns` exposing the optable public names (Ray, Mirror, Lens, ...): the reference
package in the build container, optable_b200 everywhere. The geometry restates the reference's example scripts
(examples/*.py, cited per builder). Bundles are generated from the ray index with splitmix64 (bundle.uniform01), so
any shard of any batch is produced independently and identically on every rank.
"""
from __future__ import annotations

import numpy as np

SEED = 20261018


class Scene:
    def __init__(self, components, rays, monitors=(), limit=None):
        self.components, self.rays, self.monitors, self.limit = list(components), list(rays), list(monitors), limit

    def flat(self):
        """Device tables of the scene (the rays' wavelengths ride along for per-wavelength material tables)."""
        from .flatten import FlatScene

        wl = sorted({(0.0 if r.wavelength is None else float(r.wavelength)) * float(r.unit) for r in self.rays})
        return FlatScene(self.components, self.monitors, wavelengths_m=wl or None)


def cavity(ns, dt1=0.02, dt2=0.02, gaussian=False, n_rays=1, limit=None):
    """examples/cavity_4mir.py:17-40 (misaligned: escapes after 21 bounces; aligned: runs to the cap)."""
    L, D, R = 10 * 4 / 3, 4, 0.9
    comps = [
        ns.Mirror([0, 0, 0], radius=D, reflectivity=R).RotZ(-np.pi / 4),
        ns.Mirror([L, 0, 0], radius=D, reflectivity=R).RotZ(+np.pi / 4 + dt1),
        ns.Mirror([L, -L, 0], radius=D, reflectivity=R).RotZ(-np.pi / 4 + dt2),
        ns.Mirror([0, -L, 0], radius=D, reflectivity=R).RotZ(+np.pi / 4),
    ]
    rng = np.random.default_rng(SEED)
    rays = []
    for i in range(n_rays):
        kw = dict(wavelength=780e-7, w0=61e-4) if gaussian else {}
        if i == 0:
            rays.append(ns.Ray([2, 0, 0], [1, 0, 0], **kw))
        else:
            y, z = rng.uniform(-1, 1, 2)
            ty, tz = rng.uniform(-2e-5, 2e-5, 2)
            rays.append(ns.Ray([2, y, z], [1, ty, tz], **kw))
    return Scene(comps, rays, limit=limit)


def asphere_lens9(ns, origin):
    """examples/calibrate_4f.py:149-180 (LENS == 9)."""
    EFL, CT = 43.17, 0.8
    n = ns.Glass_UVFS()
    R = EFL * (n.n(780e-9) - 1)
    return ns.ASphericParametricLens(origin, CT=CT, diameter=2.54 * 3, R=R, n=n, kappa=-1.03113,
                                     a4=-0.00223 * (1e-3 / 1e-2) ** 4, a6=0.006353 * (1e-3 / 1e-2) ** 6, name="L0")


def telescope_4f(ns, n_rays=7, disc=True):
    """C2: two LENS-9 aspheres as a 4f relay with monitors at x=0 and x=2F1+2F2
    (optical_table.py:328-336 geometry; SURVEY 8(d))."""
    F1 = F2 = 43.17
    l0 = asphere_lens9(ns, [F1, 0, 0])
    l1 = asphere_lens9(ns, [F1 + 2 * F2, 0, 0]).RotZ(np.pi)
    mon0 = ns.Monitor([0, 0, 0], width=5, height=5)
    mon1 = ns.Monitor([2 * F1 + 2 * F2, 0, 0], width=5, height=5)
    rng = np.random.default_rng(SEED + 2)
    rays = []
    for i in range(n_rays):
        if disc:
            rr, th = 3.0 * np.sqrt(rng.uniform()), rng.uniform(0, 2 * np.pi)
            y, z = rr * np.cos(th), rr * np.sin(th)
        else:
            y, z = (i - n_rays // 2) * 0.6, 0.0
        rays.append(ns.Ray([-10, y, z], [1, 0, 0], wavelength=780e-7, w0=61e-4))
    return Scene([l0, l1], rays, [mon0, mon1])


def telescope_4f_grid(ns, F1, F2):
    """The C2 relay as `calibrate_symmetric_4f` scans it (optical_table.py:328-336): lens 1 stays at its focal length
    F0 = 43.17, lens 2 sits at F0 + F1 + F2 and monitor 1 at F0 + F1 + 2 F2 (F1 = F2 = F0: the C2 scene). No rays."""
    F0 = 43.17
    l0 = asphere_lens9(ns, [F0, 0, 0])
    l1 = asphere_lens9(ns, [F0 + F1 + F2, 0, 0]).RotZ(np.pi)
    mon0 = ns.Monitor([0, 0, 0], width=5, height=5)
    mon1 = ns.Monitor([F0 + F1 + 2 * F2, 0, 0], width=5, height=5)
    return Scene([l0, l1], [], [mon0, mon1])


def ripa(ns, n_rays=1, limit=300, jitter=True):
    """C5: examples/ripa_gen2_lensless.py:54-299 (7,689 leaves: two MMA arrays of 80x15 and 80x80 spherical
    micro-mirrors, a 80x1 back MMA, fold mirrors, a TriangularPrism, a Block; nesting depth 2; 3 monitors).
    Rays: the script's R1rays0 plus copies with origin jitter +-R1w0 and angle jitter +-1e-3 (SURVEY 8(d))."""
    from scipy.optimize import brentq

    BW, R1ultraR, R1R, wl = 6.83, 0.9999, 0.98, 780e-7
    DMLA, R1NMLA, R1MMLA = 420e-4, 80, 15
    Lrt = 3e8 / (2 * BW * 1e9) / 0.01
    R1MMAshify = DMLA / (R1MMLA + 1)
    R1ZRay = (R1MMLA / 2) * DMLA
    R1W, R1H = DMLA * R1NMLA, DMLA * R1MMLA
    R1d = np.sqrt((Lrt / 2) ** 2 - (R1MMAshify / 2) ** 2 - (DMLA / 2) ** 2)
    R1MLAroc = Lrt * 1.0
    R1w0 = np.sqrt(wl * (np.sqrt(Lrt * (R1MLAroc / 2 - Lrt / 4))) / np.pi)
    R1theta0 = np.arctan(DMLA / R1d / 2)
    vec_input = np.array([R1d, -R1MMAshify / 2, DMLA / 2])
    vec_input = vec_input / np.linalg.norm(vec_input)
    vec_output = np.array([-R1d, -R1MMAshify / 2, DMLA / 2])
    vec_output = vec_output / np.linalg.norm(vec_output)
    vec_output_projxz = np.array([vec_output[0], vec_output[2]])
    vec_output_projxz /= np.linalg.norm(vec_output_projxz)
    origin_output = np.array([0, -R1MMAshify / 2, R1ZRay])
    R1DMMA = 0.1

    def hit_point(t):
        p = origin_output + vec_output * t
        vec2 = p - np.array([-R1DMMA, 0, 0])
        t2 = np.linalg.norm(vec2)
        v2 = np.array([vec2[0], vec2[2]]) / np.linalg.norm([vec2[0], vec2[2]])
        mid = (v2 + vec_output_projxz) / 2
        mid /= np.linalg.norm(mid)
        return t + t2, p, np.arcsin(mid[1])

    t_solution = brentq(lambda t: hit_point(t)[0] - Lrt / 2, 0, Lrt)
    _, p, angle_solution = hit_point(t_solution)
    R1delta = 2 * R1w0
    R1Wm0 = R1NMLA * DMLA + 2 * R1delta
    R1Hm0 = R1MMLA * DMLA - 2 * R1delta
    R2Wm0 = R1NMLA * DMLA - 2 * R1delta
    R1mp1 = ns.SquareMirror([p[0], 0, p[2]], width=R1Wm0, height=0.2, reflectivity=R1ultraR).RotY(angle_solution)
    R1mp2 = ns.SquareMirror([p[0], 0, -p[2]], width=R1Wm0, height=0.2, reflectivity=R1R, transmission=1).RotY(-angle_solution)
    R1mp2_origin_xz = np.array([p[0], -p[2]])
    v = R1mp2_origin_xz - np.array([-R1DMMA, 0])
    ripa2_rotate_angle = np.arctan(v[1] / v[0])
    v /= np.linalg.norm(v)
    ripa1_output_xz = R1mp2_origin_xz + v * np.linalg.norm(np.array([0, -R1ZRay]) - R1mp2_origin_xz)
    refpoint = ns.PointObj([ripa1_output_xz[0], -DMLA / 2, ripa1_output_xz[1]])
    midpoint = (refpoint.origin + R1mp2.origin) / 2
    R1BMMAshift = -(DMLA / 2) * R1MMLA / (R1MMLA + 1)
    R1m0 = ns.MMA(origin=[-R1DMMA, 0, 0], N=(R1NMLA, 1), pitch=DMLA, roc=R1MLAroc, n=1.5, thickness=R1DMMA,
                  reflectivity=R1ultraR, transmission=0, mma_width=R1Wm0, mma_height=R1Hm0, mma_shifty=R1BMMAshift,
                  back_transmission=0, back_reflectivity=1)
    R1mma = ns.MMA(origin=[R1d, 0, 0], N=(R1NMLA, R1MMLA), pitch=DMLA, roc=R1MLAroc, n=1.5, thickness=0.1,
                   reflectivity=R1ultraR, transmission=0.0, render_comp_vec=False, name="R1MMA",
                   shifty_z=-R1MMAshify).TY(DMLA / 2 - R1MMAshify / 2)
    mons1 = [ns.Monitor([R1d - 1e-4, 0, 0], width=R1W / 2 * 3, height=R1H / 2 * 3),
             ns.Monitor([-R1DMMA - 1e-4, 0, 0], width=R1Wm0 * 2, height=R1Hm0 * 2)]
    ripa1 = ns.ComponentGroup([0, 0, 0])
    ripa1.add_components([R1m0, R1mp1, R1mp2, R1mma])
    ripa1.add_monitors(mons1)
    ripa1.add_refpoint(refpoint)
    R12blk0 = ns.Block(midpoint, width=R2Wm0, height=R1W).TY(-4 * R1delta)
    R2mma = ns.MMA(origin=[R1d, 0, 0], N=(R1NMLA, R1NMLA), pitch=DMLA, roc=R1MLAroc, n=1.5, thickness=0.1,
                   reflectivity=R1ultraR, transmission=0.0, render_comp_vec=False, name="R2MMA", shifty_z=0).TZ(-R1W / 2)
    R2m0 = ns.TriangularPrism(origin=[0, 0, 0], width=R1Wm0, height=R1Wm0 * 2, n1=1, n2=1.55, alpha=np.pi / 4,
                              beta=np.pi / 2, reflectivity_1=1, transmission_1=0.03, reflectivity_2=1, transmission_2=0,
                              reflectivity_3=0, transmission_3=1, max_interact_count_2=1e5,
                              max_interact_count_3=1e5).RotX(np.pi / 2).TZ(-R1Wm0 - R1delta)
    R2Mon0 = ns.Monitor([R1d - 1e-4, 0, 0], width=R1W * 3, height=R1H * 3).TZ(-R1W / 2)
    ripa2 = ns.ComponentGroup([0, 0, 0])
    ripa2.add_components([R2mma, R2m0])
    ripa2.add_monitors([R2Mon0])
    ripa2.RotY(np.pi - ripa2_rotate_angle - R1theta0)
    ripa2._Translate(refpoint.origin)
    rng = np.random.default_rng(SEED + 6)
    rays = []
    for k in range(n_rays):
        o = np.array([0, R1W / 2, -R1ZRay])
        d = vec_input.copy()
        if k and jitter:
            o = o + np.array([0, *rng.uniform(-R1w0, R1w0, 2)])
            d = d + np.array([0, *rng.uniform(-1e-3, 1e-3, 2)])
        rays.append(ns.Ray(o, d, wavelength=wl, w0=R1w0))
    sc = Scene([ripa1, ripa2, R12blk0], rays, mons1 + [R2Mon0], limit={"max_trace_num": limit})
    sc.params = dict(R1w0=R1w0, origin=np.array([0, R1W / 2, -R1ZRay]), direction=vec_input, wavelength=wl)
    return sc




def doublet_pair(ns):
    """C3: two Edmund #88-597 doublets (examples/calibrate_4f.py:126-147: NBK7/NSF5, R = 18.405/-13.734/-39.933,
    CT 1.359/0.6, diameter 7.5) 60 apart + one monitor (SURVEY 8(d))."""
    mk = lambda x: ns.Doublet([x, 0, 0], CT1=1.359, CT2=0.6, R1=18.405, R2=-13.734, R3=-39.933,
                              n12=ns.Glass_NBK7(), n23=ns.Glass_NSF5(), diameter=7.5)
    return Scene([mk(30.3964), mk(90.3964)], [], [ns.Monitor([150, 0, 0], 10, 10)])


# ---- synthetic bundles (SURVEY 8(d)) -----------------------------------------------------------------------------
def _c2_rays(n, start):
    from .bundle import RayBundle

    return RayBundle.collimated_disc(n, start=start, x0=-10.0, radius=3.0, wavelength=780e-7, w0=61e-4)


def _c3_rays(n, start):
    from .bundle import RayBundle

    b = RayBundle.collimated_disc(n, start=start, x0=0.0, radius=3.0, wavelength=780e-7, w0=61e-4)
    wl = np.linspace(400e-7, 1100e-7, 16)[(np.arange(start, start + n) % 16)]
    b.columns["wavelength"] = wl
    b.columns["q_im"] = np.pi * 61e-4 ** 2 / wl
    return b


def _c4_rays(n, start):
    from .bundle import RayBundle, uniform01

    idx = np.arange(start, start + n, dtype=np.uint64)
    u = [uniform01(idx, k) for k in range(4)]
    d = np.stack([np.ones(n), (2 * u[2] - 1) * 2e-5, (2 * u[3] - 1) * 2e-5], 1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    b = RayBundle.collimated_disc(n, start=start, x0=2.0, wavelength=780e-7, w0=61e-4)
    b.columns.update(oy=2 * u[0] - 1, oz=2 * u[1] - 1, dx=d[:, 0].copy(), dy=d[:, 1].copy(), dz=d[:, 2].copy())
    return b


_RIPA_PARAMS = {}


def _c5_rays(n, start):
    import optable_b200 as ob

    from .bundle import RayBundle, uniform01

    if not _RIPA_PARAMS:
        _RIPA_PARAMS.update(ripa(ob, n_rays=0).params)
    p = _RIPA_PARAMS
    idx = np.arange(start, start + n, dtype=np.uint64)
    u = [uniform01(idx, k) for k in range(4)]
    o, d0, w0 = p["origin"], p["direction"], p["R1w0"]
    d = np.stack([np.full(n, d0[0]), d0[1] + (2 * u[2] - 1) * 1e-3, d0[2] + (2 * u[3] - 1) * 1e-3], 1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    b = RayBundle.collimated_disc(n, start=start, x0=o[0], wavelength=p["wavelength"], w0=w0)
    b.columns.update(oy=o[1] + (2 * u[0] - 1) * w0, oz=o[2] + (2 * u[1] - 1) * w0,
                     dx=d[:, 0].copy(), dy=d[:, 1].copy(), dz=d[:, 2].copy())
    return b


class Workload:
    """One benchmark configuration: scene builder, bundle maker(n, start), pop cap, rays per GPU per step, an upper
    bound on monitor rows per ray (result capacity) and the live-ray budget of the wavefront (splitting scenes)."""

    def __init__(self, name, config, scene, rays, max_trace_num, rays_per_gpu, rows_per_ray, max_live=0, cpu_rays=400_000):
        self.name, self.config, self._scene, self._rays = name, config, scene, rays
        self.max_trace_num, self.rays_per_gpu, self.rows_per_ray, self.max_live = max_trace_num, rays_per_gpu, rows_per_ray, max_live
        self.cpu_rays = cpu_rays

    def scene(self, ns=None):
        if ns is None:
            import optable_b200 as ns
        return self._scene(ns)

    def flat(self):
        from .flatten import FlatScene

        sc = self.scene()
        return FlatScene(sc.components, sc.monitors)

    def bundle(self, n, start=0):
        return self._rays(n, start)


WORKLOADS = {w.name: w for w in (
    Workload("c2_4f_telescope", "BASELINE configs[1]: calibrate_4f.py 4f telescope (two LENS-9 aspheres), 10M collimated rays, monitor spot capture",
             lambda ns: telescope_4f(ns, n_rays=0), _c2_rays, 2000, 10_000_000, 2),
    Workload("c3_doublets_16wl", "BASELINE configs[2]: Sellmeier-glass doublet stack (NBK7/NSF5), rays x 16 wavelengths",
             doublet_pair, _c3_rays, 2000, 10_000_000, 1),
    Workload("c4_cavity_4000", "BASELINE configs[3]: cavity_4mir.py four-mirror cavity, 1M Gaussian rays x 1000 round trips (4000 bounces)",
             lambda ns: cavity(ns, 0.0, 0.0), _c4_rays, 4001, 1_000_000, 0, cpu_rays=2_000),
    Workload("c5_ripa_64", "BASELINE configs[4]: ripa_gen2_lensless.py MMA-array scene (7,689 leaves), 64 pops per root; 12.5M rays per GPU = 100M rays on 8 GPUs",
             lambda ns: ripa(ns, n_rays=0), _c5_rays, 64, 12_500_000, 64, max_live=8, cpu_rays=100_000),
)}
DEFAULT = "c2_4f_telescope"
