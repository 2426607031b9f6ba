// optb_device.cuh -- device-side geometry and physics of the optable bounce loop (fp64, sm_100a).
//
// Semantics follow the reference decision by decision (tolerances, branch order, tie-breaks); the
// arithmetic is re-derived for the GPU (closed-form roots under the reference's own sign-scan,
// reciprocal-multiply normalisation, Horner polynomials) and agrees to ~1e-13 relative.
// Reference citations are relative to /root/reference/optable/.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include "../../include/optb.h"

// Everything is inlined, the once-per-pop physics and segment code included (measured on B200: 10 % faster than
// __noinline__ calls for those). Deciding the special operands of divisions (1/0, 0/x, x/inf) up front measured
// slower or equal on B200 (DESIGN.md §4), so the divisions below are plain.
#define OPTB_DEV __device__ __forceinline__

namespace optb {

// Device-side monitor record = the ABI record (OPTB_MON_STRIDE doubles) + per-monitor constants the upload derives from
// it: [24] nb / w, [25] w / nb, [26] nb / h, [27] h / nb (np.histogram's norm and step for the y and z binning).
constexpr int kMonBlobStride = OPTB_MON_STRIDE + 4;

struct Ray {
  double ox, oy, oz, dx, dy, dz;
  double I, wl, qre, qim, pl, n, len;
  uint32_t flags, root, pop;
  int32_t family;
};

// Pointers into the staged scene tables (shared memory when they fit, else global/L2).
struct SceneView {
  const double* trav;  // 64 B per node: lab AABB (6 doubles) + {geometry kind, skip} + {box-test flag, pad}: all the
                       // pre-order walk reads; the 368-B node rows are only touched for leaves that get tested
  const double* nf;
  const int32_t* ni;
  const int32_t* matk;
  const double* matf;
  const double* mon;
  const double* aux;
  int n_nodes, n_mons;
  unsigned long long* status;  // OPTB_C_STATUS word of the call (device memory)
};

OPTB_DEV double dot3(double ax, double ay, double az, double bx, double by, double bz) {
  return fma(ax, bx, fma(ay, by, az * bz));
}

// ray_to_local_coordinates optical_component.py:106-111 (+ direction setter ray.py:115-119)
OPTB_DEV void to_local(const double* __restrict__ c, const double* __restrict__ Ti, const Ray& r, bool ortho,
                       double& ox, double& oy, double& oz, double& dx, double& dy, double& dz) {
  double vx = r.ox - c[0], vy = r.oy - c[1], vz = r.oz - c[2];
  ox = dot3(Ti[0], Ti[1], Ti[2], vx, vy, vz);
  oy = dot3(Ti[3], Ti[4], Ti[5], vx, vy, vz);
  oz = dot3(Ti[6], Ti[7], Ti[8], vx, vy, vz);
  dx = dot3(Ti[0], Ti[1], Ti[2], r.dx, r.dy, r.dz);
  dy = dot3(Ti[3], Ti[4], Ti[5], r.dx, r.dy, r.dz);
  dz = dot3(Ti[6], Ti[7], Ti[8], r.dx, r.dy, r.dz);
  if (!ortho) {  // an orthonormal frame keeps |d| = 1 to rounding: the reference's re-normalisation is a no-op
    double rn = rsqrt(dot3(dx, dy, dz, dx, dy, dz));
    dx *= rn; dy *= rn; dz *= rn;
  }
}

// solve_ray_bboxes_intersections solver.py:5-48, one box
OPTB_DEV bool slab(double ox, double oy, double oz, double dx, double dy, double dz,
                   const double* __restrict__ bb, double& t1o, double& t2o) {
  double t1 = 0.0, t2 = INFINITY;
  const double o[3] = {ox, oy, oz}, d[3] = {dx, dy, dz};
#pragma unroll
  for (int ax = 0; ax < 3; ax++) {
    double bmin = bb[2 * ax], bmax = bb[2 * ax + 1];
    if (fabs(d[ax]) <= 1e-8) {  // np.isclose(d, 0.0)
      if (o[ax] < bmin || o[ax] > bmax) { t1 = 1.0; t2 = 0.0; }
    } else {
      const double inv = 1.0 / d[ax];
      const bool fwd = d[ax] > 0.0;  // min(ta, tb) / max(ta, tb) picked by the sign of d (bmin <= bmax)
      const double tn = ((fwd ? bmin : bmax) - o[ax]) * inv, tf = ((fwd ? bmax : bmin) - o[ax]) * inv;
      t1 = tn > t1 ? tn : t1;
      t2 = tf < t2 ? tf : t2;
    }
  }
  t1o = t1; t2o = t2;
  return (t2 + 1e-12 >= t1) && (t2 >= 0.0);
}

OPTB_DEV double dmax(double a, double b) { return a > b ? a : b; }  // no NaN canonicalisation needed here
OPTB_DEV double dmin(double a, double b) { return a < b ? a : b; }

// Per-pop constants of the lab-frame box tests: one ray meets many boxes (groups + their children), so
// everything that depends on the ray only is hoisted out of the node loop (solver.py:24-41).
struct BoxRay {
  double o[3], inv[3];           // origin, 1/d
  int near[3];                   // which box face (0 = min, 1 = max) is entered first on each axis
  bool par[3], any_par;          // axes that are "parallel" by np.isclose(d, 0); any -> take the general path
  OPTB_DEV BoxRay(double ox, double oy, double oz, double dx, double dy, double dz) {
    o[0] = ox; o[1] = oy; o[2] = oz;
    const double d[3] = {dx, dy, dz};
    any_par = false;
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
      par[ax] = fabs(d[ax]) <= 1e-8;
      any_par |= par[ax];
      inv[ax] = 1.0 / d[ax];
      near[ax] = inv[ax] < 0.0 ? 1 : 0;
    }
  }
};

// slab_hit plus front-to-back dismissal: 0 = the reference's test fails; 1 = it passes; 2 = it passes, but the ray
// point at `t_best` (the closest hit found so far) lies in front of the box's near face on some axis by more than a
// margin, so nothing inside the box can win. Callers only use 2 on boxes the upload marked cullable (optb.cu
// cull_bits: the box contains everything hittable below it to 1e-9 relative; curved leaves report roots up to 1e-9
// outside their bracket). The margin is a DISTANCE along the axis (1e-8 max(1, |face|)), not a ray parameter, so a ray
// almost parallel to the face is never dismissed on that axis. Rays that take the parallel-axis branch get 0 / 1.
OPTB_DEV int slab_hit_far(const BoxRay& r, const double* __restrict__ bb, double t_best);

// hit flag of solve_ray_bboxes_intersections for one lab box. With no parallel axis:
// t_near/t_far per axis are picked by the sign of d instead of min/max of the two plane parameters (identical for
// a well-formed box, bmin <= bmax).
OPTB_DEV bool slab_hit(const BoxRay& r, const double* __restrict__ bb) {
  if (!r.any_par) {
    double tn[3], tf[3];
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
      tn[ax] = (bb[2 * ax + r.near[ax]] - r.o[ax]) * r.inv[ax];
      tf[ax] = (bb[2 * ax + 1 - r.near[ax]] - r.o[ax]) * r.inv[ax];
    }
    // t2 + 1e-12 >= max(0, tn0, tn1, tn2) and t2 >= 0, without forming the maximum: one compare per candidate
    // (a double max is a compare plus two selects); the comparison against 0 is implied by t2 >= 0.
    const double t2 = dmin(dmin(tf[0], tf[1]), tf[2]);
    const double e = t2 + 1e-12;
    return (t2 >= 0.0) && (e >= tn[0]) && (e >= tn[1]) && (e >= tn[2]);
  }
  double t1 = 0.0, t2 = INFINITY;
#pragma unroll
  for (int ax = 0; ax < 3; ax++) {
    double bmin = bb[2 * ax], bmax = bb[2 * ax + 1];
    if (r.par[ax]) {
      if (r.o[ax] < bmin || r.o[ax] > bmax) { t1 = 1.0; t2 = 0.0; }
    } else {
      double ta = (bmin - r.o[ax]) * r.inv[ax], tb = (bmax - r.o[ax]) * r.inv[ax];
      t1 = dmax(t1, dmin(ta, tb));
      t2 = dmin(t2, dmax(ta, tb));
    }
  }
  return (t2 + 1e-12 >= t1) && (t2 >= 0.0);
}

OPTB_DEV int slab_hit_far(const BoxRay& r, const double* __restrict__ bb, double t_best) {
  if (r.any_par) return slab_hit(r, bb) ? 1 : 0;
  double tn[3], tf[3], face[3];
#pragma unroll
  for (int ax = 0; ax < 3; ax++) {
    face[ax] = bb[2 * ax + r.near[ax]];
    tn[ax] = (face[ax] - r.o[ax]) * r.inv[ax];
    tf[ax] = (bb[2 * ax + 1 - r.near[ax]] - r.o[ax]) * r.inv[ax];
  }
  const double t2 = dmin(dmin(tf[0], tf[1]), tf[2]);
  const double e = t2 + 1e-12;
  if (!((t2 >= 0.0) && (e >= tn[0]) && (e >= tn[1]) && (e >= tn[2]))) return 0;
  if (!(t_best < INFINITY)) return 1;  // nothing found yet: nothing to be beyond
  bool far = false;
#pragma unroll
  for (int ax = 0; ax < 3; ax++)  // (tn - t_best) |d_ax| = distance from the best hit's point to the near face, along ax
    far |= (tn[ax] - t_best) > 1e-8 * fmax(1.0, fabs(face[ax])) * fabs(r.inv[ax]);
  return far ? 2 : 1;
}

// The dismissal half of slab_hit_far alone, for a box already known to pass the reference's test and a finite t_best
// (no parallel axis).
OPTB_DEV bool slab_far_only(const BoxRay& r, const double* __restrict__ bb, double t_best) {
  bool far = false;
#pragma unroll
  for (int ax = 0; ax < 3; ax++) {
    const double face = bb[2 * ax + r.near[ax]];
    const double tn = (face - r.o[ax]) * r.inv[ax];
    far |= (tn - t_best) > 1e-8 * fmax(1.0, fabs(face)) * fabs(r.inv[ax]);
  }
  return far;
}

// ---- ASphere profile (component_group.py:1065-1107) ----
// The reference differentiates this profile numerically (h = 1e-4 radius, surfaces.py:351-369); the second
// difference amplifies every rounding of f by ~1e8, so the operation order of the Python closure is kept
// exactly and FMA contraction is ruled out with the _rn intrinsics.
OPTB_DEV double f_asphere(int form, const double* __restrict__ c, double r) {
  double r2 = __dmul_rn(r, r);
  if (form == OPTB_ASPH_PARAMETRIC) {
    // r**2 / (R * (1 + sqrt(1 - (1 + kappa) * (r**2) / (R**2)))) + a4 r**4 + a6 r**6 + a8 r**8
    double R = c[0];
    double u = __ddiv_rn(__dmul_rn(__dadd_rn(1.0, c[1]), r2), __dmul_rn(R, R));
    double s = __dsqrt_rn(__dsub_rn(1.0, u));
    double acc = __ddiv_rn(r2, __dmul_rn(R, __dadd_rn(1.0, s)));
    double r4 = __dmul_rn(r2, r2);
    acc = __dadd_rn(acc, __dmul_rn(c[2], r4));
    acc = __dadd_rn(acc, __dmul_rn(c[3], __dmul_rn(r4, r2)));
    acc = __dadd_rn(acc, __dmul_rn(c[4], __dmul_rn(r4, r4)));
    return acc;
  }
  // (EFL / (n + 1)) * (-1 + sqrt(1 + (n + 1) / (n - 1) * (r**2) / (EFL**2)))
  double EFL = c[0], n = c[1];
  double u = __ddiv_rn(__dmul_rn(__ddiv_rn(__dadd_rn(n, 1.0), __dsub_rn(n, 1.0)), r2), __dmul_rn(EFL, EFL));
  return __dmul_rn(__ddiv_rn(EFL, __dadd_rn(n, 1.0)), __dadd_rn(-1.0, __dsqrt_rn(__dadd_rn(1.0, u))));
}

// ---- Polygon.within_boundary surfaces.py:534-558 ----
OPTB_DEV bool poly_within(const double* __restrict__ rec, double Px, double Py, double Pz) {
  const double tol = 1e-9;
  int nv = (int)rec[0];
  const double* v = rec + OPTB_POLY_HEADER;
  double ex = Px - rec[4], ey = Py - rec[5], ez = Pz - rec[6];
  double px = dot3(ex, ey, ez, rec[7], rec[8], rec[9]);
  double py = dot3(ex, ey, ez, rec[10], rec[11], rec[12]);
  bool inside = false;
  for (int i = 0; i < nv; i++) {
    int j = (i + 1 == nv) ? 0 : i + 1;
    double x1 = v[2 * i], y1 = v[2 * i + 1], x2 = v[2 * j], y2 = v[2 * j + 1];
    double cr = (x2 - x1) * (py - y1) - (y2 - y1) * (px - x1);
    if (fabs(cr) <= tol && fmin(x1, x2) - tol <= px && px <= fmax(x1, x2) + tol &&
        fmin(y1, y2) - tol <= py && py <= fmax(y1, y2) + tol)
      return true;
    if ((y1 > py) != (y2 > py)) {
      double x_at_y = x1 + (py - y1) * (x2 - x1) / (y2 - y1);
      if (x_at_y >= px) inside = !inside;
    }
  }
  return inside;
}

OPTB_DEV bool planar_within(const SceneView& sv, int kind, double p0, double p1, double Px, double Py, double Pz) {
  if (kind == OPTB_G_CIRCLE) return dot3(Px, Py, Pz, Px, Py, Pz) <= p0 * p0 && p0 >= 0.0;  // |P| <= r (3-D norm, surfaces.py:144-145), on squares
  if (kind == OPTB_G_RECT) return fabs(Py) <= p0 && fabs(Pz) <= p1;            // surfaces.py:170-171
  if (kind == OPTB_G_POLY2D) return poly_within(sv.aux + (long long)p0, Px, Py, Pz);
  return false;
}

// Plane.union / Plane.subtract (surfaces.py:100-136) at a local point: the flat two-operand record, or (p0 = 2) the
// postfix program of a nested composite; the value stack is a bit stack (depth checked by the upload).
OPTB_DEV bool csg_within(const SceneView& sv, const int32_t* __restrict__ ni, const double* __restrict__ p,
                         double Px, double Py, double Pz) {
  const int op = (int)p[0];
  if (op != 2) {
    const bool a = planar_within(sv, (int)p[1], p[2], p[3], Px, Py, Pz);
    const bool b = planar_within(sv, (int)p[4], p[5], p[6], Px, Py, Pz);
    return op == 0 ? (a && !b) : (a || b);
  }
  const double* prog = sv.aux + ni[OPTB_NI_AUX];
  const int n = (int)prog[0];
  unsigned st = 0u;
  for (int k = 0; k < n; k++) {
    const int code = (int)prog[1 + 3 * k];
    if (code > 0) {
      st = (st << 1) | (planar_within(sv, code, prog[2 + 3 * k], prog[3 + 3 * k], Px, Py, Pz) ? 1u : 0u);
    } else {
      const bool b = st & 1u, a = (st >> 1) & 1u;
      st = ((st >> 2) << 1) | ((code == OPTB_CSG_SUBTRACT ? (a && !b) : (a || b)) ? 1u : 0u);
    }
  }
  return st & 1u;
}

// surface within_boundary for curved kinds (surfaces.py:230-235, 300-303, 390-393)
OPTB_DEV bool curved_within(const SceneView& sv, int g, const int32_t* __restrict__ ni, const double* __restrict__ p,
                            double Px, double Py, double Pz) {
  if (g == OPTB_G_SPHERE) return (p[0] - p[1] - 1e-12 <= Px) && (Px <= p[0] + 1e-12);
  if (g == OPTB_G_ASPHERE) return sqrt(Py * Py + Pz * Pz) <= p[0] + 1e-12;
  if (g == OPTB_G_CYL) {
    double th = atan2(Py, Px);
    return (p[2] <= th && th <= p[3]) && (-p[1] / 2 <= Pz && Pz <= p[1] / 2);
  }
  return poly_within(sv.aux + ni[OPTB_NI_AUX], Px, Py, Pz);  // POLY3D
}

// ASphere.f along a local ray, for the sign scan and the root solve (surfaces.py:375-378), in a division-free
// form with the same zeros and the same sign: with s = sqrt(1 - k1 r^2),
//   f = Px + r^2 / (R (1 + s)) + poly(r^2)   <=>   g = sign(R) * ((Px + poly) * R * (1 + s) + r^2) = f * |R| (1 + s)
// and |R| (1 + s) > 0. The sag only depends on r^2, so no square root is needed for r either. Constants are
// folded once per intersection. (The bit-exact form f_asphere() above is reserved for the finite-difference
// normal / curvature, where the reference's own rounding matters.)
struct AsphF {
  int form;
  double k1, R, sgn, a4, a6, a8;  // parametric: k1 = (1+kappa)/R^2 ; exact: k1 = (n+1)/((n-1) EFL^2), R = EFL/(n+1)
  double ox, oy, oz, dx, dy, dz;
  OPTB_DEV AsphF(int form_, const double* __restrict__ c, double k1_, double ox_, double oy_, double oz_, double dx_, double dy_, double dz_)
      : form(form_), ox(ox_), oy(oy_), oz(oz_), dx(dx_), dy(dy_), dz(dz_) {
    k1 = k1_;  // precomputed by the upload with the expressions below (one division less per asphere test)
    if (form == OPTB_ASPH_PARAMETRIC) {
      R = c[0]; /* k1 = (1.0 + c[1]) / (R * R) */ a4 = c[2]; a6 = c[3]; a8 = c[4];
      sgn = R < 0 ? -1.0 : 1.0;
    } else {
      /* k1 = (c[1] + 1.0) / ((c[1] - 1.0) * c[0] * c[0]) */ R = c[0] / (c[1] + 1.0); a4 = a6 = a8 = 0.0; sgn = 1.0;
    }
  }
  OPTB_DEV double operator()(double t) const {
    double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
    double r2 = fma(Py, Py, Pz * Pz);
    if (form == OPTB_ASPH_PARAMETRIC) {
      double s = sqrt(fma(-k1, r2, 1.0));
      double lin = fma(r2 * r2, fma(r2, fma(r2, a8, a6), a4), Px);  // Px + a4 r^4 + a6 r^6 + a8 r^8
      return sgn * fma(lin * R, 1.0 + s, r2);
    }
    return fma(R, sqrt(fma(k1, r2, 1.0)) - 1.0, Px);
  }
  // Surface.f itself (surfaces.py:375-378), not rescaled: what scipy's brentq sees in the reference (its secant /
  // inverse-quadratic steps depend on the values of f, not only on its zeros)
  OPTB_DEV double truef(double t) const {
    double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
    double r2 = fma(Py, Py, Pz * Pz);
    if (form == OPTB_ASPH_PARAMETRIC) {
      double s = sqrt(fma(-k1, r2, 1.0));
      return Px + r2 / (R * (1.0 + s)) + r2 * r2 * fma(r2, fma(r2, a8, a6), a4);
    }
    return fma(R, sqrt(fma(k1, r2, 1.0)) - 1.0, Px);
  }
  // g and dg/dt at t (for the Newton refinement of a bracketed root)
  OPTB_DEV void eval2(double t, double& g, double& dg) const {
    double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
    double r2 = fma(Py, Py, Pz * Pz);
    double r2p = 2.0 * fma(Py, dy, Pz * dz);
    if (form == OPTB_ASPH_PARAMETRIC) {
      double s = sqrt(fma(-k1, r2, 1.0));
      double lin = fma(r2 * r2, fma(r2, fma(r2, a8, a6), a4), Px);
      double linp = fma(r2 * fma(r2, fma(r2, 4.0 * a8, 3.0 * a6), 2.0 * a4), r2p, dx);
      double sp = -0.5 * k1 * r2p / s;
      g = sgn * fma(lin * R, 1.0 + s, r2);
      dg = sgn * (fma(linp * R, 1.0 + s, lin * R * sp) + r2p);
    } else {
      double h = sqrt(fma(k1, r2, 1.0));
      g = fma(R, h - 1.0, Px);
      dg = fma(0.5 * R * k1 / h, r2p, dx);
    }
  }
  // Same sign as operator()(t) (NaN where the reference's f is NaN), without the square root:
  // g = sgn * (A s + B) with s = sqrt(s2) >= 0; when A and B disagree in sign the comparison is done on squares.
  OPTB_DEV double sign(double t) const {
    double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
    double r2 = fma(Py, Py, Pz * Pz);
    double A, B, s2;
    if (form == OPTB_ASPH_PARAMETRIC) {
      s2 = fma(-k1, r2, 1.0);
      A = fma(r2 * r2, fma(r2, fma(r2, a8, a6), a4), Px) * R;
      B = r2 + A;
    } else {
      s2 = fma(k1, r2, 1.0);
      A = R; B = Px - R;
    }
    double v;
    if ((A >= 0.0) == (B >= 0.0)) v = A + B;
    else { double d = fma(A * A, s2, -B * B); v = (A >= 0.0) ? d : -d; }
    if (!(s2 >= 0.0)) v = NAN;
    return sgn * v;
  }
  // The same decision for the ten scan samples, with the profile form a compile-time constant (with a run-time `form` the
  // compiler evaluates both forms at every sample and selects), the NaN case (s2 < 0: the reference's f is NaN, neither
  // positive nor negative) folded into the comparisons, and the sign of R applied to the two masks afterwards instead
  // of to every value. Bit i of pos / neg: sign(ts_i) > 0 / < 0 -- the masks sign() would give. c2: 5.850 -> 5.804 ms.
  template <int FORM>
  OPTB_DEV void scan10(double a, double b, double step, unsigned& pos_out, unsigned& neg_out) const {
    unsigned pos = 0u, neg = 0u;
#pragma unroll
    for (int i = 0; i < 10; i++) {
      const double t = i == 9 ? b : fma((double)i, step, a);  // np.linspace(a, b, 10)[i], as sample_t
      const double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
      const double r2 = fma(Py, Py, Pz * Pz);
      double A, B, s2;
      if (FORM == OPTB_ASPH_PARAMETRIC) {
        s2 = fma(-k1, r2, 1.0);
        A = fma(r2 * r2, fma(r2, fma(r2, a8, a6), a4), Px) * R;
        B = r2 + A;
      } else {
        s2 = fma(k1, r2, 1.0);
        A = R; B = Px - R;
      }
      double v;
      if ((A >= 0.0) == (B >= 0.0)) v = A + B;
      else { double d = fma(A * A, s2, -B * B); v = (A >= 0.0) ? d : -d; }
      const bool ok = s2 >= 0.0;
      pos |= ((ok && v > 0.0) ? 1u : 0u) << i;
      neg |= ((ok && v < 0.0) ? 1u : 0u) << i;
    }
    const bool flip = sgn < 0.0;
    pos_out = flip ? neg : pos;
    neg_out = flip ? pos : neg;
  }
};

// Root of a smooth f inside a bracket with f(lo) f(hi) < 0: safeguarded Newton from the secant point (a step that
// would leave the bracket is replaced by a bisection). The reference gets this root from scipy's brentq, whose
// answer is only defined to xtol = 2e-12; converging to the last bit instead stays well inside that.
template <class F>
OPTB_DEV double newton_bracketed(const F& f, double lo, double hi, double glo, double ghi) {
  if (glo == 0.0) return lo;
  if (ghi == 0.0) return hi;
  double x = lo - glo * (hi - lo) / (ghi - glo);
  const bool lo_pos = glo > 0.0;
  for (int it = 0; it < 12; it++) {
    double g, dg;
    f.eval2(x, g, dg);
    if (g == 0.0) break;
    if ((g > 0.0) == lo_pos) lo = x; else hi = x;
    double xn = x - g / dg;
    if (fabs(xn - x) <= 2e-15 * fmax(fabs(x), 1.0)) { x = xn; break; }  // converged to rounding level
    if (!(xn > fmin(lo, hi) && xn < fmax(lo, hi))) xn = 0.5 * (lo + hi);
    x = xn;
  }
  return x;
}

// scipy.optimize.brentq (scipy/optimize/Zeros/brentq.c; xtol = 2e-12, rtol = 4 eps, maxiter = 100: the defaults the
// reference calls it with, optical_component.py:132) restated for the device. The reference's hit distance on a curved
// surface IS this iteration's last iterate, up to 2e-12 away from the true root; with `reference_roots` the device
// runs the same iteration on the same bracket and lands on the same iterate (to the rounding of f), instead of on the
// root itself. f(xa) f(xb) < 0 is guaranteed by the caller (the sign scan).
template <class F>
OPTB_DEV double brentq_dev(const F& f, double xa, double xb) {
  const double xtol = 2e-12, rtol = 8.881784197001252e-16;
  double xpre = xa, xcur = xb, xblk = 0.0, fblk = 0.0, spre = 0.0, scur = 0.0;
  double fpre = f(xpre), fcur = f(xcur);
  if (fpre == 0.0) return xpre;
  if (fcur == 0.0) return xcur;
  for (int it = 0; it < 100; it++) {
    if (fpre != 0.0 && fcur != 0.0 && (signbit(fpre) != signbit(fcur))) {
      xblk = xpre; fblk = fpre;
      spre = scur = xcur - xpre;
    }
    if (fabs(fblk) < fabs(fcur)) {
      xpre = xcur; xcur = xblk; xblk = xpre;
      fpre = fcur; fcur = fblk; fblk = fpre;
    }
    const double delta = (xtol + rtol * fabs(xcur)) / 2;
    const double sbis = (xblk - xcur) / 2;
    if (fcur == 0.0 || fabs(sbis) < delta) return xcur;
    if (fabs(spre) > delta && fabs(fcur) < fabs(fpre)) {
      double stry;
      if (xpre == xblk) {
        stry = -fcur * (xcur - xpre) / (fcur - fpre);                       // secant
      } else {
        const double dpre = (fpre - fcur) / (xpre - xcur), dblk = (fblk - fcur) / (xblk - xcur);
        stry = -fcur * (fblk * dblk - fpre * dpre) / (dblk * dpre * (fblk - fpre));  // inverse quadratic
      }
      if (2 * fabs(stry) < fmin(fabs(spre), 3 * fabs(sbis) - delta)) { spre = scur; scur = stry; }
      else { spre = sbis; scur = sbis; }
    } else {
      spre = sbis; scur = sbis;
    }
    xpre = xcur; fpre = fcur;
    if (fabs(scur) > delta) xcur += scur;
    else xcur += (sbis > 0 ? delta : -delta);
    fcur = f(xcur);
  }
  return xcur;
}

// Surface.f along a local ray for the quadric kinds (surfaces.py:224-225, 294-295), as brentq_dev's functor
struct QuadF {
  int cyl; double R, ox, oy, oz, dx, dy, dz;
  OPTB_DEV double operator()(double t) const {
    const double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
    return sqrt(cyl ? fma(Px, Px, Py * Py) : dot3(Px, Py, Pz, Px, Py, Pz)) - R;
  }
};
template <class F>
struct TrueF {  // adapts AsphF::truef to operator()
  const F& f;
  OPTB_DEV double operator()(double t) const { return f.truef(t); }
};

// np.linspace(a, b, 10)[i]
OPTB_DEV double sample_t(int i, double a, double b, double step) {
  // (double)i from a constant table: avoids an I2F.F64 per sample
  const double fi = (double)i;
  return i == 9 ? b : fma(fi, step, a);
}

// (one shift and one AND instead of four compares: it runs once or twice per leaf test)
// (measured: c3 6.64 -> 6.58 ms, c4 110.7 -> 109.8 ms)
OPTB_DEV bool is_planar_kind(int g) {
  constexpr unsigned kPlanar = (1u << OPTB_G_CIRCLE) | (1u << OPTB_G_RECT) | (1u << OPTB_G_POLY2D) | (1u << OPTB_G_CSG);
  return (kPlanar >> g) & 1u;
}

// Planar leaves, straight from the lab ray (ray_to_local_coordinates :106-111 + intersect_point_local :165-196 in
// one, evaluated in stages): the plane is local x = 0, so the x row of Tinv alone decides whether the ray can reach
// it at all (t = -ox/dx >= 1e-9 needs ox, dx of opposite signs; the sign of dx does not change under the
// re-normalisation of the direction), and for an orthonormal frame it also gives t itself. The y and z rows are
// only paid for by rays that get as far as the aperture test. Returns t or -1.
OPTB_DEV double intersect_planar(const SceneView& sv, const int32_t* __restrict__ ni, const double* __restrict__ nf,
                                 const Ray& r, double t_beat) {
  const double* c = nf + OPTB_NF_ORIGIN;
  const double* Ti = nf + OPTB_NF_TINV;
  const double vx = r.ox - c[0], vy = r.oy - c[1], vz = r.oz - c[2];
  const double ox = dot3(Ti[0], Ti[1], Ti[2], vx, vy, vz);
  double dx = dot3(Ti[0], Ti[1], Ti[2], r.dx, r.dy, r.dz);
  if (!((ox < 0.0 && dx > 0.0) || (ox > 0.0 && dx < 0.0))) return -1.0;
  double dy, dz;
  const bool ortho = ni[OPTB_NI_ORTHO] != 0;
  if (!ortho) {
    dy = dot3(Ti[3], Ti[4], Ti[5], r.dx, r.dy, r.dz);
    dz = dot3(Ti[6], Ti[7], Ti[8], r.dx, r.dy, r.dz);
    const double rn = rsqrt(dot3(dx, dy, dz, dx, dy, dz));
    dx *= rn; dy *= rn; dz *= rn;
  }
  const double t = -ox / dx;
  if (!(t >= 1e-9) || t > r.len || t > t_beat) return -1.0;  // |t|<EPS, t<0, t>length, NaN; or cannot win any more
  if (ortho) {
    dy = dot3(Ti[3], Ti[4], Ti[5], r.dx, r.dy, r.dz);
    dz = dot3(Ti[6], Ti[7], Ti[8], r.dx, r.dy, r.dz);
  }
  const double oy = dot3(Ti[3], Ti[4], Ti[5], vx, vy, vz);
  const double oz = dot3(Ti[6], Ti[7], Ti[8], vx, vy, vz);
  const double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
  const int g = ni[OPTB_NI_GEOM];
  const double* p = nf + OPTB_NF_P;
  bool in;
  if (g == OPTB_G_CSG) {
    in = csg_within(sv, ni, p, Px, Py, Pz);
  } else if (g == OPTB_G_POLY2D) {
    in = poly_within(sv.aux + ni[OPTB_NI_AUX], Px, Py, Pz);
  } else {
    in = planar_within(sv, g, p[0], p[1], Px, Py, Pz);
  }
  return in ? t : -1.0;
}

// intersect_point_local optical_component.py:197-233 (curved branch) for one leaf, local-frame ray. Returns t or -1.
template <bool ASPH, bool BRENT = false>
OPTB_DEV double intersect_leaf(const SceneView& sv, const int32_t* __restrict__ ni, const double* __restrict__ nf,
                               double ox, double oy, double oz, double dx, double dy, double dz, double len,
                               double t_beat = INFINITY) {
  // t_beat: a hit is only useful to the caller if t <= t_beat (the closest hit found so far). The curved branch
  // only ever reports roots inside its bracket [a, b], so a bracket that starts beyond t_beat is skipped whole.
  const int g = ni[OPTB_NI_GEOM];
  const double* p = nf + OPTB_NF_P;
  // (planar kinds never get here: intersect_planar)
  // curved branch :197-233. Local AABB (Surface.get_bbox_local) -> bracket -> 10-point sign scan -> roots.
  double bb[6];
  if (g == OPTB_G_SPHERE) {
#pragma unroll
    for (int i = 0; i < 6; i++) bb[i] = p[2 + i];
  } else if (ASPH && g == OPTB_G_ASPHERE) {
    bb[0] = p[6]; bb[1] = p[7]; bb[2] = -p[0]; bb[3] = p[0]; bb[4] = -p[0]; bb[5] = p[0];
  } else if (g == OPTB_G_CYL) {
    bb[0] = -p[0]; bb[1] = p[0]; bb[2] = -p[0]; bb[3] = p[0]; bb[4] = -p[1] / 2; bb[5] = p[1] / 2;
  } else {
    const double* rec = sv.aux + ni[OPTB_NI_AUX];
#pragma unroll
    for (int i = 0; i < 6; i++) bb[i] = rec[13 + i];
  }
  double t1, t2;
  slab(ox, oy, oz, dx, dy, dz, bb, t1, t2);
  if (t2 + 1e-9 < t1) return -1.0;
  t1 = fmax(t1, 0.0);
  t2 = fmin(t2, 100.0);
  const double a = t1 - 1e-9, b = t2 + 1e-9;
  if (b >= a && a > t_beat) return -1.0;
  const double step = (b - a) / 9.0;
  // roots found by the sign scan, ascending in t (sub-intervals are visited in order)
  if (ASPH && g == OPTB_G_ASPHERE) {
    // Scan first, solve after: the (expensive) root solve runs once for the whole warp instead of once per
    // sub-interval (lane efficiency 21 -> 31 of 32).
    const AsphF f(ni[OPTB_NI_AUX], p + 1, nf[OPTB_NF_FOCAL], ox, oy, oz, dx, dy, dz);  // (FOCAL slot of an asphere row: k1, set by the upload)
    const bool asc = (b >= a);
    // All ten sample signs first, as two bit masks: the evaluations are independent, so the fp64 pipe sees ten
    // interleaved dependency chains instead of one (and nothing but 20 bits stays live afterwards).
    unsigned pos = 0u, neg = 0u;
    if (f.form == OPTB_ASPH_PARAMETRIC) f.template scan10<OPTB_ASPH_PARAMETRIC>(a, b, step, pos, neg);
    else f.template scan10<OPTB_ASPH_EXACT_SPH>(a, b, step, pos, neg);
    unsigned chg = ((pos & (neg >> 1)) | (neg & (pos >> 1))) & 0x1ffu;  // bit i: f(ts_i) * f(ts_i+1) < 0
    double best = -1.0;
    while (chg) {
      const int i = __ffs(chg) - 1;
      chg &= chg - 1u;
      const double ta = sample_t(i, a, b, step), tb = sample_t(i + 1, a, b, step);
      const bool fa_pos = (pos >> i) & 1u;
      bool solve = true;
      double lo = ta;
      if (asc) {
        if ((BRENT ? tb < 1e-9 : tb <= 1e-9) || ta > len) solve = false;  // every root in here fails t >= EPS (or t <= length)
        else if (!BRENT && ta < 1e-9) {
          // The sub-interval straddles the admissibility threshold (the usual case right after leaving this
          // very surface: the root is the self-intersection at t ~ 0). One sample at t = EPS tells on which
          // side the root lies; below it the reference finds it with brentq and then filters it out.
          const double fe = f.sign(1e-9);
          if (fa_pos ? fe < 0.0 : fe > 0.0) solve = false;       // f(ta) * f(EPS) < 0
          else if (fa_pos ? fe > 0.0 : fe < 0.0) lo = 1e-9;      // f(EPS) * f(tb) < 0
        }
      }
      if (solve) {
        double r = BRENT ? brentq_dev(TrueF<AsphF>{f}, ta, tb) : newton_bracketed(f, lo, tb, f(lo), f(tb));
        if (r >= 1e-9 && r <= len) {
          double Py = fma(r, dy, oy), Pz = fma(r, dz, oz);
          const double rmax = p[0] + 1e-12;
          if (fma(Py, Py, Pz * Pz) <= rmax * rmax) {   // ASphere.within_boundary (r <= radius + 1e-12, on squares)
            if (asc) return r;   // sub-intervals ascend: the first admissible root is the smallest
            if (best < 0 || r < best) best = r;
          }
        }
      }
    }
    return best;
  }
  // Quadratic / linear surfaces: g(t) has the sign of Surface.f(o + t d); closed-form roots.
  double A, B, Cc;  // g(t) = A t^2 + 2 B t + C
  if (g == OPTB_G_SPHERE) {          // f = |P| - R            surfaces.py:294-295
    A = 1.0; B = dot3(ox, oy, oz, dx, dy, dz); Cc = dot3(ox, oy, oz, ox, oy, oz) - p[0] * p[0];
  } else if (g == OPTB_G_CYL) {      // f = |P_xy| - r         surfaces.py:224-225
    A = fma(dx, dx, dy * dy); B = fma(ox, dx, oy * dy); Cc = fma(ox, ox, oy * oy) - p[0] * p[0];
  } else {                           // 3-D polygon: f = n.(P - v0), linear       surfaces.py:530-532
    const double* rec = sv.aux + ni[OPTB_NI_AUX];
    A = 0.0;
    B = 0.5 * dot3(rec[1], rec[2], rec[3], dx, dy, dz);
    Cc = dot3(rec[1], rec[2], rec[3], ox - rec[4], oy - rec[5], oz - rec[6]);
  }
  double lo, hi;  // the two real roots (lo <= hi) or NaN
  if (A != 0.0) {
    double disc = fma(B, B, -A * Cc);
    if (!(disc >= 0.0)) return -1.0;  // g never changes sign
    double sq = sqrt(disc);
    double qv = -(B + copysign(sq, B));
    double ra = qv / A, rb = (qv != 0.0) ? Cc / qv : ra;
    lo = fmin(ra, rb); hi = fmax(ra, rb);
  } else {
    if (B == 0.0) return -1.0;
    lo = hi = -Cc / (2.0 * B);
  }
  // ten sample signs as bit masks (independent evaluations), then the sub-intervals with a sign change in order
  unsigned pos = 0u, neg = 0u;
#pragma unroll
  for (int i = 0; i < 10; i++) {
    const double ts = sample_t(i, a, b, step);
    const double gv = fma(fma(A, ts, 2.0 * B), ts, Cc);
    pos |= (gv > 0.0 ? 1u : 0u) << i;
    neg |= (gv < 0.0 ? 1u : 0u) << i;
  }
  unsigned chg = ((pos & (neg >> 1)) | (neg & (pos >> 1))) & 0x1ffu;  // bit i: g(ts_i) * g(ts_i+1) < 0
  const bool asc = (b >= a);
  double best = -1.0;
  while (chg) {
    const int i = __ffs(chg) - 1;
    chg &= chg - 1u;
    // exactly one root of g inside this sub-interval: entering (g: + -> -, seen along increasing t) is `lo`
    const bool ga_pos = (pos >> i) & 1u;
    double r = (A != 0.0) ? ((ga_pos == asc) ? lo : hi) : lo;
    if (BRENT && A != 0.0) {  // the reference's own iterate on this sub-interval instead of the closed-form root
      const QuadF qf{g == OPTB_G_CYL, p[0], ox, oy, oz, dx, dy, dz};
      r = brentq_dev(qf, sample_t(i, a, b, step), sample_t(i + 1, a, b, step));
    }
    if (r >= 1e-9 && r <= len) {
      double Px = fma(r, dx, ox), Py = fma(r, dy, oy), Pz = fma(r, dz, oz);
      if (curved_within(sv, g, ni, p, Px, Py, Pz)) {
        if (asc) return r;
        if (best < 0 || r < best) best = r;
      }
    }
  }
  return best;
}

// Surface.normal at a local hit point
template <bool ASPH>
OPTB_DEV void surf_normal(const SceneView& sv, const int32_t* __restrict__ ni, const double* __restrict__ nf,
                          double Px, double Py, double Pz, double& nx, double& ny, double& nz, double& roc_fd) {
  const int g = ni[OPTB_NI_GEOM];
  const double* p = nf + OPTB_NF_P;
  roc_fd = INFINITY;
  if (g == OPTB_G_SPHERE) { double ir = 1.0 / p[0]; nx = Px * ir; ny = Py * ir; nz = Pz * ir; return; }
  if (g == OPTB_G_CYL) { double ir = 1.0 / p[0]; nx = Px * ir; ny = Py * ir; nz = 0.0; return; }
  if (ASPH && g == OPTB_G_ASPHERE) {
    // central differences with h = 1e-4 * radius  surfaces.py:351-388
    double r = __dsqrt_rn(__dadd_rn(__dmul_rn(Py, Py), __dmul_rn(Pz, Pz)));
    double h = 1e-4 * p[0];
    int form = ni[OPTB_NI_AUX];
    double fp = f_asphere(form, p + 1, r + h), fm = f_asphere(form, p + 1, r - h);
    double d1 = (fp - fm) / (2 * h);
    if (ni[OPTB_NI_ROCKIND] == OPTB_ROC_ASPHERE_FD) {
      double f0 = f_asphere(form, p + 1, r);
      double d2 = (fp - 2 * f0 + fm) / (h * h);
      double w = 1.0 + d1 * d1;
      roc_fd = w * sqrt(w) / d2;  // (1 + f'^2)^1.5 / f''
    }
    if (r < 1e-12) { nx = 1.0; ny = 0.0; nz = 0.0; return; }
    double ir = 1.0 / r;
    double ax = 1.0, ay = d1 * (Py * ir), az = d1 * (Pz * ir);
    double rn = rsqrt(dot3(ax, ay, az, ax, ay, az));
    nx = ax * rn; ny = ay * rn; nz = az * rn;
    return;
  }
  if (g == OPTB_G_POLY2D || g == OPTB_G_POLY3D) {
    const double* rec = sv.aux + ni[OPTB_NI_AUX];
    nx = rec[1]; ny = rec[2]; nz = rec[3];
    return;
  }
  nx = 1.0; ny = 0.0; nz = 0.0;
}

// Material.n / SellmeierMaterial.sellmeier_n material.py:12-21, 106-120
OPTB_DEV double material_n(const SceneView& sv, int m, double wl_m) {
  const double* f = sv.matf + m * OPTB_MF_STRIDE;
  const int kind = sv.matk[m];
  if (kind == OPTB_MAT_CONST) return f[0];
  if (kind == OPTB_MAT_LUT) {
    // Material(n=<Python callable>): evaluated by the host once per distinct wavelength of the batch; (wavelength in
    // metres, n) pairs sorted by wavelength. wavelength * unit is the same IEEE product on both sides: exact match.
    const double* tab = sv.aux + (long long)f[0];
    int lo = 0, hi = (int)f[1] - 1;
    while (lo <= hi) {
      const int mid = (lo + hi) >> 1;
      const double w = tab[2 * mid];
      if (w == wl_m) return tab[2 * mid + 1];
      if (w < wl_m) lo = mid + 1; else hi = mid - 1;
    }
    atomicOr(sv.status, (unsigned long long)OPTB_ST_LUT_MISS);
    return NAN;
  }
  double wl_um = wl_m / 1e-6;
  double w2 = wl_um * wl_um;
  double n2 = 1.0;
#pragma unroll
  for (int i = 0; i < 3; i++) n2 += f[i] * w2 / (w2 - f[3 + i]);
  return sqrt(n2);
}

// Per-thread memo of Sellmeier evaluations: a ray keeps its wavelength for life and meets the same one or two glasses
// again and again (every face of a lens), so n(material, wavelength) is looked up in two slots kept in shared memory
// before paying three divisions and a square root. Slots are keyed by (wavelength, material index).
struct IndexCache {
  volatile double* wl; volatile double* n0; volatile double* n1; volatile int* m0; volatile int* m1;
};
OPTB_DEV double material_n_cached(const SceneView& sv, const IndexCache& c, int m, double wl_m) {
  if (sv.matk[m] == OPTB_MAT_CONST) return sv.matf[m * OPTB_MF_STRIDE];
  const bool same_wl = (*c.wl == wl_m);
  if (same_wl && *c.m0 == m) return *c.n0;
  if (same_wl && *c.m1 == m) return *c.n1;
  const double n = material_n(sv, m, wl_m);
  if (!same_wl) { *c.wl = wl_m; *c.m0 = m; *c.n0 = n; *c.m1 = -1; }
  else if (*c.m1 < 0 || (m & 1)) { *c.m1 = m; *c.n1 = n; }
  else { *c.m0 = m; *c.n0 = n; }
  return n;
}

// numpy complex128 division (Smith)
OPTB_DEV void cdiv(double a, double b, double c, double d, double& re, double& im) {
  if (fabs(c) >= fabs(d)) {
    double r = d / c, den = fma(d, r, c);
    double id = 1.0 / den;
    re = fma(b, r, a) * id; im = fma(-a, r, b) * id;
  } else {
    double r = c / d, den = fma(c, r, d);
    double id = 1.0 / den;
    re = fma(a, r, b) * id; im = fma(b, r, -a) * id;
  }
}

// What one interaction emits: all children start at the same lab point. N = most children any interaction of the
// scene can emit (1 for scenes that cannot split: the second slot and its code disappear at compile time).
template <int N>
struct Children {
  int n;
  double ox, oy, oz;    // lab origin
  double pl;            // _pathlength of the children
  double dx[N], dy[N], dz[N], I[N], qre[N], qim[N], nmed[N];
  // slot k with k a run-time value: an indexed store (writing it through selects to keep the arrays in registers
  // measured no faster on B200 and spilled more)
  OPTB_DEV void set(int k, double ax, double ay, double az, double i, double qr, double qi, double nm) {
    if (N == 1) k = 0;
    dx[k] = ax; dy[k] = ay; dz[k] = az; I[k] = i; qre[k] = qr; qim[k] = qi; nmed[k] = nm;
  }
};

// local child direction -> lab (ray_to_lab_coordinates :119-124; both normalisations)
OPTB_DEV void dir_to_lab(const double* __restrict__ T, bool ortho, double lx, double ly, double lz,
                         double& gx, double& gy, double& gz) {
  if (!ortho) {  // for an orthonormal T one normalisation (after the rotation) is the same as the reference's two
    double rn = rsqrt(dot3(lx, ly, lz, lx, ly, lz));
    lx *= rn; ly *= rn; lz *= rn;
  }
  double ex = dot3(T[0], T[1], T[2], lx, ly, lz);
  double ey = dot3(T[3], T[4], T[5], lx, ly, lz);
  double ez = dot3(T[6], T[7], T[8], lx, ly, lz);
  double r2 = rsqrt(dot3(ex, ey, ez, ex, ey, ez));
  gx = ex * r2; gy = ey * r2; gz = ez * r2;
}

// interact_local bodies for the winning leaf. (ox..dz) is the ray in the leaf's local frame, t the hit parameter.
template <bool ASPH, int N, bool PASSK>
OPTB_DEV void interact(const SceneView& sv, const int32_t* __restrict__ ni, const double* __restrict__ nf,
                       const Ray& ray, double unit, double ox, double oy, double oz, double dx, double dy, double dz,
                       double t, Children<N>& ch, const IndexCache& ic) {
  const double* T = nf + OPTB_NF_T;
  const double* c = nf + OPTB_NF_ORIGIN;
  const bool ortho = ni[OPTB_NI_ORTHO] != 0;
  const int kind = ni[OPTB_NI_INTER];
  // OPTB_I_PASS (PointObj / Monitor `return [ray]`, optical_component.py:438-440, monitor.py:174-175), PASSK variants
  // only, rides on the thin lens body: the child is the popped ray itself taken through Tinv and T once (:366-372),
  // i.e. a thin lens with f = inf and transmission 1 (the flattener writes both) applied at the ray's own ORIGIN
  // (t = 0 below: fma(0, d, o) is o exactly) that leaves q alone. It is compiled into the general kernel variants only
  // (trace_impl routes scenes with such a leaf there): in the specialised ones a branch of its own cost c4 +7 %, an
  // out-of-line body +16 %, this select +2 % -- for a degenerate case no example scene contains.
  const double tp = (PASSK && kind == OPTB_I_PASS) ? 0.0 : t;
  double Px = fma(tp, dx, ox), Py = fma(tp, dy, oy), Pz = fma(tp, dz, oz);
  ch.n = 0;
  ch.ox = dot3(T[0], T[1], T[2], Px, Py, Pz) + c[0];
  ch.oy = dot3(T[3], T[4], T[5], Px, Py, Pz) + c[1];
  ch.oz = dot3(T[6], T[7], T[8], Px, Py, Pz) + c[2];
  const bool hasq = (ray.flags & OPTB_RF_HASQ) != 0;
  const double refl = nf[OPTB_NF_REFL], trans = nf[OPTB_NF_TRANS];
  ch.pl = fma(t, ray.n, ray.pl);  // Ray.pathlength ray.py:145-147
  if (kind == OPTB_I_ABSORB) return;  // Block :501-503
  double gx, gy, gz;
  if (PASSK ? kind >= OPTB_I_THINLENS : kind == OPTB_I_THINLENS) {  // Lens :930-948 (and OPTB_I_PASS, see above)
    double f = nf[OPTB_NF_FOCAL];
    double qre = ray.qre, qim = ray.qim;
    if (hasq && (!PASSK || kind == OPTB_I_THINLENS)) {
      double q1r = ray.qre + t, q1i = ray.qim;
      cdiv(q1r, q1i, 1.0 - q1r / f, -(q1i / f), qre, qim);
    }
    double inv_f = 1.0 / f;
    dir_to_lab(T, ortho, dx - Px * inv_f, dy - Py * inv_f, dz - Pz * inv_f, gx, gy, gz);
    ch.set(0, gx, gy, gz, ray.I * trans, qre, qim, ray.n);
    ch.pl = ray.pl;  // the thin lens leaves _pathlength untouched
    ch.n = 1;
    return;
  }
  double nx, ny, nz, roc_fd;
  surf_normal<ASPH>(sv, ni, nf, Px, Py, Pz, nx, ny, nz, roc_fd);
  double dn = dot3(dx, dy, dz, nx, ny, nz);
  if (kind == OPTB_I_MIRROR) {  // BaseMirror :536-570, children [reflected, transmitted]
    double qre = ray.qre + t, qim = ray.qim;
    int k = 0;
    if (refl > 0) {
      dir_to_lab(T, ortho, fma(-2 * dn, nx, dx), fma(-2 * dn, ny, dy), fma(-2 * dn, nz, dz), gx, gy, gz);
      ch.set(k, gx, gy, gz, ray.I * refl, qre, qim, ray.n); k++;
    }
    if (trans > 0 && k < N) {
      dir_to_lab(T, ortho, dx, dy, dz, gx, gy, gz);
      ch.set(k, gx, gy, gz, ray.I * trans, qre, qim, ray.n); k++;
    }
    ch.n = k;
    return;
  }
  // BaseRefraciveSurface :617-717, children [transmitted | TIR, reflected]
  double wl_m = ray.wl * unit;
  double n1 = material_n_cached(sv, ic, ni[OPTB_NI_MAT1], wl_m);
  double n2 = material_n_cached(sv, ic, ni[OPTB_NI_MAT2], wl_m);
  double ROC = INFINITY;
  int rk = ni[OPTB_NI_ROCKIND];
  if (rk == OPTB_ROC_CONST) ROC = nf[OPTB_NF_ROC];
  else if (rk == OPTB_ROC_ASPHERE_FD) ROC = roc_fd;
  double nin, nout;
  if (dn < 0) { nin = n1; nout = n2; }
  else { nin = n2; nout = n1; ROC = -ROC; }
  double rtx = fma(-dn, nx, dx), rty = fma(-dn, ny, dy), rtz = fma(-dn, nz, dz);
  double sgn = dn > 0 ? 1.0 : -1.0;
  double cos_i = fmin(fmax(dn, -1.0), 1.0);
  double sin_i = sqrt(1.0 - cos_i * cos_i);
  double sin_t = (nin * sin_i) / nout;
  const double ratio = nin / nout;  // D of the refraction ABCD and the tangential scale of Snell's law
  const bool want_refl = (N > 1) && refl > 0;  // a scene whose interactions emit one ray at most has refl == 0 here
  double qtr = 0, qti = 0, qrr = 0, qri = 0;
  if (hasq) {  // ABCD of the refraction / of the reflection (:648-666); each only when a child will carry it
    double qr = ray.qre + t, qi = ray.qim;
    if (sin_t < 1 && trans > 0) {
      double Cc = (nin - nout) / (ROC * nout);
      cdiv(qr, qi, fma(Cc, qr, ratio), Cc * qi, qtr, qti);
    }
    if (!(sin_t < 1) || want_refl) {
      double C2 = 2.0 / ROC;
      cdiv(qr, qi, fma(C2, qr, 1.0), C2 * qi, qrr, qri);
    }
  }
  // reflected direction d + 2 cos_i (-n)
  double rfx = fma(-2 * cos_i, nx, dx), rfy = fma(-2 * cos_i, ny, dy), rfz = fma(-2 * cos_i, nz, dz);
  int k = 0;
  double g0x = 0, g0y = 0, g0z = 0;
  if (sin_t < 1) {
    if (trans > 0) {
      double cos_t = sqrt(1.0 - sin_t * sin_t);
      double kk = ratio, cs = cos_t * sgn;
      dir_to_lab(T, ortho, fma(kk, rtx, cs * nx), fma(kk, rty, cs * ny), fma(kk, rtz, cs * nz), g0x, g0y, g0z);
      ch.set(0, g0x, g0y, g0z, ray.I * trans, qtr, qti, nout); k = 1;
    }
  } else {  // total internal reflection (also taken when sin_t is NaN, as `sin_t < 1` is False)
    dir_to_lab(T, ortho, rfx, rfy, rfz, g0x, g0y, g0z);
    ch.set(0, g0x, g0y, g0z, ray.I, qrr, qri, ray.n); k = 1;
  }
  if (want_refl) {
    if (k == 1 && !(sin_t < 1)) {  // TIR + reflectivity: same direction twice
      gx = g0x; gy = g0y; gz = g0z;
    } else {
      dir_to_lab(T, ortho, rfx, rfy, rfz, gx, gy, gz);
    }
    ch.set(k, gx, gy, gz, ray.I * refl, qrr, qri, ray.n); k++;
  }
  ch.n = k;
}

// np.histogram(x, bins=30, range=(lo, hi)) bin index, -1 outside
// (norm = nb / (hi - lo) and step = (hi - lo) / nb depend on the monitor only: the upload precomputes them)
// The edges are np.linspace's: i * step and + lo each rounded, the last edge = hi. A fused i * step + lo differs from
// them by one ulp at many interior edges and would put a value on such an edge into the neighbouring bin.
OPTB_DEV int hist_bin(double x, double lo, double hi, double norm, double step) {
  const int nb = OPTB_HIST_BINS;
  if (!(x >= lo && x <= hi)) return -1;
  int idx = (int)((x - lo) * norm);
  if (idx == nb) idx = nb - 1;
  double e0 = __dadd_rn(__dmul_rn((double)idx, step), lo);
  double e1 = (idx + 1 == nb) ? hi : __dadd_rn(__dmul_rn((double)(idx + 1), step), lo);
  if (x < e0) idx--;
  else if (x >= e1 && idx != nb - 1) idx++;
  return idx;
}
OPTB_DEV int hist_bin(double x, double lo, double hi) {
  return hist_bin(x, lo, hi, OPTB_HIST_BINS / (hi - lo), (hi - lo) / OPTB_HIST_BINS);
}

}  // namespace optb
