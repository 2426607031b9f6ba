/*
 * optb.h -- C ABI of the B200 ray-propagation engine that replaces the per-ray
 * Python bounce loop of optable (reference: tim4431/optable).
 *
 * The reference has no FFI layer: its boundary for this path is the Python method
 *   OpticalTable.ray_tracing            optable/optical_table.py:57-72
 *   OpticalTable._single_ray_tracing    optable/optical_table.py:74-147
 * which, per popped ray, calls
 *   OpticalComponent.interact           optable/optical_component.py:337-378
 *   ComponentGroup.interact             optable/component_group.py:93-122
 * and, after the queue drains, Monitor.record  optable/monitor.py:183-193.
 * Every entry point below states which of those it replaces.
 *
 * Rules of the ABI: extern "C", plain pointers and sizes, int status returns
 * (0 = ok, <0 = error, text via optb_last_error). The library never allocates
 * caller-visible memory: ray, result and workspace buffers are device pointers
 * owned by the caller (host pointers for the *_host entry point). Opaque
 * handles (ctx, scene) are owned by the library.
 *
 * The same structs are consumed by oracle/optb_oracle.c (test infrastructure,
 * host pointers) so that the CUDA path and the CPU restatement are fed
 * byte-identical tables.
 */
#ifndef OPTB_H
#define OPTB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OPTB_ABI_VERSION 8  /* 8: OPTB_G_CSG rows may carry a postfix program (p0 = 2) for nested composites */

/* ---- scene node table ------------------------------------------------------
 * The component tree (OpticalTable.components, groups nested to any depth) is
 * flattened in DFS pre-order: one node per ComponentGroup and one per leaf
 * OpticalComponent. "skip" is the index of the first node after the node's
 * subtree, so a failed bounding-box test is `i = skip` and the traversal is a
 * forward scan (component_group.py:98-115 restated as a linear walk).
 * Tie-break of the reference (strict '<' at table level, np.argmin inside a
 * group: optical_table.py:121, component_group.py:118-120) = smallest t, then
 * smallest pre-order index.
 */

/* geometry kinds: which Surface subclass the leaf carries (optable/surfaces.py) */
enum {
  OPTB_G_GROUP = 0,   /* ComponentGroup: lab AABB only                        */
  OPTB_G_CIRCLE = 1,  /* Circle        surfaces.py:139-162   p0 = radius       */
  OPTB_G_RECT = 2,    /* Rectangle     surfaces.py:165-209   p0 = w/2, p1 = h/2 */
  OPTB_G_SPHERE = 3,  /* Sphere        surfaces.py:284-336   p0 = R, p1 = height, p2..p7 = local bbox */
  OPTB_G_ASPHERE = 4, /* ASphere       surfaces.py:339-423   p0 = radius, p1..p5 = coeffs, p6 = xmin, p7 = xmax */
  OPTB_G_CYL = 5,     /* Cylinder      surfaces.py:212-281   p0 = r, p1 = height, p2 = theta0, p3 = theta1 */
  OPTB_G_POLY2D = 6,  /* Polygon, planar=True   surfaces.py:426-568   aux -> polygon record */
  OPTB_G_POLY3D = 7,  /* Polygon, planar=False  (curved branch, linear f)  aux -> polygon record */
  OPTB_G_GRID = 9,    /* a ComponentGroup whose leaf children sit on a regular 2-D lattice (MMA, MLA, DMD:
                         component_group.py:228-391): a group for every purpose, plus a lattice descriptor in the aux
                         pool (NI_AUX) from which the device lists the few cells a ray can reach instead of
                         descending a box hierarchy over thousands of children. See OPTB_GRID_* below.         */
  OPTB_G_CSG = 8      /* Plane.union / Plane.subtract  surfaces.py:100-136
                         p0 = op (0 = A and not B, 1 = A or B),
                         p1 = kind A, p2,p3 = params A (or aux offset for poly),
                         p4 = kind B, p5,p6 = params B (or aux offset for poly);
                         p0 = 2: nested composite (an operand is itself a union / subtract): NI_AUX -> postfix
                         program in the aux pool, [n_tokens, then n_tokens x (code, a, b)]: code = OPTB_G_CIRCLE /
                         OPTB_G_RECT / OPTB_G_POLY2D pushes that shape's within_boundary (a, b = its params or aux
                         offset), OPTB_CSG_SUBTRACT / OPTB_CSG_UNION pop B then A and push (A and not B) / (A or B);
                         at most OPTB_CSG_MAX_DEPTH values on the stack, exactly one left at the end */
};

#define OPTB_CSG_SUBTRACT (-1)
#define OPTB_CSG_UNION (-2)
#define OPTB_CSG_MAX_DEPTH 30

/* interaction kinds: which interact_local body applies (optical_component.py) */
enum {
  OPTB_I_NONE = 0,
  OPTB_I_MIRROR = 1,   /* BaseMirror.interact_local            :536-570 */
  OPTB_I_REFRACT = 2,  /* BaseRefraciveSurface.interact_local  :617-717 */
  OPTB_I_THINLENS = 3, /* Lens.interact_local                  :930-948 */
  OPTB_I_ABSORB = 4,   /* Block.interact_local                 :501-503 */
  OPTB_I_PASS = 5      /* PointObj / Monitor.interact_local    :438-440, monitor.py:174-175: `return [ray]` -- the child is
                          the popped ray itself (origin NOT moved to the hit point, q and path length untouched), so it
                          hits the same surface again at the same t until the pop cap: a Monitor listed in
                          table.components. Degenerate, reproduced as is. */
};

/* radius-of-curvature source for the ABCD matrices (optical_component.py:631-639) */
enum { OPTB_ROC_INF = 0, OPTB_ROC_CONST = 1, OPTB_ROC_ASPHERE_FD = 2 };

/* ASphere.f_asphere closures shipped by the reference (component_group.py:1065-1107) */
enum {
  OPTB_ASPH_PARAMETRIC = 1, /* coeffs = R, kappa, a4, a6, a8 */
  OPTB_ASPH_EXACT_SPH = 2   /* coeffs = EFL, n               */
};

/* node_i columns (int32 per node) */
enum {
  OPTB_NI_GEOM = 0,
  OPTB_NI_INTER = 1,
  OPTB_NI_SKIP = 2,
  OPTB_NI_AABB = 3,   /* 1: test NF_AABB against the lab ray before descending/testing
                         (groups, and leaves that are children of a group;
                         top-level leaves are never box-tested: SURVEY A.3)      */
  OPTB_NI_MAT1 = 4,   /* index into the material table (_n1; local x>0 side)     */
  OPTB_NI_MAT2 = 5,   /* (_n2; local x<0 side)                                   */
  OPTB_NI_CAPSLOT = 6,/* -1, or row of the interact-count table (max_interact_count) */
  OPTB_NI_AUX = 7,    /* offset (in doubles) into aux pool, or asphere form       */
  OPTB_NI_ROCKIND = 8,
  OPTB_NI_LEAF = 9,   /* dense leaf number (-1 for groups); reported as hit index */
  OPTB_NI_ORTHO = 10, /* 1: Tinv is orthonormal to 1e-14, so |Tinv d| = 1 to rounding and the device skips the
                         re-normalisations of ray_to_local/lab_coordinates (a 1e-16 relative difference)      */
  OPTB_NI_STRIDE = 12
};

/* node_f columns (double per node) */
enum {
  OPTB_NF_AABB = 0,    /* xmin,xmax,ymin,ymax,zmin,zmax: the object's own cached .bbox */
  OPTB_NF_ORIGIN = 6,  /* component origin c                                        */
  OPTB_NF_TINV = 9,    /* np.linalg.inv(transform_matrix), row-major 3x3            */
  OPTB_NF_T = 18,      /* transform_matrix, row-major 3x3                           */
  OPTB_NF_P = 27,      /* p0..p7 geometry parameters (see geometry kinds)           */
  OPTB_NF_REFL = 35,
  OPTB_NF_TRANS = 36,
  OPTB_NF_FOCAL = 37,
  OPTB_NF_ROC = 38,
  OPTB_NF_CAPMAX = 39, /* max_interact_count as double (the reference compares count < max) */
  OPTB_NF_STRIDE = 40
};

/* polygon record in the aux pool (doubles):
 * [0] nverts, [1..3] unit normal, [4..6] vertices[0], [7..9] basis u, [10..12] basis v,
 * [13..18] bbox, [19 ..] verts2d as (x,y) pairs.                                    */
enum { OPTB_POLY_HEADER = 19 };

/* lattice descriptor of an OPTB_G_GRID node in the aux pool (doubles). Child k = i * n_inner + j of the group (list
 * order, component_group.py:104-115) has the centre of its lab box within `R - |half diagonal|` of
 * c00 + i U + j V. A ray can only pass the reference's own box test of child (i, j) at a point P with
 * |P - (c00 + i U + j V)| <= R, i.e. |(P - c00).nhat| <= R, |(P - c00).Ud - i| <= rho_a, |(P - c00).Vd - j| <= rho_b
 * (Ud, Vd: dual basis of U, V in the lattice plane). The device tests exactly the children inside that window with
 * their own stored boxes: a superset of what the reference's test passes, so the tested set is the reference's.   */
enum {
  OPTB_GRID_NOUTER = 0, OPTB_GRID_NINNER = 1, OPTB_GRID_NEXT = 2, /* lattice size; children outside the lattice (tested always) */
  OPTB_GRID_R = 3, OPTB_GRID_C00 = 4, OPTB_GRID_NHAT = 7, OPTB_GRID_UD = 10, OPTB_GRID_VD = 13,
  OPTB_GRID_RHOA = 16, OPTB_GRID_RHOB = 17,
  OPTB_GRID_CELLS = 18 /* node index of every lattice child (n_outer * n_inner doubles), then of the extra children */
};

/* material table (optable/material.py): kind 0 = constant n (f[0]),
 * kind 1 = Sellmeier-3 (f[0..2] = B, f[3..5] = C in um^2)                  :93-120,
 * kind 2 = per-wavelength table for Material(n=<any Python callable>)      :4-21: the host evaluates the callable
 *          once per distinct wavelength of the batch (SURVEY App. D); f[0] = offset (in doubles) into the aux pool,
 *          f[1] = number of entries; entries are (wavelength_in_metres, n) pairs sorted by wavelength. The device
 *          looks the ray's wavelength*unit up by exact match; a miss raises OPTB_ST_LUT_MISS.                  */
enum { OPTB_MAT_CONST = 0, OPTB_MAT_SELLMEIER = 1, OPTB_MAT_LUT = 2, OPTB_MF_STRIDE = 8 };

/* monitor table (optable/monitor.py:5-13): c[3], Tinv[9], w/2, h/2, then the LAB-frame
 * tangent_Y / tangent_Z (columns 1,2 of transform_matrix). Monitor.get_yList dots the
 * monitor-LOCAL hit point with the LAB tangent (monitor.py:78-100, a reference quirk for
 * rotated monitors); the histograms reproduce exactly that.                               */
enum {
  OPTB_MON_ORIGIN = 0, OPTB_MON_TINV = 3, OPTB_MON_HW = 12, OPTB_MON_HH = 13,
  OPTB_MON_TY = 14, OPTB_MON_TZ = 17, OPTB_MON_ORTHO = 20 /* 1.0 when Tinv is orthonormal */, OPTB_MON_STRIDE = 24
};
enum { OPTB_HIST_BINS = 30 };

typedef struct optb_scene_desc {
  int32_t abi_version;
  int32_t n_nodes;
  int32_t n_leaves;
  int32_t n_materials;
  int32_t n_monitors;
  int32_t n_capslots;
  int64_t n_aux;           /* doubles in aux pool */
  const int32_t* node_i;   /* [n_nodes][OPTB_NI_STRIDE] */
  const double* node_f;    /* [n_nodes][OPTB_NF_STRIDE] */
  const int32_t* mat_kind; /* [n_materials] */
  const double* mat_f;     /* [n_materials][OPTB_MF_STRIDE] */
  const double* mon_f;     /* [n_monitors][OPTB_MON_STRIDE] */
  const double* aux;       /* [n_aux] */
} optb_scene_desc;

/* ---- rays ------------------------------------------------------------------
 * SoA fp64 ray state = the numeric fields of optable.Ray (ray.py:58-105).
 * One entry per *initial* ray (a "root"); descendants created by splitting
 * live in library workspace. 104 B per ray.
 */
enum {
  OPTB_RF_ALIVE = 1u, /* Ray.alive                                  */
  OPTB_RF_HASQ = 2u   /* Ray.qo is not None                         */
};

typedef struct optb_rays {
  int64_t n;
  const double* ox; const double* oy; const double* oz; /* Ray.origin                */
  const double* dx; const double* dy; const double* dz; /* Ray._direction (unit)     */
  const double* intensity;
  const double* wavelength; /* scene units; 0.0 when None (ray.py:90-92)              */
  const double* q_re; const double* q_im; /* Ray.qo (ignored unless OPTB_RF_HASQ)     */
  const double* pathlength; /* Ray._pathlength                                        */
  const double* n_medium;   /* Ray.n (vars(ray)["_n"] evaluated)                      */
  const double* length;     /* Ray.length limit; +inf when None. May be NULL (= all +inf) */
  const uint32_t* flags;    /* OPTB_RF_*. May be NULL (= alive, has q)                */
  const int32_t* family;    /* dense index of Ray._id for interact caps; may be NULL (= root index) */
  uint32_t broadcast;       /* bit f set: fp64 column f (order above, ox = bit 0 ... length = bit 12) holds ONE
                               value shared by all n rays (a collimated, monochromatic bundle then costs two
                               columns of host->device traffic instead of thirteen)                          */
  uint32_t reserved;
} optb_rays;

/* ---- parameters ------------------------------------------------------------ */
typedef struct optb_params {
  int64_t max_trace_num;  /* perfomance_limit["max_trace_num"], default 2000 (optical_table.py:87-97) */
  double unit;            /* Ray.unit (metres per scene unit; base.py:31); index evaluated at wavelength*unit */
  int32_t record_segments;/* 1: fill optb_result.seg_* (= OpticalTable.rays)           */
  int32_t record_hits;    /* 1: fill optb_result.hit_* (= Monitor._data_raw)           */
  int32_t record_hist;    /* 1: accumulate Monitor._get_hist_y-style 30-bin + 30x30 histograms */
  int32_t chain_len;      /* max in-thread pops per launch for a root whose alive set is one ray
                             (0 = unlimited). Scheduling only; results do not depend on it.   */
  int32_t n_families;     /* rows of cap_counts per slot                                */
  int32_t caps_slack;     /* 1: the caller guarantees that no interact cap can bind in this call (every cap >=
                             initial count + max_trace_num * rays per family). Counts are still kept, but the
                             scene is traced on the parallel path instead of the family-serial one. If a cap
                             binds anyway, OPTB_ST_CAP_ORDER is raised.                                  */
  int32_t flag_ambiguity; /* 1: evaluate the ambiguity mask of SURVEY A.9 at every pop (OPTB_AMB_* bits OR-ed per
                             initial ray into optb_result.root_flags, flagged roots counted in OPTB_C_FLAGGED).
                             A diagnostics mode: it runs the general kernel variant.                        */
  int32_t sorted_rows;    /* optb_trace_host only: 1 = deliver the monitor rows in (root, monitor, pop) order and the
                             segments in (root, pop) order -- the order Monitor.record / OpticalTable.rays have after
                             the reference traced the initial rays one after another -- instead of device append
                             order. Sorted on the device (optb_sort_rows) before the copy back.                  */
  int32_t reference_roots;/* 1: curved-surface hit distances are the last iterate of the reference's own root finder
                             (scipy.optimize.brentq with its default xtol = 2e-12, optical_component.py:126-134) run
                             on the same sign-scan bracket, instead of the closed-form / Newton root the default path
                             converges to rounding. The two differ by up to 2e-12 (brentq's tolerance), which long
                             chaotic paths amplify; this mode follows the reference's path, the default one is
                             faster and closer to the true surface. Decisions (hit index, bounce count) agree. */
  int32_t reserved;
} optb_params;

/* Ambiguity bits (SURVEY A.9, the "stated epsilon" of the parity bar): set for an initial ray when, at some pop,
 * a decision of the reference hinges on less than the stated margin, so that hit index / bounce count of that
 * ray are excluded from bit-exact comparison.                                                               */
enum {
  OPTB_AMB_TIE = 1,       /* the two closest candidate surfaces are hit within 1e-9 relative of each other   */
  OPTB_AMB_APERTURE = 2,  /* a hit or near-hit lies within 1e-9 * scale of an aperture edge (r - radius, |y| - w/2,
                             |z| - h/2, cap x limits, cylinder theta / z limits, polygon edge)                 */
  OPTB_AMB_GRAZING = 4,   /* |d.n| < 1e-6 at the interaction                                                  */
  OPTB_AMB_TIR = 8,       /* |sin_t - 1| < 1e-9 (transmission vs total internal reflection)                    */
  OPTB_AMB_EPS = 16,      /* a candidate t within 1e-11 of the 1e-9 self-intersection guard, or within 1e-9
                             relative of the ray's length limit                                               */
  OPTB_AMB_SCAN = 32,     /* curved leaf: a sign-scan sample with |f| < 1e-12, or the bracket within 1e-9 of the
                             t = 100 clip                                                                      */
  OPTB_AMB_SLAB = 64      /* a box test with | |d_axis| - 1e-8 | < 1e-10, or passed/failed by less than 1e-11   */
};

/* ---- results ---------------------------------------------------------------
 * Segments: one per pop (optical_table.py:115-134): the truncated parent on a
 * hit (length = t, alive = 0) or the ray itself on a miss (length = +inf or its
 * own limit, alive as it was). Reference order = (root, pop_seq); the GPU
 * appends unordered and the host sorts by that key.
 * Hits: Monitor.record rows (P_local, intensity, t, ray) with the ray replaced
 * by its key (root, pop_seq) plus the lab direction and q of that segment.
 */
typedef struct optb_result {
  int64_t seg_capacity;
  int64_t hit_capacity;
  /* segments (all may be NULL when record_segments == 0) */
  double* seg_ox; double* seg_oy; double* seg_oz;
  double* seg_dx; double* seg_dy; double* seg_dz;
  double* seg_length;      /* +inf = None */
  double* seg_intensity;
  double* seg_wavelength;
  double* seg_q_re; double* seg_q_im;
  double* seg_pathlength;
  double* seg_n;
  uint32_t* seg_flags;     /* OPTB_RF_* of the segment */
  uint32_t* seg_root;
  uint32_t* seg_pop;
  int32_t* seg_leaf;       /* dense leaf index that ended the segment; -1 = escaped  */
  /* monitor hits. hit_monitor is required when record_hits == 1; every other hit_* column may be NULL
   * (not wanted by the caller: it is then neither written nor copied back)                        */
  int32_t* hit_monitor;
  uint32_t* hit_root;
  uint32_t* hit_pop;
  double* hit_px; double* hit_py; double* hit_pz; /* P in monitor-local coordinates */
  double* hit_intensity;
  double* hit_t;
  double* hit_dx; double* hit_dy; double* hit_dz; /* lab direction of the segment    */
  double* hit_q_re; double* hit_q_im;
  uint64_t* hit_key;       /* optional packed row key: root << 32 | monitor << 24 | pop (needs max_trace_num <= 2^24
                              and <= 256 monitors). Numeric order of the key = (root, monitor, pop) = the order
                              Monitor.record fills _data_raw when the initial rays are traced one after another.
                              8 B instead of the 12 B of hit_monitor + hit_root + hit_pop (which may then be NULL,
                              hit_monitor included)                                                        */
  uint32_t* root_flags;    /* [rays.n] OPTB_AMB_* bits per initial ray (params.flag_ambiguity = 1); may be NULL */
  /* histograms: int64 [n_monitors][30] over local y in +-w/2, [n_monitors][30][30] over (y,z) */
  int64_t* hist_y;
  int64_t* hist_yz;
  /* interact-count table: int32 [n_capslots][n_families], in/out (persists across calls like
   * OpticalComponent._interact_count, optical_component.py:136-149)                    */
  int32_t* cap_counts;
  /* counters: int64[OPTB_C_COUNT], written by the library */
  int64_t* counters;
} optb_result;

enum {
  OPTB_C_SEGMENTS = 0,     /* pops = output segments                                  */
  OPTB_C_INTERACTIONS = 1, /* segments that ended on a surface (finite length): THE metric unit */
  OPTB_C_HITS = 2,         /* monitor rows                                            */
  OPTB_C_TESTS = 3,        /* ray-leaf intersection tests performed                   */
  OPTB_C_DROPPED = 4,      /* queued rays dropped by the pop cap (optical_table.py:86-97) */
  OPTB_C_STATUS = 5,       /* bit flags OPTB_ST_*                                     */
  OPTB_C_GENERATIONS = 6,  /* wavefront generations executed                          */
  OPTB_C_LAUNCHES = 7,     /* kernels launched by this call                           */
  OPTB_C_TESTS_CURVED = 8, /* the part of OPTB_C_TESTS that ran the curved branch (local box + sign scan) */
  OPTB_C_BOX_TESTS = 9,    /* lab-frame bounding-box tests performed                  */
  OPTB_C_FLAGGED = 10,     /* initial rays with any OPTB_AMB_* bit (params.flag_ambiguity) */
  OPTB_C_RESERVED = 11,
  OPTB_C_COUNT = 12
};

enum {
  OPTB_ST_SEG_OVERFLOW = 1,  /* seg_capacity too small: counts are right, rows beyond capacity dropped */
  OPTB_ST_HIT_OVERFLOW = 2,
  OPTB_ST_WORK_OVERFLOW = 4, /* workspace too small for the live ray set                */
  OPTB_ST_CAP_ORDER = 8,     /* an interact cap bound while its family had concurrent rays:
                                reference result depends on sequential order          */
  OPTB_ST_LUT_MISS = 16      /* a ray's wavelength is missing from a material's per-wavelength table */
};

/* ---- entry points ---------------------------------------------------------- */
typedef struct optb_ctx optb_ctx;
typedef struct optb_scene optb_scene;

/* Library/ABI version (compile-time constant). */
int optb_abi_version(void);

/* One context per device. Replaces nothing in the reference (it is single-process, single-thread). */
int optb_ctx_create(int device, optb_ctx** out);
int optb_ctx_destroy(optb_ctx* ctx);
const char* optb_last_error(const optb_ctx* ctx);

/* Upload the flattened component tree: the device-side form of OpticalTable.components /
 * OpticalTable.monitors (optical_table.py:25-43). Host pointers in `desc`.              */
int optb_scene_upload(optb_ctx* ctx, const optb_scene_desc* desc, optb_scene** out);
int optb_scene_destroy(optb_ctx* ctx, optb_scene* scene);

/* Sweep scene: K = n_configs configurations of one scene with the same topology (descs[0..K-1], host pointers), e.g.
 * one table built over a parameter grid (the GUI's scan, optimize: optable/interact.py:465-630) or the draws of a
 * tolerance study. The handle is an ordinary optb_scene; every optb_trace / optb_trace_host on it traces the bundle
 * of rays.n = N rays through all K configurations in one call:
 *   - K * N roots: root k * N + r is ray r in configuration k (seg_root, hit_root and hit_key carry that number, so
 *     optb_sort_rows gives configuration-major order); K * N must stay below 2^32 (-7 otherwise);
 *   - hist_y / hist_yz are [K][n_monitors][...]; root_flags would be [K * N]; counters are totals over all configurations;
 *   - rays.family must be NULL (every root is its own family), except on a scene with interact caps and
 *     params.caps_slack = 0: there rays.family (dense, < n_families) runs the family-serial sweep, with
 *     params.n_families = F families per configuration and cap_counts [n_capslots][n_configs * n_families], in and
 *     out, column k * F + f = family f in configuration k. A capped scene without a family column needs
 *     params.caps_slack when it can split (-7 otherwise); flag_ambiguity and reference_roots are rejected (-7);
 *   - optb_workspace_bytes(scene, N, max_live) sizes for K * N roots (max_live counts over all configurations);
 *   - optb_scene_update_nodes is rejected (-7): upload the configurations again.
 * Every desc must have the same n_nodes, n_leaves, n_materials, n_monitors, n_capslots and n_aux, identical node_i rows
 * except column OPTB_NI_ORTHO (a leaf index, skip pointer, material and cap slot mean the same in every configuration)
 * and identical mat_kind; node_f, mat_f, mon_f and aux may differ (poses, boxes, apertures, lattice descriptors,
 * reflectivity, glass coefficients, monitor placement). Violations fail with -5 and name the configuration.
 * Added without a change of OPTB_ABI_VERSION: that number stamps the layout and meaning of the structs above, which every
 * consumer of a scene description (this library, the C restatement in oracle/) checks, and none of them changed; a host
 * written for this entry point against an older library fails to link instead.                                     */
int optb_scene_upload_sweep(optb_ctx* ctx, const optb_scene_desc* descs, int32_t n_configs, optb_scene** out);

/* Sweep scene from one base scene plus the rows that differ: for a sweep that varies a few components and monitors of
 * a large scene (a tolerance or Monte Carlo study), only those rows travel, and the K configuration blobs are written on
 * the device. Configuration k is `base` with
 *   - node_i / node_f row nodes[v] replaced by node_i[k][v] / node_f[k][v] (host arrays [K][n_var_nodes][OPTB_NI_STRIDE]
 *     and [K][n_var_nodes][OPTB_NF_STRIDE]), and
 *   - mon_f record monitors[w] replaced by mon_f[k][w] ([K][n_var_monitors][OPTB_MON_STRIDE]);
 * mat_kind, mat_f and aux are the base's in every configuration. The handle has exactly the contract of
 * optb_scene_upload_sweep (the K * N root numbering, [K][n_monitors] histograms, the same -7 rejections, update_nodes
 * refused), and every configuration blob is byte for byte the one optb_scene_upload_sweep builds from the K materialised
 * descriptions, cull bits and kernel choice included (a reflectivity that is > 0 in one configuration picks the
 * splitting kernels). Synchronous: the scene is ready when the call returns.
 * Fails with -5 when a node or monitor index is out of range or repeated, when a varied node_i row differs from the
 * base's in a column other than OPTB_NI_ORTHO (naming the configuration, row and column) or a varied row fails the checks
 * optb_scene_upload applies to a node (naming the configuration and row); with -6 when the K blobs exceed the scene
 * size limit. Added without a change of OPTB_ABI_VERSION: no struct changed.                                        */
int optb_scene_upload_sweep_rows(optb_ctx* ctx, const optb_scene_desc* base, int32_t n_configs,
                                 const int32_t* nodes, int32_t n_var_nodes, const double* node_f, const int32_t* node_i,
                                 const int32_t* monitors, int32_t n_var_monitors, const double* mon_f, optb_scene** out);

/* Rewrite the rows of the listed nodes of an uploaded scene from `desc` (the tables the scene was uploaded from, with
 * those rows changed in place: same node count, kinds, skip pointers, materials and aux pool). What a GUI loop needs
 * when one component moved (optable/interact.py:455-457 re-runs the user's script per slider event): a few hundred
 * bytes go to the device instead of the whole scene, the scene handle -- and any CUDA graph captured over traces of
 * it -- stays valid. Stream-ordered on `stream`.                                                                 */
int optb_scene_update_nodes(optb_ctx* ctx, optb_scene* scene, const optb_scene_desc* desc,
                            const int32_t* nodes, int32_t n_nodes, void* stream);

/* Bytes of device workspace optb_trace needs for `n_rays` roots when at most
 * `max_live` rays are alive at once (max_live >= n_rays). Sweep scene: n_rays rays per configuration, sized for
 * n_configs * n_rays roots.                                                            */
int64_t optb_workspace_bytes(const optb_scene* scene, int64_t n_rays, int64_t max_live);

/* The bounce loop: replaces OpticalTable.ray_tracing/_single_ray_tracing for a whole batch of
 * initial rays (optical_table.py:57-147) including Monitor.record (monitor.py:183-193).
 * All pointers in `rays`/`out` and `workspace` are DEVICE pointers. Work is enqueued on
 * `stream` (a cudaStream_t); the call may synchronise that stream between generations when the
 * scene can split rays. out->counters is valid after the stream is synchronised.           */
int optb_trace(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays,
               const optb_params* params, optb_result* out,
               void* workspace, int64_t workspace_bytes, void* stream);

/* Same call with HOST buffers (pinned or pageable): stages rays to the device, traces, and copies
 * the filled prefix of every requested result array back. Used for end-to-end timing.         */
int optb_trace_host(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays,
                    const optb_params* params, optb_result* out);

/* The launch plan of a trace, without tracing: which trace kernel variant optb_trace / optb_trace_host would run for
 * (scene, rays, params) and with how much shared memory. Runs the same parameter checks as a trace that do not read
 * the result buffers (the plan reads only rays->n and whether rays->family is set) and sets the kernel's shared-memory
 * attribute as a trace does; enqueues nothing. out[5]:
 *   out[0]  variant bits (OPTB_PLAN_*)
 *   out[1]  scene blob bytes (all configurations of a sweep scene)
 *   out[2]  dynamic shared memory the trace kernel launches with (blob and / or histograms)
 *   out[3]  the selected kernel's static shared memory
 *   out[4]  the device's opt-in shared memory per block (cudaDevAttrMaxSharedMemoryPerBlockOptin)
 * A scene's tables are staged in shared memory when its blob fits the opt-in limit less the largest static shared
 * memory of the shared-memory trace kernels, so that any later trace of the scene (diagnostics modes and family column
 * included) can launch. Added without a change of OPTB_ABI_VERSION: no struct changed.                          */
#define OPTB_PLAN_SMEM      (1u << 0)   /* tables staged in shared memory (else read from global memory) */
#define OPTB_PLAN_SERIAL    (1u << 1)   /* family-serial path (binding interact caps) */
#define OPTB_PLAN_BOX_SHIFT 2           /* 2 bits: 0 no boxes, 1 box walk, 2 box walk + lattice windows */
#define OPTB_PLAN_BOX_MASK  (3u << OPTB_PLAN_BOX_SHIFT)
#define OPTB_PLAN_ASPH      (1u << 4)   /* asphere root search compiled in */
#define OPTB_PLAN_SPLIT     (1u << 5)   /* wavefront (splitting) form */
#define OPTB_PLAN_FLAG      (1u << 6)   /* params.flag_ambiguity */
#define OPTB_PLAN_BRENT     (1u << 7)   /* params.reference_roots */
#define OPTB_PLAN_PASSK     (1u << 8)   /* pass-through leaves (OPTB_I_PASS) */
#define OPTB_PLAN_SWEEP     (1u << 9)   /* sweep scene */
#define OPTB_PLAN_HIST_SMEM (1u << 10)  /* histograms accumulated in shared memory (else global atomics); 0 without record_hist */
int optb_trace_plan(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* params,
                    int64_t out[5]);

/* Put the first n_seg segment rows of `res` into (root, pop) order and its first n_hit monitor rows into
 * (root, monitor, pop) order, in place: what a caller of optb_trace does once it has read the counters (rows are
 * appended in device order). DEVICE pointers; NULL columns are skipped; the key columns (seg_root + seg_pop;
 * hit_key, or hit_root + hit_pop + hit_monitor) must be present. Needs pop < 2^24 and <= 256 monitors (-7 otherwise).
 * workspace: optb_sort_workspace_bytes(max(n_seg, n_hit)) bytes of device memory.                                */
int64_t optb_sort_workspace_bytes(int64_t n_rows);
int optb_sort_rows(optb_ctx* ctx, const optb_result* res, int64_t n_seg, int64_t n_hit,
                   void* workspace, int64_t workspace_bytes, void* stream);

/* ---- monitor analytics on the device (SURVEY 8f item 2; monitor.py:78-253) ----------------------------------------
 * Monitor rows that are still in HBM, reduced per group of rows (optb_monitor_stats_grouped below). For every row it
 * evaluates, in its group's frame, what the reference's Monitor accessors derive per row --
 *   y = P_local . tangent_Y, z = P_local . tangent_Z   (get_yList / get_zList :78-100; LOCAL point, LAB tangent: the
 *                                                        reference's own convention, kept)
 *   tY = d . tangent_Y, tZ = d . tangent_Z             (get_tYList / tZList :137-157)
 *   waist distance = +-Re(q + t), minus when d . normal > 0   (get_waist_distance :202-216)
 * -- writes them to the optional per-row columns and accumulates, per group, the row count, sum of intensities
 * (sum_intensity / avg_intensity :236-242), first and second moments and extrema of y and z, the sum of the waist
 * distances and the 30-bin np.histogram of y over +-width/2 (_get_hist_y :195-200, from which std_histy :244-249
 * follows) in the OPTB_MS_* slots. No row leaves the device.                                                     */
typedef struct optb_monitor_frame {
  double tangent_y[3], tangent_z[3], normal[3]; /* Monitor.tangent_Y / tangent_Z / normal (lab frame) */
  double half_width, half_height;
} optb_monitor_frame;
enum {
  OPTB_MS_COUNT = 0, OPTB_MS_SUM_I = 1, OPTB_MS_SUM_Y = 2, OPTB_MS_SUM_YY = 3, OPTB_MS_SUM_Z = 4, OPTB_MS_SUM_ZZ = 5,
  OPTB_MS_SUM_WD = 6, OPTB_MS_MIN_Y = 7, OPTB_MS_MAX_Y = 8, OPTB_MS_MIN_Z = 9, OPTB_MS_MAX_Z = 10,
  OPTB_MS_SUM_TY = 11, OPTB_MS_SUM_TYTY = 12,
  /* sums of (y - mean_y)^2, (z - mean_z)^2, (tY - mean_tY)^2 over a group's rows, taken in a second pass about the
   * means of the first (std_y = sqrt(M2_Y / count) keeps full precision where SUM_YY / count - mean_y^2 cancels, e.g.
   * a small spot far off the monitor's axis). M2_TY is 0 without hit_dx..dz. Added in slots that were unused before,
   * without a change of OPTB_ABI_VERSION: no struct changed.                                                      */
  OPTB_MS_M2_Y = 13, OPTB_MS_M2_Z = 14, OPTB_MS_M2_TY = 15,
  OPTB_MS_HIST = 16, /* 30 counts */
  OPTB_MS_STRIDE = 48
};
/* The summaries of every (configuration, monitor) group of the rows [first, first + n) in one call: what a scan, an
 * optimizer or a tolerance study ranks after one sweep (optb_scene_upload_sweep), or all monitors of one trace.
 *   - rows: DEVICE pointers (hit_px/py/pz, hit_intensity, hit_t required; hit_dx..dz for tY/tZ/waist sign, hit_q_re for
 *     the waist distance).
 *   - group of a row: g = k * n_monitors + m, k = root / rays_per_config (the K x N root numbering of a sweep scene;
 *     rays_per_config = 0: one configuration, k = 0), root from hit_root or else hit_key >> 32, m from hit_monitor or
 *     else (hit_key >> 24) & 0xff. A row with k >= n_configs or m outside [0, n_monitors) belongs to no group: its
 *     per-row outputs are NaN and it is counted nowhere (the counts then add up to less than n).
 *   - frames: DEVICE optb_monitor_frame[n_configs * n_monitors], group g evaluated in frames[g].
 *   - stats: DEVICE double[n_configs * n_monitors][OPTB_MS_STRIDE], overwritten; group g's OPTB_MS_* slots over its
 *     own rows (M2_* about that group's own means; the histogram bins like np.histogram); a group without rows reads
 *     zeros, min +inf, max -inf.
 *   - y, z, ty, tz, waist: DEVICE double[n] or NULL, row first + i at [i], evaluated in its group's frame.
 *   - rows may come in any order (sorted by optb_sort_rows, or in device append order).
 *   - deterministic: the same rows in the same order give bit-identical stats on every call, on any stream, whatever
 *     the device's SM count (rows are sorted by group, each group is reduced in tiles of a fixed size in a fixed order,
 *     and its tile partials are combined in tile order).
 *   - workspace: optb_monitor_stats_grouped_workspace_bytes(n, n_configs * n_monitors) bytes of device memory
 *     (-1: n >= 2^31 - 1 or a group count outside [1, 2^20]).
 * Fails with -7 when a required column is missing (the monitor column; the root column when rays_per_config > 0),
 * slopes or waist distances are requested without hit_dx..dz / hit_q_re, n_monitors > 256, n_configs * n_monitors
 * > 2^20, n >= 2^31 - 1, or the workspace is too small. Enqueued on `stream`, without a host synchronisation.
 * Added without a change of OPTB_ABI_VERSION: no struct changed, and a host written for this entry point against an
 * older library fails to link instead.                                                                           */
int64_t optb_monitor_stats_grouped_workspace_bytes(int64_t n_rows, int32_t n_groups);
int optb_monitor_stats_grouped(optb_ctx* ctx, const optb_result* rows, int64_t first, int64_t n,
                               int64_t rays_per_config, int32_t n_configs, int32_t n_monitors,
                               const optb_monitor_frame* frames, double* stats, double* y, double* z, double* ty,
                               double* tz, double* waist, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- ABCD matrices of every configuration of a sweep (OpticalTable.calculate_abcd_matrix, optical_table.py:239-297) --
 * For K configurations whose monitor mon0 and everything in front of it are the same, the three bundles of the finite
 * differences are the same in every configuration, so two sweep traces over one sweep scene give every configuration's
 * matrices:
 *   sweep A: 2N rays, the nominal rays r (roots k * 2N + r) and the same rays shifted by disp along mon0's tangent_Y
 *            (roots k * 2N + N + r);
 *   sweep B: N rays, the shifted rays turned by rot about mon0's tangent_Z through their pivots (roots k * N + r).
 * optb_sweep_abcd_pivots reads sweep A's rows of mon0: pivots[r][3] = configuration 0's nominal mon0 hit point of ray r
 * (monitor-local, the reference's pivot; NaN when that ray has no single row), and first_bad = the smallest k * N + r
 * whose nominal ray has not exactly one mon0 row or whose hit point differs in any bit from configuration 0's, else -1.
 * A caller builds sweep B only when first_bad is -1.
 * optb_sweep_abcd reads both sweeps' rows of mon1 and writes, for configuration k and ray r,
 *   abcd[k][r][4] = A, B, C, D = (y1 - y0) / disp, (y2 - y0) / rot, (t1 - t0) / disp, (t2 - t0) / rot
 * with y = local point . tangent_Y and t = lab direction . tangent_Y in frames[k] (DEVICE optb_monitor_frame[K], the
 * per-row values optb_monitor_stats_grouped writes, bit for bit) for the nominal (0), shifted (1) and turned (2) ray,
 * and counts[k][r][3] = that ray's mon1 rows in each of the three traces. A matrix is NaN unless all three counts are 1.
 *   - rows: DEVICE columns (root: hit_root or hit_key; monitor: hit_monitor or hit_key; hit_px/py/pz; for
 *     optb_sweep_abcd also hit_dx/dy/dz), in any order: a slot per (trace, k, r) counts its rows and is read only when
 *     it holds exactly one, so equal rows give equal bits in any order and on every call.
 *   - pivots, first_bad, abcd, counts: DEVICE memory; workspace: optb_sweep_abcd_workspace_bytes(N, K) bytes of device
 *     memory (-1: N < 1, K < 1 or 2 K N >= 2^32), enough for either call.
 * Fails with -7 when a column is missing, the monitor index is outside [0, 256), 2 K N >= 2^32, a row count is >= 2^31 - 1
 * or the workspace is too small. Enqueued on `stream`, without a host synchronisation. Added without a change of
 * OPTB_ABI_VERSION: no struct changed.                                                                               */
int64_t optb_sweep_abcd_workspace_bytes(int64_t n_rays, int32_t n_configs);
int optb_sweep_abcd_pivots(optb_ctx* ctx, const optb_result* rows, int64_t n, int64_t n_rays, int32_t n_configs,
                           int32_t mon0, double* pivots, int64_t* first_bad, void* workspace, int64_t workspace_bytes,
                           void* stream);
int optb_sweep_abcd(optb_ctx* ctx, const optb_result* rows_a, int64_t n_a, const optb_result* rows_b, int64_t n_b,
                    int64_t n_rays, int32_t n_configs, int32_t mon1, const optb_monitor_frame* frames, double disp,
                    double rot, double* abcd, int32_t* counts, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- multi-GPU monitor merge (SURVEY 8e) -----------------------------------------------------------------------
 * The path shards without a data-path collective: every rank (one process per GPU, one ctx each) traces its own block
 * of the initial rays against its own copy of the scene. The only exchange is the merge of the monitors at the end,
 * which the reference -- single process -- gets for free from Monitor.record appending to one list (monitor.py:183-193):
 * an all-reduce (sum) of the histograms and counters over NCCL. Python hosts use torch.distributed
 * (optable_b200/dist.py); these entry points give a C host the same thing. NCCL is loaded at run time (dlopen of
 * $OPTB_NCCL_LIB, else the libnccl.so.2 already in the process or on the loader path): the library has no link-time
 * dependency on it.
 *   optb_comm_unique_id   rank 0: fills the 128-byte ncclUniqueId to hand to the other ranks (any transport)
 *   optb_comm_init        all ranks: joins the communicator (collective call)
 *   optb_monitor_merge    all ranks: in-place sum over ranks of hist_y [n_monitors][30], hist_yz [n_monitors][30][30]
 *                         and counters [OPTB_C_COUNT] (device pointers; any may be NULL; the status word is OR-ed,
 *                         OPTB_C_GENERATIONS takes the maximum), enqueued on `stream`. The histograms of a sweep
 *                         scene are contiguous [K][n_monitors][...]: pass n_monitors = K * n_monitors
 *   optb_comm_destroy     leaves the communicator                                                                  */
int optb_comm_unique_id(optb_ctx* ctx, void* id128);
int optb_comm_init(optb_ctx* ctx, const void* id128, int rank, int nranks);
int optb_monitor_merge(optb_ctx* ctx, int64_t* hist_y, int64_t* hist_yz, int n_monitors, int64_t* counters, void* stream);
int optb_comm_destroy(optb_ctx* ctx);

/* Device micro-benchmarks used for the roofline denominators: returns achieved FP64 FMA
 * TFLOP/s (dfma) measured with CUDA events.                                            */
int optb_measure_fp64_peak(optb_ctx* ctx, double* tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* OPTB_H */
