// optb.cu -- C-ABI CUDA library (include/optb.h) for the optable bounce loop on B200 (sm_100a).
//
// Kernels:
//   trace_kernel      whole bounce loop. One thread owns one ray of the current wavefront; warps pull 32-ray
//                     chunks from a global work counter (persistent grid). The scene tables are staged into
//                     shared memory with a TMA bulk copy (cp.async.bulk + mbarrier). A root whose alive set
//                     is a single ray keeps bouncing in registers (closest hit -> physics -> monitors ->
//                     next bounce); split interactions park their children in a sparse slot pair.
//   tile_sums/scan_sums/slots     ordered, index-only stream compaction: the list of occupied child slots in
//                     reference BFS order (which the pop cap of optical_table.py:86-97 needs); rays are not moved.
//   mark_kernel       first/last wavefront index of every root (rank of a ray inside its root's generation).
//   sort_prep + cub radix sort    processing order of a generation by coherence key (storage order stays BFS).
// Segments and monitor rows are appended with warp-aggregated atomics and carry their (root, pop) key.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <stddef.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <new>
#include <vector>

#include "optb_device.cuh"
#include "optb_flags.cuh"

using namespace optb;

namespace {

constexpr int kBlock = 128;  // trace_kernel threads per CTA
constexpr int kTile = 2048;  // children-scan tile (entries per block)
constexpr int kScanBlock = 256;
constexpr int kRayF64 = 13;

// Ray storage in the workspace (wavefront W and sparse children C): one 128-byte record per ray. The wavefront is read
// through two indirections (coherence order -> dense BFS index -> sparse slot), i.e. by gathers: with a record per ray a
// gather touches exactly four full 32-byte sectors, where one column per field touched seventeen sectors for the same
// 128 bytes (measured on the ripa scene: 7.5 GB of DRAM reads in one 2.4 ms generation). The caller-facing ray batch
// stays SoA (optb_rays): it is read once, in order, fully coalesced.
struct __align__(16) RayRec {
  double ox, oy, oz, dx, dy, dz, I, wl, qre, qim, pl, n, len;
  uint32_t flags, root, pop;  // pop: pop number of the first ray of this root's generation (the ray's own = pop + rank)
  int32_t family;
  uint32_t rank, gcount;      // rank of the ray inside its root's generation / size of that generation (rank_kernel)
};
static_assert(sizeof(RayRec) == 128, "RayRec must be four sectors");
struct RayBuf {
  RayRec* rec;
  // Dense side arrays, one entry per record slot. The wavefront bookkeeping between two generations (mark, rank,
  // sort_prep) reads and writes ONLY these: 8 bytes per slot, visited in slot order, instead of one 32-byte sector of
  // every 128-byte record (ripa: 23.8 -> 21.7 ms per 1e6 rays).
  uint2* key;  // written with the child: x = coherence key (leaf it left) * 2 + child index, y = root
  uint2* rk;   // written by rank_kernel: x = rank of the ray inside its root's generation, y = size of that generation
};

struct Header {  // first bytes of the workspace
  unsigned int work_ctr;
  unsigned int n_next;      // size of the wavefront the last compaction produced
  unsigned int n_prev;      // size of the wavefront that compaction consumed (for generations launched unseen)
  unsigned int empty_gens;  // generations launched unseen that found nothing to do
  unsigned int pad[12];
};

struct SceneOff { uint32_t trav, nf, ni, matk, matf, mon, aux; };

struct TraceArgs {
  const unsigned char* blob; uint32_t blob_bytes; SceneOff off; int n_nodes, n_mons;
  // input wavefront: either the caller's rays (gen0) or the workspace wavefront
  optb_rays in0; RayBuf w; int gen0;
  int hist_mons;       // SWEEP kernels: histograms this launch accumulates (n_configs * n_mons)
  long long n_in; const unsigned int* n_in_dev;  // n_in_dev overrides when non-null
  const uint32_t* gen_first; const uint32_t* gen_last;
  const uint32_t* perm;  // processing order of the wavefront (sorted by coherence key), or null
  const uint32_t* slot;  // wavefront index (reference order, dense) -> slot of the ray in the sparse buffer `w`
  // split output
  RayBuf c; uint8_t* nchild;
  // params
  long long max_trace; double unit; int rec_seg, rec_hit, rec_hist, chain_len, n_families, fam_shared;
  int hist_smem;
  optb_result out;
  unsigned long long* counters;
  Header* hdr;
  // family-serial mode (scenes with interact caps): one thread owns one Ray._id family and replays the
  // reference's sequential order; w is then a per-family FIFO ring of qcap entries
  const uint32_t* fam_off; uint32_t* fam_roots; uint32_t qcap;
  uint32_t root_base;  // global index of ray 0 of this launch (chunked host traces)
  int has_boxes;       // some node carries a lab-box test
  uint32_t sweep_n;    // SWEEP kernels: rays per configuration (root k * sweep_n + r = ray r in configuration k);
                       // blob_bytes is then the stride between the configurations' blobs
};

OPTB_DEV uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

OPTB_DEV void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
OPTB_DEV void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
OPTB_DEV void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
OPTB_DEV void mbar_wait(unsigned long long* bar, uint32_t phase) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(phase) : "memory");
}

OPTB_DEV unsigned long long warp_alloc(unsigned long long* ctr) {
  unsigned m = __activemask();
  int lane = threadIdx.x & 31;
  int leader = __ffs(m) - 1;
  unsigned long long base = 0;
  if (lane == leader) base = atomicAdd(ctr, (unsigned long long)__popc(m));
  base = __shfl_sync(m, base, leader);
  return base + __popc(m & ((1u << lane) - 1u));
}

// SERIAL (with SWEEP): the family-serial sweep numbers the families itself, so the family column is not read here
template <bool SWEEP = false, bool SERIAL = false>
OPTB_DEV void load_ray(const TraceArgs& a, long long i, Ray& r, bool& solo, uint32_t& gcount, uint32_t& pop_base) {
  if (a.gen0) {
    const optb_rays& s = a.in0;
    const uint32_t bc = s.broadcast;
    // a sweep traces the one bundle through every configuration: root i reads input ray i % N
    const long long in = SWEEP ? i % a.sweep_n : i;
#define OPTB_COL(ptr, bit) ((ptr)[((bc >> (bit)) & 1u) ? 0 : in])
    r.ox = OPTB_COL(s.ox, 0); r.oy = OPTB_COL(s.oy, 1); r.oz = OPTB_COL(s.oz, 2);
    r.dx = OPTB_COL(s.dx, 3); r.dy = OPTB_COL(s.dy, 4); r.dz = OPTB_COL(s.dz, 5);
    r.I = OPTB_COL(s.intensity, 6); r.wl = OPTB_COL(s.wavelength, 7);
    r.qre = OPTB_COL(s.q_re, 8); r.qim = OPTB_COL(s.q_im, 9);
    r.pl = OPTB_COL(s.pathlength, 10); r.n = OPTB_COL(s.n_medium, 11);
    r.len = s.length ? OPTB_COL(s.length, 12) : INFINITY;
#undef OPTB_COL
    r.flags = s.flags ? s.flags[in] : (OPTB_RF_ALIVE | OPTB_RF_HASQ);
    r.root = (uint32_t)i + a.root_base; r.pop = 0;
    if constexpr (!(SWEEP && SERIAL)) r.family = s.family ? s.family[i] : (int32_t)r.root;
    solo = true; gcount = 1; pop_base = 0;
  } else {
    // Children stay where the previous generation's kernel wrote them (slot 2*parent + k of the sparse buffer);
    // `slot` lists the occupied slots in reference order, so nothing is copied between generations.
    const uint32_t sl = a.slot[i];
    const uint2 rg = a.w.rk[sl];         // issued together with the record's loads (neither depends on the other)
    const RayRec q = a.w.rec[sl];        // eight 16-byte loads of one contiguous record
    r.ox = q.ox; r.oy = q.oy; r.oz = q.oz; r.dx = q.dx; r.dy = q.dy; r.dz = q.dz;
    r.I = q.I; r.wl = q.wl; r.qre = q.qre; r.qim = q.qim; r.pl = q.pl; r.n = q.n; r.len = q.len;
    r.flags = q.flags; r.root = q.root; r.family = q.family;
    gcount = rg.y;
    solo = (gcount == 1);
    pop_base = q.pop;
    r.pop = q.pop + rg.x;  // pop_base of this generation + rank inside the root
  }
}

OPTB_DEV void store_child(const RayBuf& c, long long j, const Ray& parent, double ox, double oy, double oz, double pl,
                           double dx, double dy, double dz, double I, double qre, double qim, double nmed, int k,
                           uint32_t pop_base, int leaf) {
  RayRec q;
  q.ox = ox; q.oy = oy; q.oz = oz; q.dx = dx; q.dy = dy; q.dz = dz;
  q.I = I; q.wl = parent.wl; q.qre = qre; q.qim = qim; q.pl = pl; q.n = nmed; q.len = parent.len;
  q.flags = parent.flags; q.root = parent.root; q.pop = pop_base; q.family = parent.family;
  q.rank = 0u; q.gcount = 1u;  // (unused by the wavefront: rank and generation size live in RayBuf::rk)
  c.rec[j] = q;                 // eight 16-byte stores: four full sectors
  c.key[j] = make_uint2(((uint32_t)leaf << 1) | (uint32_t)k, parent.root);
}

OPTB_DEV void ring_put(const RayBuf& w, long long j, const Ray& r) {
  RayRec q;
  q.ox = r.ox; q.oy = r.oy; q.oz = r.oz; q.dx = r.dx; q.dy = r.dy; q.dz = r.dz;
  q.I = r.I; q.wl = r.wl; q.qre = r.qre; q.qim = r.qim; q.pl = r.pl; q.n = r.n; q.len = r.len;
  q.flags = r.flags; q.root = r.root; q.pop = r.pop; q.family = r.family; q.rank = 0u; q.gcount = 1u;
  w.rec[j] = q;
}
OPTB_DEV void ring_get(const RayBuf& w, long long j, Ray& r) {
  const RayRec q = w.rec[j];
  r.ox = q.ox; r.oy = q.oy; r.oz = q.oz; r.dx = q.dx; r.dy = q.dy; r.dz = q.dz;
  r.I = q.I; r.wl = q.wl; r.qre = q.qre; r.qim = q.qim; r.pl = q.pl; r.n = q.n; r.len = q.len;
  r.flags = q.flags;
}

// The tables of one configuration of a sweep scene (configuration blobs back to back at stride a.blob_bytes).
OPTB_DEV void sweep_view(const TraceArgs& a, uint32_t root, SceneView& sv) {
  const unsigned char* base = a.blob + (size_t)(root / a.sweep_n) * a.blob_bytes;
  sv.trav = (const double*)(base + a.off.trav);
  sv.nf = (const double*)(base + a.off.nf);
  sv.ni = (const int32_t*)(base + a.off.ni);
  sv.matk = (const int32_t*)(base + a.off.matk);
  sv.matf = (const double*)(base + a.off.matf);
  sv.mon = (const double*)(base + a.off.mon);
  sv.aux = (const double*)(base + a.off.aux);
}

// One pop's dead segment: append to the segment log and test it against every monitor (monitor.py:183-193).
template <bool SWEEP = false>
OPTB_DEV void emit_segment(const TraceArgs& a, const SceneView& sv, const Ray& r, double seg_len, uint32_t seg_flags,
                           int leaf, unsigned int* s_hist, unsigned int& n_hits_local) {
  if (a.rec_seg) {
    unsigned long long j = warp_alloc(&a.counters[OPTB_C_SEGMENTS]);
    if (j < (unsigned long long)a.out.seg_capacity) {
      const optb_result& o = a.out;
      o.seg_ox[j] = r.ox; o.seg_oy[j] = r.oy; o.seg_oz[j] = r.oz;
      o.seg_dx[j] = r.dx; o.seg_dy[j] = r.dy; o.seg_dz[j] = r.dz;
      o.seg_length[j] = seg_len; o.seg_intensity[j] = r.I; o.seg_wavelength[j] = r.wl;
      o.seg_q_re[j] = r.qre; o.seg_q_im[j] = r.qim; o.seg_pathlength[j] = r.pl; o.seg_n[j] = r.n;
      o.seg_flags[j] = seg_flags; o.seg_root[j] = r.root; o.seg_pop[j] = r.pop; o.seg_leaf[j] = leaf;
    } else {
      atomicOr(&a.counters[OPTB_C_STATUS], (unsigned long long)OPTB_ST_SEG_OVERFLOW);
    }
  }
  for (int m = 0; m < sv.n_mons; m++) {
    const double* mf = sv.mon + m * kMonBlobStride;
    // Monitor.record (monitor.py:183-193) = to-local + planar hit with t <= length, in stages like intersect_planar:
    // the x row of Tinv decides "in front, not parallel" and (orthonormal frame) gives t; most segments end here
    const double* c = mf + OPTB_MON_ORIGIN;
    const double* Ti = mf + OPTB_MON_TINV;
    const double vx = r.ox - c[0], vy = r.oy - c[1], vz = r.oz - c[2];
    const double ox = dot3(Ti[0], Ti[1], Ti[2], vx, vy, vz);
    double dx = dot3(Ti[0], Ti[1], Ti[2], r.dx, r.dy, r.dz);
    if (!((ox < 0.0 && dx > 0.0) || (ox > 0.0 && dx < 0.0))) continue;  // t = -ox/dx >= 1e-9 needs opposite signs
    double dy, dz;
    const bool ortho = mf[OPTB_MON_ORTHO] != 0.0;
    if (!ortho) {
      dy = dot3(Ti[3], Ti[4], Ti[5], r.dx, r.dy, r.dz);
      dz = dot3(Ti[6], Ti[7], Ti[8], r.dx, r.dy, r.dz);
      const double rn = rsqrt(dot3(dx, dy, dz, dx, dy, dz));
      dx *= rn; dy *= rn; dz *= rn;
    }
    const double t = -ox / dx;
    if (!(t >= 1e-9) || t > seg_len) continue;
    if (ortho) {
      dy = dot3(Ti[3], Ti[4], Ti[5], r.dx, r.dy, r.dz);
      dz = dot3(Ti[6], Ti[7], Ti[8], r.dx, r.dy, r.dz);
    }
    const double oy = dot3(Ti[3], Ti[4], Ti[5], vx, vy, vz);
    const double oz = dot3(Ti[6], Ti[7], Ti[8], vx, vy, vz);
    const double Px = fma(t, dx, ox), Py = fma(t, dy, oy), Pz = fma(t, dz, oz);
    if (!(fabs(Py) <= mf[OPTB_MON_HW] && fabs(Pz) <= mf[OPTB_MON_HH])) continue;
    if (a.rec_hist) {
      const int hm = SWEEP ? (int)(r.root / a.sweep_n) * sv.n_mons + m : m;  // sweeps: histograms [config][monitor]
      double y = dot3(Px, Py, Pz, mf[OPTB_MON_TY], mf[OPTB_MON_TY + 1], mf[OPTB_MON_TY + 2]);
      double z = dot3(Px, Py, Pz, mf[OPTB_MON_TZ], mf[OPTB_MON_TZ + 1], mf[OPTB_MON_TZ + 2]);
      int by = hist_bin(y, -mf[OPTB_MON_HW], mf[OPTB_MON_HW], mf[OPTB_MON_STRIDE], mf[OPTB_MON_STRIDE + 1]);
      int bz = hist_bin(z, -mf[OPTB_MON_HH], mf[OPTB_MON_HH], mf[OPTB_MON_STRIDE + 2], mf[OPTB_MON_STRIDE + 3]);
      const int per = OPTB_HIST_BINS * (OPTB_HIST_BINS + 1);
      if (by >= 0) {
        if (a.hist_smem) {
          atomicAdd(&s_hist[hm * per + by], 1u);
          if (bz >= 0) atomicAdd(&s_hist[hm * per + OPTB_HIST_BINS + by * OPTB_HIST_BINS + bz], 1u);
        } else {
          atomicAdd((unsigned long long*)&a.out.hist_y[hm * OPTB_HIST_BINS + by], 1ull);
          if (bz >= 0)
            atomicAdd((unsigned long long*)&a.out.hist_yz[(hm * OPTB_HIST_BINS + by) * OPTB_HIST_BINS + bz], 1ull);
        }
      }
    }
    if (a.rec_hit) {
      unsigned long long j = warp_alloc(&a.counters[OPTB_C_HITS]);
      if (j < (unsigned long long)a.out.hit_capacity) {
        const optb_result& o = a.out;
        if (o.hit_monitor) o.hit_monitor[j] = m;
        if (o.hit_key) o.hit_key[j] = ((unsigned long long)r.root << 32) | ((unsigned long long)m << 24) | (unsigned long long)r.pop;
        if (o.hit_root) o.hit_root[j] = r.root;
        if (o.hit_pop) o.hit_pop[j] = r.pop;
        if (o.hit_px) o.hit_px[j] = Px;
        if (o.hit_py) o.hit_py[j] = Py;
        if (o.hit_pz) o.hit_pz[j] = Pz;
        if (o.hit_intensity) o.hit_intensity[j] = r.I;
        if (o.hit_t) o.hit_t[j] = t;
        if (o.hit_dx) o.hit_dx[j] = r.dx;
        if (o.hit_dy) o.hit_dy[j] = r.dy;
        if (o.hit_dz) o.hit_dz[j] = r.dz;
        if (o.hit_q_re) o.hit_q_re[j] = r.qre;
        if (o.hit_q_im) o.hit_q_im[j] = r.qim;
      } else {
        atomicOr(&a.counters[OPTB_C_STATUS], (unsigned long long)OPTB_ST_HIT_OVERFLOW);
      }
    } else {
      n_hits_local++;
    }
  }
}

// Closest hit over the flattened tree (optical_table.py:119-123 + component_group.py:93-122): smallest t, ties to
// the smallest pre-order index. Leaves are visited in pre-order except that aspheres (a 10-sample scan plus an
// iterative root solve each) are parked and tested last, when the closest cheap hit is known: a parked asphere
// whose bracket starts beyond that hit is dismissed without evaluating its profile once. The (t, index) ordering
// makes the result independent of the visiting order.
template <bool ASPH, bool BRENT = false>
struct HitSearch {
  const TraceArgs& a; const SceneView& sv; const Ray& ray; bool solo;
  double best_t; int best_node; unsigned int* cnt;  // cnt: this thread's {leaf tests, curved tests, box tests} in smem

  OPTB_DEV void test_leaf(int i, const int32_t* __restrict__ ni, const double* __restrict__ nf) {
    atomicAdd(cnt, 1u);  // shared-memory add without a result: one instruction, no register held across the search
    const int slot = ni[OPTB_NI_CAPSLOT];
    // a capped surface counts every geometric hit, closest or not (optical_component.py:359-362): no early exit
    const double t_beat = slot >= 0 ? INFINITY : best_t;
    double t;
    if (is_planar_kind(ni[OPTB_NI_GEOM])) {
      t = intersect_planar(sv, ni, nf, ray, t_beat);
    } else {
      atomicAdd(cnt + kBlock, 1u);
      double ox, oy, oz, dx, dy, dz;
      to_local(nf + OPTB_NF_ORIGIN, nf + OPTB_NF_TINV, ray, ni[OPTB_NI_ORTHO] != 0, ox, oy, oz, dx, dy, dz);
      t = intersect_leaf<ASPH, BRENT>(sv, ni, nf, ox, oy, oz, dx, dy, dz, ray.len, t_beat);
    }
    if (!(t >= 0.0)) return;
    if (slot >= 0) {  // should_interact / increase_interact_count :136-149
      int32_t* cnt = a.out.cap_counts + (long long)slot * a.n_families + ray.family;
      int old = atomicAdd(cnt, 1);
      if (!((double)old < nf[OPTB_NF_CAPMAX])) {
        atomicSub(cnt, 1);
        if (!solo || a.fam_shared) atomicOr(&a.counters[OPTB_C_STATUS], (unsigned long long)OPTB_ST_CAP_ORDER);
        return;
      }
    }
    if (t < best_t || (t == best_t && i < best_node)) { best_t = t; best_node = i; }
  }
};

// Lattice window of a ray in an OPTB_G_GRID group (descriptor layout: include/optb.h OPTB_GRID_*): index ranges
// [i0, i1] x [j0, j1] of the children whose lab box the ray can touch. False = no cheap window (ray nearly in the
// lattice plane, or more than 64 cells): the caller descends the group's box hierarchy instead.
OPTB_DEV bool grid_window(const double* __restrict__ gd, const Ray& r, int& i0, int& i1, int& j0, int& j1) {
  const double R = gd[OPTB_GRID_R];
  const double px = r.ox - gd[OPTB_GRID_C00], py = r.oy - gd[OPTB_GRID_C00 + 1], pz = r.oz - gd[OPTB_GRID_C00 + 2];
  const double w0 = dot3(px, py, pz, gd[OPTB_GRID_NHAT], gd[OPTB_GRID_NHAT + 1], gd[OPTB_GRID_NHAT + 2]);
  const double wd = dot3(r.dx, r.dy, r.dz, gd[OPTB_GRID_NHAT], gd[OPTB_GRID_NHAT + 1], gd[OPTB_GRID_NHAT + 2]);
  if (!(fabs(wd) >= 1e-3)) return false;
  // |w0 + t wd| <= R, t >= 0
  const double inv = 1.0 / wd;
  double ta = (-R - w0) * inv, tb = (R - w0) * inv;
  if (ta > tb) { const double x = ta; ta = tb; tb = x; }
  i0 = j0 = 0; i1 = j1 = -1;
  if (!(tb >= 0.0)) return true;  // the lattice slab lies behind the ray: no lattice child can pass its box test
  ta = fmax(ta, 0.0);
  const double a0 = dot3(px, py, pz, gd[OPTB_GRID_UD], gd[OPTB_GRID_UD + 1], gd[OPTB_GRID_UD + 2]);
  const double ad = dot3(r.dx, r.dy, r.dz, gd[OPTB_GRID_UD], gd[OPTB_GRID_UD + 1], gd[OPTB_GRID_UD + 2]);
  const double b0 = dot3(px, py, pz, gd[OPTB_GRID_VD], gd[OPTB_GRID_VD + 1], gd[OPTB_GRID_VD + 2]);
  const double bd = dot3(r.dx, r.dy, r.dz, gd[OPTB_GRID_VD], gd[OPTB_GRID_VD + 1], gd[OPTB_GRID_VD + 2]);
  const double a1 = fma(ta, ad, a0), a2 = fma(tb, ad, a0), b1 = fma(ta, bd, b0), b2 = fma(tb, bd, b0);
  const double no = gd[OPTB_GRID_NOUTER] - 1.0, ni = gd[OPTB_GRID_NINNER] - 1.0;
  const double alo = ceil(fmin(a1, a2) - gd[OPTB_GRID_RHOA]), ahi = floor(fmax(a1, a2) + gd[OPTB_GRID_RHOA]);
  const double blo = ceil(fmin(b1, b2) - gd[OPTB_GRID_RHOB]), bhi = floor(fmax(b1, b2) + gd[OPTB_GRID_RHOB]);
  if (!(alo <= ahi && blo <= bhi)) return alo == alo && ahi == ahi && blo == blo && bhi == bhi;  // empty (NaN: no window)
  if (ahi < 0.0 || alo > no || bhi < 0.0 || blo > ni) return true;  // window beside the lattice
  i0 = (int)fmax(alo, 0.0); i1 = (int)fmin(ahi, no);
  j0 = (int)fmax(blo, 0.0); j1 = (int)fmin(bhi, ni);
  if ((i1 - i0 + 1) * (j1 - j0 + 1) > 64) { i1 = j1 = -1; return false; }
  return true;
}

// BOXES: 0 = the scene has no lab-box test at all (top-level leaves only, SURVEY A.3);
//        1 = pre-order walk, a failed box test skips the subtree (component_group.py:98-115 as a forward scan);
//        2 = the same walk, and groups whose children form a regular lattice (OPTB_G_GRID: MMA / MLA / DMD arrays)
//            hand the walk the few children inside the ray's lattice window instead of a descent through their
//            box hierarchy; each candidate still has to pass the reference's own test of its own box.
template <int BOXES, bool ASPH, bool BRENT = false, bool VOTE = true>
OPTB_DEV void closest_hit(const TraceArgs& a, const SceneView& sv, const Ray& ray, bool solo,
                          double& best_t, int& best_node, unsigned int* cnt) {
  best_t = INFINITY; best_node = -1;
  const bool no_work = !(ray.flags & OPTB_RF_ALIVE);  // optical_component.py:349-350: a dead ray hits nothing
  HitSearch<ASPH, BRENT> hs{a, sv, ray, solo, INFINITY, -1, cnt};
  if constexpr (BOXES == 0 && !ASPH) {
    // No node carries a box test, so there is no group (groups always do): every node is a top-level leaf, and without
    // aspheres nothing is parked. The walk is a plain loop (c4: 687 -> ~600 warp instructions per pop).
    if (!no_work) {
      const int n = sv.n_nodes;
      // (one counter add per pop instead of one per leaf measured SLOWER on c4, 110.7 -> 113.6 ms: code layout)
#pragma unroll 1
      for (int i = 0; i < n; i++) hs.test_leaf(i, sv.ni + i * OPTB_NI_STRIDE, sv.nf + i * OPTB_NF_STRIDE);
    }
    best_t = hs.best_t; best_node = hs.best_node;
    return;
  }
  // Boxes the upload marked cullable are tested with front-to-back dismissal (slab_hit_far), in the walk and before a
  // parked test.
  unsigned int n_box = 0;
  constexpr int kPark = 4;
  int parked[kPark];
  int n_parked = 0, n_done = 0;
  int i = 0;
  const int n = sv.n_nodes;
  // BOXES = 0: a scene of top-level leaves only has no box test at all (and pays no reciprocals for one)
  const BoxRay br(ray.ox, ray.oy, ray.oz, BOXES ? ray.dx : 1.0, BOXES ? ray.dy : 1.0, BOXES ? ray.dz : 1.0);
  // lattice cursor (BOXES = 2): group being listed (-1: none), cell cursor, window, cursor over the extra children
  int g_node = -1, g_i = 0, g_j = 0, g_i1 = -1, g_j0 = 0, g_j1 = -1, g_x = 0;
  unsigned long long g_mask = 0ull;  // window cells whose box test passed and that are still to be visited
  const double* gd = nullptr;
  // Warp-synchronous "walk, then test": in every round each lane walks boxes until it holds a leaf (or runs out of
  // nodes and takes a parked asphere), then the lanes that called in together meet again at the vote and run the
  // one, long leaf test side by side. Without the explicit vote the compiler is free to fold the test into the
  // walk loop, and lanes that reach their leaves at different box counts then execute it one after another
  // (measured: 3x on the 7,689-leaf scene). One test_leaf call site also keeps the kernel's code size down.
  const unsigned group = __activemask();
  bool searching = !no_work;
  // (scenes without box tests yield a leaf per walk step: all lanes are in lock-step anyway, no vote needed)
  // VOTE = false (scenes staged in shared memory: a few dozen nodes, mostly coherent bundles): no vote either
  while ((BOXES && VOTE) ? __any_sync(group, searching) : searching) {
    int leaf = -1;
    if (searching) {
      while (true) {
        if (BOXES == 2 && g_node >= 0) {
          // next candidate child of the lattice group: window cells in list order, then the off-lattice children
          int cand;
          if (g_mask) {
            // (batched window: the boxes of all window cells were tested when the window was set up)
            const int b = __ffsll((long long)g_mask) - 1;
            g_mask &= g_mask - 1ull;
            cand = (int)gd[OPTB_GRID_CELLS + (g_i + (b >> 3)) * (int)gd[OPTB_GRID_NINNER] + g_j0 + (b & 7)];
            if ((*reinterpret_cast<const int*>(sv.trav + cand * 8 + 7) & 2) && hs.best_t < INFINITY &&
                slab_far_only(br, sv.trav + cand * 8, hs.best_t)) continue;
            leaf = cand;
            break;
          }
          if (g_i <= g_i1) {
            cand = (int)gd[OPTB_GRID_CELLS + g_i * (int)gd[OPTB_GRID_NINNER] + g_j];
            if (++g_j > g_j1) { g_j = g_j0; g_i++; }
          } else if (g_x < (int)gd[OPTB_GRID_NEXT]) {
            cand = (int)gd[OPTB_GRID_CELLS + (int)gd[OPTB_GRID_NOUTER] * (int)gd[OPTB_GRID_NINNER] + g_x];
            g_x++;
          } else {  // done: leave the group's subtree
            i = reinterpret_cast<const int2*>(sv.trav + g_node * 8 + 6)->y;
            g_node = -1;
            continue;
          }
          n_box++;
          if (*reinterpret_cast<const int*>(sv.trav + cand * 8 + 7) & 2) {
            if (slab_hit_far(br, sv.trav + cand * 8, hs.best_t) != 1) continue;
          } else if (!slab_hit(br, sv.trav + cand * 8)) continue;  // the child's own lab box (component_group.py:104-107)
          leaf = cand;  // (lattice children are leaves without interact caps, never aspheres to park: flatten._grid)
          break;
        }
        if (i >= n) break;
        const double* tv = sv.trav + i * 8;
        const int2 gs = *reinterpret_cast<const int2*>(tv + 6);  // {geometry kind, skip}
        if (BOXES) {
          const int word = *reinterpret_cast<const int*>(tv + 7);  // bit 0: test the box; bit 1: may dismiss by distance
          if (word) {
            n_box++;
            if (word & 2) {
              // front to back: a cullable box entered beyond the closest hit so far cannot hold the winner
              if (slab_hit_far(br, tv, hs.best_t) != 1) { i = gs.y; continue; }
            } else if (!slab_hit(br, tv)) { i = gs.y; continue; }
          }
        }
        const int g = gs.x;
        const int cur = i++;
        if (BOXES == 2 && g == OPTB_G_GRID && !br.any_par) {
          gd = sv.aux + sv.ni[cur * OPTB_NI_STRIDE + OPTB_NI_AUX];
          int i0;
          if (grid_window(gd, ray, i0, g_i1, g_j0, g_j1)) {
            g_node = cur; g_i = i0; g_j = g_j0; g_x = 0;
            if (g_i1 - i0 < 8 && g_j1 - g_j0 < 8 && g_i1 >= i0 && g_j1 >= g_j0) {
              // The window's box tests as one batch, two at a time: they are independent (each child's own stored box,
              // component_group.py:104-107), and taken one by one each is a dependent chain of L2 round trips (cell
              // index -> box -> test -> branch; ripa 21.45 -> 21.19 ms per 1e6 rays). Bit (row * 8 + column) of g_mask
              // = that cell's box is hit; the walk then visits the set bits in list order and applies the front-to-back
              // dismissal when it gets to each.
              const int nin = (int)gd[OPTB_GRID_NINNER];
              const int total = (g_i1 - i0 + 1) * (g_j1 - g_j0 + 1);
              int ii = i0, jj = g_j0;
              unsigned long long m = 0ull;
#pragma unroll 1
              for (int c = 0; c < total; c += 2) {
                int ii2 = ii, jj2 = jj + 1;
                if (jj2 > g_j1) { jj2 = g_j0; ii2++; }
                const bool two = c + 1 < total;
                if (!two) { ii2 = ii; jj2 = jj; }
                const int ca = (int)gd[OPTB_GRID_CELLS + ii * nin + jj];
                const int cb = (int)gd[OPTB_GRID_CELLS + ii2 * nin + jj2];
                const bool ha = slab_hit(br, sv.trav + ca * 8);
                const bool hb = slab_hit(br, sv.trav + cb * 8);
                m |= (unsigned long long)(ha ? 1u : 0u) << ((ii - i0) * 8 + (jj - g_j0));
                m |= (unsigned long long)((hb && two) ? 1u : 0u) << ((ii2 - i0) * 8 + (jj2 - g_j0));
                jj = jj2 + 1; ii = ii2;
                if (jj > g_j1) { jj = g_j0; ii++; }
              }
              n_box += (unsigned int)total;
              g_mask = m;
              g_i1 = i0 - 1;  // the cell cursor below is spent: after the mask come the off-lattice children
            }
          }
          continue;  // (no window: fall through into the box hierarchy below this node)
        }
        if (g == OPTB_G_GROUP || g == OPTB_G_GRID) continue;
        if (ASPH && g == OPTB_G_ASPHERE && n_parked < kPark) {
#pragma unroll
          for (int k = 0; k < kPark; k++) if (k == n_parked) parked[k] = cur;
          n_parked++;
          continue;
        }
        leaf = cur;
        break;
      }
      if (leaf < 0) {
        if (n_done < n_parked) {
#pragma unroll
          for (int k = 0; k < kPark; k++) if (k == n_done) leaf = parked[k];
          n_done++;
          // parked while the closest cheap hit was not known yet: its box may be out of reach by now
          if (BOXES && (*reinterpret_cast<const int*>(sv.trav + leaf * 8 + 7) & 2) &&
              slab_hit_far(br, sv.trav + leaf * 8, hs.best_t) == 2) leaf = -1;
        } else {
          searching = false;
        }
      }
    }
    if (leaf >= 0) hs.test_leaf(leaf, sv.ni + leaf * OPTB_NI_STRIDE, sv.nf + leaf * OPTB_NF_STRIDE);
  }
  best_t = hs.best_t; best_node = hs.best_node;
  if (BOXES) atomicAdd(cnt + 2 * kBlock, n_box);
}

// SPLIT = some interaction of the scene can emit two rays (or the caller bounded the in-register chain): the
// wavefront machinery (child slots, per-root generation ranks) is compiled in. Scenes that cannot split run the
// whole life of a ray in registers with none of it.
// FLAG = diagnostics variant: the ambiguity mask of SURVEY A.9 is evaluated at every pop (optb_flags.cuh).
// BRENT = params.reference_roots: curved-surface roots from the reference's own brentq iteration (brentq_dev) instead
// of the closed-form / Newton root.
// PASSK = the scene has an OPTB_I_PASS leaf (a Monitor listed as a component): only the general variants carry that body.
// SWEEP = a sweep scene (optb_scene_upload_sweep): every lane reads the tables of its root's configuration from global
// memory (a warp may straddle configurations); the kernels of ordinary scenes do not carry it. With SERIAL, work item
// i is family i % F of configuration i / F (F = families per configuration), and all its roots read that configuration.
template <bool SMEM, bool SERIAL, int BOXES, bool ASPH, bool SPLIT, bool FLAG = false, bool BRENT = false, bool PASSK = false,
          bool SWEEP = false>
// Resident CTAs per SM: scenes staged in shared memory are bound by dependent fp64 chains and lose more to the
// spills of a tighter register budget than they gain from a fifth CTA (measured 6.32 -> 7.62 ms on c2); scenes
// whose tables stay in L1/L2 (thousands of leaves) are memory-latency bound and gain from it (ripa 30.6 -> 29.8 ms).
__global__ void __launch_bounds__(kBlock, (SMEM || ASPH || SERIAL) ? 4 : 5)
trace_kernel(const __grid_constant__ TraceArgs a) {
  constexpr int MAXCH = (SPLIT || SERIAL) ? 2 : 1;
  static_assert(!SWEEP || (!SMEM && !FLAG && !BRENT), "sweeps run from global memory, without the diagnostics modes");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long mbar;
  // The closest-hit search only needs a ray's geometry. Its radiometric state (intensity, wavelength, q, path
  // length, index: 12 registers) is parked here for the duration of the search so that the hot loop has them.
  __shared__ double s_park[6][kBlock];
  __shared__ double s_icn[3][kBlock];   // index memo: wavelength, n of slot 0, n of slot 1
  __shared__ int s_icm[2][kBlock];      // material index of slot 0 / slot 1
  __shared__ unsigned int s_cnt[3][kBlock];  // per thread: leaf tests, curved leaf tests, lab-box tests
  s_cnt[0][threadIdx.x] = 0u; s_cnt[1][threadIdx.x] = 0u; s_cnt[2][threadIdx.x] = 0u;
  unsigned int* const my_cnt = &s_cnt[0][threadIdx.x];
  s_icn[0][threadIdx.x] = -1.0; s_icm[0][threadIdx.x] = -1; s_icm[1][threadIdx.x] = -1;
  const IndexCache ic{&s_icn[0][threadIdx.x], &s_icn[1][threadIdx.x], &s_icn[2][threadIdx.x], &s_icm[0][threadIdx.x],
                      &s_icm[1][threadIdx.x]};
  const unsigned char* base = a.blob;
  if constexpr (SMEM) {
    // Stage the whole scene blob with TMA bulk copies; completion is signalled on the mbarrier.
    if (threadIdx.x == 0) mbar_init(&mbar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
      mbar_expect_tx(&mbar, a.blob_bytes);
      constexpr uint32_t kChunk = 32768;
      for (uint32_t off = 0; off < a.blob_bytes; off += kChunk)
        tma_bulk_g2s(smem_raw + off, a.blob + off, min(kChunk, a.blob_bytes - off), &mbar);
    }
    mbar_wait(&mbar, 0);
    base = smem_raw;
  }
  SceneView sv;
  sv.trav = (const double*)(base + a.off.trav);
  sv.nf = (const double*)(base + a.off.nf);
  sv.ni = (const int32_t*)(base + a.off.ni);
  sv.matk = (const int32_t*)(base + a.off.matk);
  sv.matf = (const double*)(base + a.off.matf);
  sv.mon = (const double*)(base + a.off.mon);
  sv.aux = (const double*)(base + a.off.aux);
  sv.n_nodes = a.n_nodes; sv.n_mons = a.n_mons;
  sv.status = &a.counters[OPTB_C_STATUS];

  const int per = OPTB_HIST_BINS * (OPTB_HIST_BINS + 1);
  unsigned int* s_hist = (unsigned int*)(smem_raw + (SMEM ? ((a.blob_bytes + 15u) & ~15u) : 0u));
  if (a.hist_smem) {
    for (int k = threadIdx.x; k < (SWEEP ? a.hist_mons : a.n_mons) * per; k += blockDim.x) s_hist[k] = 0u;
    __syncthreads();
  }

  const long long n_in = a.n_in_dev ? (long long)*a.n_in_dev : a.n_in;
  const int lane = threadIdx.x & 31;
  unsigned int c_pops = 0, c_inter = 0, c_drop = 0, c_hits = 0;  // per thread; widened when reduced

  while (true) {
    constexpr bool PHASE = !SERIAL && !FLAG && BOXES != 0 && !ASPH;
    // REFILL: a lane whose ray is finished (its chain ended, or it was a one-pop ray) takes the next ray from the work
    // counter at once instead of idling until the slowest of its warp's 32 rays is done. Chains of a splitting scene end
    // after very different numbers of pops (ripa generation 0: 23.8 of 32 lanes busy on average). The work counter of
    // these variants counts rays, not 32-ray chunks.
    constexpr bool REFILL = PHASE && SPLIT;
    unsigned int chunk = 0;
    if (lane == 0) chunk = atomicAdd(&a.hdr->work_ctr, REFILL ? 32u : 1u);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    long long i = (REFILL ? (long long)chunk : (long long)chunk * 32) + lane;
    // PHASE: the warps of a CTA start every pop together (one barrier per pop). The kernel's hot code (35-55 KB) is
    // larger than the 32 KB instruction cache; rays of one launch follow similar paths, so warps that start a pop
    // together run the same stretch of code at the same time and share the cache instead of thrashing it (ncu on the
    // ripa scene: 4.8 issue slots lost to instruction fetch per instruction issued). Used where it measured faster
    // (B200, r2n): scenes with a box walk and no aspheres -- lens groups of spheres (c3 -5 %), large arrays
    // (ripa -6 %); not for bare mirror scenes, whose pops are too short to pay for a barrier (c4 +17 %), nor for
    // asphere scenes (c2 +-0). A warp that ran out of rays keeps meeting the barrier until the whole CTA is done.
    const bool has = i < n_in;
    if (PHASE) { if (!__syncthreads_or(has ? 1 : 0)) break; }
    else {
      if ((long long)chunk * 32 >= n_in) break;
      if (!has) continue;
    }
    // Wavefront entries are stored in reference (BFS) order, which the pop numbering needs, but processed in the
    // order of their coherence key: rays that left the same surface the same way sit in the same warp.
    if (SPLIT && !SERIAL && a.perm && has) i = a.perm[i];

    if constexpr (SERIAL) {
      // Work item = one Ray._id family. Its initial rays are traced one after another in input order, each
      // with the reference's own FIFO loop (optical_table.py:74-147), so interact counts evolve exactly as
      // in the reference (optical_component.py:136-149, 359-362).
      const uint32_t lo = a.fam_off[i], hi = a.fam_off[i + 1];
      for (uint32_t x = lo + 1; x < hi; x++) {  // the scatter is unordered: restore input order
        uint32_t v = a.fam_roots[x]; uint32_t y = x;
        while (y > lo && a.fam_roots[y - 1] > v) { a.fam_roots[y] = a.fam_roots[y - 1]; y--; }
        a.fam_roots[y] = v;
      }
      if constexpr (SWEEP) { if (lo < hi) sweep_view(a, a.fam_roots[lo], sv); }
      const long long ring = (long long)i * a.qcap;
      for (uint32_t x = lo; x < hi; x++) {
        Ray ray; bool solo; uint32_t gcount, pop_base0;
        const uint32_t root = a.fam_roots[x];
        load_ray<SWEEP, true>(a, root, ray, solo, gcount, pop_base0);
        uint32_t head = 0, tail = 0, pops = 0;
        ring_put(a.w, ring, ray); tail = 1;
        while ((long long)pops < a.max_trace && head != tail) {
          ring_get(a.w, ring + head % a.qcap, ray); head++;
          ray.root = root; ray.family = (int32_t)i; ray.pop = pops++;
          double t; int node;
          closest_hit<BOXES, ASPH, BRENT>(a, sv, ray, true, t, node, my_cnt);
          c_pops++;
          const bool hit = node >= 0;
          const int32_t* ni = sv.ni + (hit ? node : 0) * OPTB_NI_STRIDE;
          const double* nf = sv.nf + (hit ? node : 0) * OPTB_NF_STRIDE;
          emit_segment<SWEEP>(a, sv, ray, hit ? t : ray.len, hit ? (ray.flags & ~OPTB_RF_ALIVE) : ray.flags,
                              hit ? ni[OPTB_NI_LEAF] : -1, s_hist, c_hits);
          if (!hit) continue;
          c_inter++;
          double ox, oy, oz, dx, dy, dz;
          to_local(nf + OPTB_NF_ORIGIN, nf + OPTB_NF_TINV, ray, ni[OPTB_NI_ORTHO] != 0, ox, oy, oz, dx, dy, dz);
          Children<MAXCH> ch;
          interact<ASPH, MAXCH, PASSK || SERIAL || FLAG || BRENT>(sv, ni, nf, ray, a.unit, ox, oy, oz, dx, dy, dz, t, ch, ic);
          for (int k = 0; k < ch.n; k++) {
            if (tail - head >= a.qcap) { atomicOr(&a.counters[OPTB_C_STATUS], (unsigned long long)OPTB_ST_WORK_OVERFLOW); break; }
            Ray c = ray;
            c.ox = ch.ox; c.oy = ch.oy; c.oz = ch.oz;
            const bool second = (k == 1);
            c.dx = second ? ch.dx[MAXCH - 1] : ch.dx[0]; c.dy = second ? ch.dy[MAXCH - 1] : ch.dy[0];
            c.dz = second ? ch.dz[MAXCH - 1] : ch.dz[0]; c.I = second ? ch.I[MAXCH - 1] : ch.I[0];
            c.qre = second ? ch.qre[MAXCH - 1] : ch.qre[0]; c.qim = second ? ch.qim[MAXCH - 1] : ch.qim[0];
            c.n = second ? ch.nmed[MAXCH - 1] : ch.nmed[0]; c.pl = ch.pl;
            ring_put(a.w, ring + tail % a.qcap, c); tail++;
          }
        }
        c_drop += tail - head;
      }
      continue;
    }

    Ray ray; bool solo = true; uint32_t gcount = 1, pop_base0 = 0;
    if (has) load_ray<SWEEP>(a, i, ray, solo, gcount, pop_base0);
    if constexpr (SWEEP) { if (has) sweep_view(a, ray.root, sv); }
    if (!SPLIT) solo = true;
    uint32_t pop_base_next = (!SPLIT || a.gen0) ? 0u : (pop_base0 + gcount);
    int nch = 0;
    int chained = 0;
    int hit_leaf = 0;
    Children<MAXCH> ch;
    ch.n = 0;
    // one pop of this lane's ray; true = its only child carries on in registers (chain)
    auto pop_step = [&]() -> bool {
      if ((long long)ray.pop >= a.max_trace) { c_drop++; nch = 0; return false; }  // queued but never popped
      double t; int node;
      // Only the asphere and lattice variants park: for the others it measured slower on B200 (c4 110.8 -> 115.0 ms,
      // c3 7.81 -> 8.00 ms).
      if constexpr (ASPH || BOXES == 2) {
        volatile double* pk = &s_park[0][threadIdx.x];
        pk[0 * kBlock] = ray.I; pk[1 * kBlock] = ray.wl; pk[2 * kBlock] = ray.qre;
        pk[3 * kBlock] = ray.qim; pk[4 * kBlock] = ray.pl; pk[5 * kBlock] = ray.n;
        closest_hit<BOXES, ASPH, BRENT, !SMEM>(a, sv, ray, solo, t, node, my_cnt);
        ray.I = pk[0 * kBlock]; ray.wl = pk[1 * kBlock]; ray.qre = pk[2 * kBlock];
        ray.qim = pk[3 * kBlock]; ray.pl = pk[4 * kBlock]; ray.n = pk[5 * kBlock];
      } else {
        closest_hit<BOXES, ASPH, BRENT, !SMEM>(a, sv, ray, solo, t, node, my_cnt);
      }
      c_pops++;
      if constexpr (FLAG) {
        const unsigned amb = flag_pop(sv, ray, node, t, a.unit);
        if (amb && a.out.root_flags) atomicOr(&a.out.root_flags[ray.root - a.root_base], amb);
      }
      // the pop's dead segment: the ray itself when nothing was hit (optical_table.py:132-134), else the
      // truncated copy with length = t, alive = False (optical_component.py:364)
      const bool hit = node >= 0;
      const int32_t* ni = sv.ni + (hit ? node : 0) * OPTB_NI_STRIDE;
      const double* nf = sv.nf + (hit ? node : 0) * OPTB_NF_STRIDE;
      emit_segment<SWEEP>(a, sv, ray, hit ? t : ray.len, hit ? (ray.flags & ~OPTB_RF_ALIVE) : ray.flags,
                          hit ? ni[OPTB_NI_LEAF] : -1, s_hist, c_hits);
      if (!hit) { nch = 0; return false; }
      c_inter++;
      hit_leaf = ni[OPTB_NI_LEAF];
      double ox, oy, oz, dx, dy, dz;
      to_local(nf + OPTB_NF_ORIGIN, nf + OPTB_NF_TINV, ray, ni[OPTB_NI_ORTHO] != 0, ox, oy, oz, dx, dy, dz);
      interact<ASPH, MAXCH, PASSK || SERIAL || FLAG || BRENT>(sv, ni, nf, ray, a.unit, ox, oy, oz, dx, dy, dz, t, ch, ic);
      nch = ch.n;
      if (nch == 1 && solo && (!SPLIT || a.chain_len == 0 || chained + 1 < a.chain_len)) {
        // the root's alive set is this one ray: BFS order is trivially kept, continue in registers
        ray.ox = ch.ox; ray.oy = ch.oy; ray.oz = ch.oz;
        ray.dx = ch.dx[0]; ray.dy = ch.dy[0]; ray.dz = ch.dz[0];
        ray.I = ch.I[0]; ray.qre = ch.qre[0]; ray.qim = ch.qim[0]; ray.pl = ch.pl; ray.n = ch.nmed[0];
        ray.pop++; chained++;
        return true;
      }
      return false;
    };
    // what a finished ray leaves behind: its children in slots 2i / 2i + 1 of the sparse buffer
    auto store_children = [&]() {
      a.nchild[i] = (uint8_t)nch;
      uint32_t pb = solo ? ray.pop + 1u : pop_base_next;
      if (nch > 0) store_child(a.c, 2 * i, ray, ch.ox, ch.oy, ch.oz, ch.pl, ch.dx[0], ch.dy[0], ch.dz[0], ch.I[0],
                               ch.qre[0], ch.qim[0], ch.nmed[0], 0, pb, hit_leaf);
      if (nch > 1) store_child(a.c, 2 * i + 1, ray, ch.ox, ch.oy, ch.oz, ch.pl, ch.dx[MAXCH - 1], ch.dy[MAXCH - 1],
                               ch.dz[MAXCH - 1], ch.I[MAXCH - 1], ch.qre[MAXCH - 1], ch.qim[MAXCH - 1],
                               ch.nmed[MAXCH - 1], 1, pb, hit_leaf);
    };
    if constexpr (REFILL) {
      bool active = has;
      bool more = true;  // (warp-uniform) the work counter has not run past the wavefront yet
      while (__syncthreads_or(active ? 1 : 0)) {
        if (active) {
          active = pop_step();
          if (!active && a.nchild) store_children();
        }
        const unsigned need = more ? __ballot_sync(0xffffffffu, !active) : 0u;
        if (need) {
          const int leader = __ffs(need) - 1;
          unsigned int base = 0;
          if (lane == leader) base = atomicAdd(&a.hdr->work_ctr, (unsigned int)__popc(need));
          base = __shfl_sync(0xffffffffu, base, leader);
          if ((long long)base + __popc(need) >= n_in) more = false;
          if (!active) {
            i = (long long)base + __popc(need & ((1u << lane) - 1u));
            if (i < n_in) {
              if (a.perm) i = a.perm[i];
              load_ray<SWEEP>(a, i, ray, solo, gcount, pop_base0);
              if constexpr (SWEEP) sweep_view(a, ray.root, sv);
              pop_base_next = a.gen0 ? 0u : (pop_base0 + gcount);
              nch = 0; chained = 0; hit_leaf = 0; ch.n = 0;
              active = true;
            }
          }
        }
      }
      continue;  // (the next trip finds the counter exhausted and leaves through the barrier above)
    } else if constexpr (PHASE) {
      bool active = has;
      while (__syncthreads_or(active ? 1 : 0)) {
        if (active) active = pop_step();
      }
    } else {
      while (pop_step()) {}
    }
    if constexpr (SPLIT) {
      if (a.nchild && has) store_children();
    }
  }

  // counters: warp reduce then one atomic per warp
  unsigned long long v[7] = {c_pops, c_inter, my_cnt[0], c_drop, c_hits, my_cnt[kBlock], my_cnt[2 * kBlock]};
#pragma unroll
  for (int k = 0; k < 7; k++) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], s);
  }
  if (lane == 0) {
    if (!a.rec_seg && v[0]) atomicAdd(&a.counters[OPTB_C_SEGMENTS], v[0]);
    if (v[1]) atomicAdd(&a.counters[OPTB_C_INTERACTIONS], v[1]);
    if (v[2]) atomicAdd(&a.counters[OPTB_C_TESTS], v[2]);
    if (v[3]) atomicAdd(&a.counters[OPTB_C_DROPPED], v[3]);
    if (!a.rec_hit && v[4]) atomicAdd(&a.counters[OPTB_C_HITS], v[4]);
    if (v[5]) atomicAdd(&a.counters[OPTB_C_TESTS_CURVED], v[5]);
    if (v[6]) atomicAdd(&a.counters[OPTB_C_BOX_TESTS], v[6]);
  }
  if (a.hist_smem) {
    __syncthreads();
    for (int k = threadIdx.x; k < (SWEEP ? a.hist_mons : a.n_mons) * per; k += blockDim.x) {
      unsigned int cnt = s_hist[k];
      if (!cnt) continue;
      int m = k / per, r = k % per;
      if (r < OPTB_HIST_BINS) atomicAdd((unsigned long long*)&a.out.hist_y[m * OPTB_HIST_BINS + r], (unsigned long long)cnt);
      else atomicAdd((unsigned long long*)&a.out.hist_yz[m * OPTB_HIST_BINS * OPTB_HIST_BINS + (r - OPTB_HIST_BINS)],
                     (unsigned long long)cnt);
    }
  }
}

// ---- ordered compaction of the sparse children into the next wavefront --------------------------------
__global__ void __launch_bounds__(kScanBlock) tile_sums_kernel(const uint8_t* __restrict__ nchild, long long n,
                                                               unsigned int* __restrict__ sums, const Header* unseen) {
  __shared__ unsigned int s[kScanBlock / 32];
  if (unseen) n = unseen->n_next;  // generation launched without the host knowing its size
  long long base = (long long)blockIdx.x * kTile;
  unsigned int acc = 0;
  for (int k = threadIdx.x; k < kTile; k += kScanBlock) {
    long long i = base + k;
    if (i < n) acc += nchild[i];
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = 0;
    for (int w = 0; w < kScanBlock / 32; w++) t += s[w];
    sums[blockIdx.x] = t;
  }
}

// single block: exclusive scan of the tile sums in place; total -> hdr->n_next; also resets the work counter
__global__ void __launch_bounds__(1024) scan_sums_kernel(unsigned int* __restrict__ sums, int ntiles, Header* hdr,
                                                         unsigned long long* counters, unsigned int capacity,
                                                         bool unseen = false) {
  __shared__ unsigned int s[1024];
  __shared__ unsigned int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < ntiles; b0 += 1024) {
    int idx = b0 + threadIdx.x;
    unsigned int v = idx < ntiles ? sums[idx] : 0u;
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      unsigned int t = threadIdx.x >= o ? s[threadIdx.x - o] : 0u;
      __syncthreads();
      s[threadIdx.x] += t;
      __syncthreads();
    }
    unsigned int incl = s[threadIdx.x];
    if (idx < ntiles) sums[idx] = carry + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry += incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    unsigned int total = carry;
    if (total > capacity) {
      atomicOr(&counters[OPTB_C_STATUS], (unsigned long long)OPTB_ST_WORK_OVERFLOW);
      total = 0;  // stop cleanly
    }
    if (unseen) {
      hdr->n_prev = hdr->n_next;
      if (hdr->n_next == 0) hdr->empty_gens++;
    }
    hdr->n_next = total;
    hdr->work_ctr = 0;
  }
}

// Ordered compaction, index only: the k-th child of wavefront entry i sits in slot 2i+k of the sparse buffer; this
// writes the list of occupied slots in reference (BFS) order. Thread t of a block handles entries base + sub*256 + t.
__global__ void __launch_bounds__(kScanBlock) slots_kernel(const uint8_t* __restrict__ nchild, long long n,
                                                           const unsigned int* __restrict__ tile_base,
                                                           uint32_t* __restrict__ slot_next, const Header* hdr,
                                                           bool unseen) {
  __shared__ unsigned int s_warp[kScanBlock / 32];
  __shared__ unsigned int s_carry;
  if (hdr->n_next == 0) return;
  if (unseen) n = hdr->n_prev;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = tile_base[blockIdx.x];
  __syncthreads();
  for (int sub = 0; sub < kTile / kScanBlock; sub++) {
    const long long i = (long long)blockIdx.x * kTile + (long long)sub * kScanBlock + threadIdx.x;
    const unsigned int mine = (i < n) ? nchild[i] : 0u;
    unsigned int incl = mine;
    for (int o = 1; o < 32; o <<= 1) {
      unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    unsigned int woff = 0, total = 0;
    for (int k = 0; k < kScanBlock / 32; k++) { if (k < wid) woff += s_warp[k]; total += s_warp[k]; }
    const unsigned int off = s_carry + woff + incl - mine;
    for (unsigned int j = 0; j < mine; j++) slot_next[off + j] = (uint32_t)(2 * i + j);
    __syncthreads();
    if (threadIdx.x == 0) s_carry += total;
    __syncthreads();
  }
}

__global__ void mark_kernel(const uint2* __restrict__ key, const uint32_t* __restrict__ slot, const Header* hdr,
                            uint32_t* __restrict__ gen_first, uint32_t* __restrict__ gen_last) {
  long long n = hdr->n_next;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    uint32_t r = key[slot[j]].y;
    if (j == 0 || key[slot[j - 1]].y != r) gen_first[r] = (uint32_t)j;
    if (j == n - 1 || key[slot[j + 1]].y != r) gen_last[r] = (uint32_t)j;
  }
}
// rank of every wavefront entry inside its root's generation and the size of that generation, next to the ray's
// record (same slot): the trace kernel loads both at once, with no per-root lookup behind the record's root
__global__ void rank_kernel(const uint2* __restrict__ key, uint2* __restrict__ rk, const uint32_t* __restrict__ slot,
                            const Header* hdr, const uint32_t* __restrict__ gen_first, const uint32_t* __restrict__ gen_last) {
  long long n = hdr->n_next;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    const uint32_t s = slot[j];
    const uint32_t r = key[s].y, first = gen_first[r];
    rk[s] = make_uint2((uint32_t)j - first, gen_last[r] - first + 1u);
  }
}

// family -> list of initial rays (CSR) for the family-serial mode
__global__ void fam_count_kernel(const int32_t* __restrict__ family, long long n, unsigned int* __restrict__ counts) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    atomicAdd(&counts[family ? family[i] : (int32_t)i], 1u);
}
__global__ void fam_scatter_kernel(const int32_t* __restrict__ family, long long n, const unsigned int* __restrict__ off,
                                   unsigned int* __restrict__ cursor, uint32_t* __restrict__ roots) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    int f = family ? family[i] : (int32_t)i;
    roots[off[f] + atomicAdd(&cursor[f], 1u)] = (uint32_t)i;
  }
}
// The same for a sweep of n rays per configuration and n_fam families per configuration: root k * n + r belongs to
// family k * n_fam + family[r]
__global__ void fam_count_sweep_kernel(const int32_t* __restrict__ family, long long n_roots, uint32_t n, int n_fam,
                                       unsigned int* __restrict__ counts) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_roots; i += (long long)gridDim.x * blockDim.x)
    atomicAdd(&counts[(i / n) * n_fam + family[i % n]], 1u);
}
__global__ void fam_scatter_sweep_kernel(const int32_t* __restrict__ family, long long n_roots, uint32_t n, int n_fam,
                                         const unsigned int* __restrict__ off, unsigned int* __restrict__ cursor,
                                         uint32_t* __restrict__ roots) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_roots; i += (long long)gridDim.x * blockDim.x) {
    const long long f = (i / n) * n_fam + family[i % n];
    roots[off[f] + atomicAdd(&cursor[f], 1u)] = (uint32_t)i;
  }
}

// Sort input of one generation: identity permutation + the coherence key, with "this root has a single live ray"
// (it will chain many pops in registers) as the top bit so that one-pop rays and chaining rays do not share warps.
__global__ void sort_prep_kernel(uint32_t* __restrict__ idx, uint32_t* __restrict__ key_dense, const uint2* __restrict__ key,
                                 const uint2* __restrict__ rk, const uint32_t* __restrict__ slot, long long n, int key_bits) {
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    idx[j] = (uint32_t)j;
    const uint32_t s = slot[j];
    const bool solo = rk[s].y == 1u;
    key_dense[j] = (key[s].x & ((1u << key_bits) - 1u)) | ((solo ? 1u : 0u) << key_bits);
  }
}

__global__ void count_flags_kernel(const uint32_t* __restrict__ flags, long long n, unsigned long long* counters) {
  unsigned int c = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) c += flags[i] != 0u;
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(&counters[OPTB_C_FLAGGED], (unsigned long long)c);
}

__global__ void finish_kernel(unsigned long long* counters, unsigned long long gens, unsigned long long launches,
                              const Header* hdr) {
  counters[OPTB_C_GENERATIONS] = gens - hdr->empty_gens;
  counters[OPTB_C_LAUNCHES] = launches;
}

// FP64 FMA peak probe: 8 independent chains per thread
__global__ void __launch_bounds__(256) dfma_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 0.999999, c = 1e-6;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// Bytes of one varied node's rows in blob form (traversal record, node_f, node_i) and of one monitor record; every
// blob section starts 16-byte aligned and these row sizes are multiples of 16, so no 16-byte word straddles two rows.
constexpr uint32_t kTravBytes = 64, kNfBytes = OPTB_NF_STRIDE * 8, kNiBytes = OPTB_NI_STRIDE * 4;
constexpr uint32_t kVarNodeBytes = kTravBytes + kNfBytes + kNiBytes, kMonBytes = kMonBlobStride * 8;
static_assert(kNfBytes % 16 == 0 && kNiBytes % 16 == 0 && kMonBytes % 16 == 0, "blob rows must be whole 16-byte words");

// optb_scene_upload_sweep_rows: writes the K configuration blobs of a sweep scene, each 16-byte word once. A word of
// configuration k is the base blob's word unless it lies in the row of a node or monitor with a slot (slot >= 0), in
// which case it comes from configuration k's rows: `rows` holds per configuration [n_var_nodes][kVarNodeBytes] then
// [n_var_mons][kMonBytes], `cfg_bytes` apart. The base blob is read by every configuration and stays in L2.
__global__ void __launch_bounds__(256) sweep_build_kernel(uint4* __restrict__ out, const uint4* __restrict__ base,
                                                         const unsigned char* __restrict__ rows,
                                                         const int32_t* __restrict__ node_slot,
                                                         const int32_t* __restrict__ mon_slot, SceneOff off, int n_nodes,
                                                         int n_mons, uint32_t stride_words, uint32_t total_words,
                                                         uint32_t cfg_bytes, uint32_t mon_rows_at) {
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < total_words; w += gridDim.x * blockDim.x) {
    const uint32_t k = w / stride_words, o = (w - k * stride_words) * 16;
    const unsigned char* cfg = rows + (size_t)k * cfg_bytes;
    const uint4* src = base + (w - k * stride_words);
    // (section, row, byte in the row) of the word; the traversal records start at offset 0
    uint32_t row = 0, in_row = 0, at = 0;
    int slot = -1;
    if (o < off.matk) {
      if (o < off.nf) { row = o / kTravBytes; in_row = o - row * kTravBytes; at = 0; }
      else if (o < off.ni) { row = (o - off.nf) / kNfBytes; in_row = o - off.nf - row * kNfBytes; at = kTravBytes; }
      else { row = (o - off.ni) / kNiBytes; in_row = o - off.ni - row * kNiBytes; at = kTravBytes + kNfBytes; }
      if ((int)row < n_nodes) slot = node_slot[row];
      if (slot >= 0) src = (const uint4*)(cfg + (size_t)slot * kVarNodeBytes + at + in_row);
    } else if (o >= off.mon && o < off.aux) {
      row = (o - off.mon) / kMonBytes;
      if ((int)row < n_mons) slot = mon_slot[row];
      if (slot >= 0) src = (const uint4*)(cfg + mon_rows_at + (size_t)slot * kMonBytes + (o - off.mon - row * kMonBytes));
    }
    out[w] = *src;
  }
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace

// ---- host side ----------------------------------------------------------------------------------------
struct optb_ctx {
  int device;
  int sm_count;
  size_t smem_optin;
  size_t smem_static;  // largest static shared memory of the shared-memory trace kernels (smem_static_max)
  char err[512];
  // arena for optb_trace_host
  void* arena; size_t arena_bytes;
  unsigned long long* h_counters;  // pinned
  unsigned int* h_hdr;             // pinned
  cudaStream_t s_h2d, s_run, s_d2h;  // optb_trace_host
  unsigned long long* h_chunk; size_t h_chunk_n;  // pinned per-chunk counters
  // Retired scene blobs, kept for the next upload: cudaMalloc/cudaFree cost milliseconds each (and cudaFree
  // synchronises the device), which is most of the latency of a small trace that re-uploads its scene per call.
  struct { unsigned char* p; size_t cap; } pool[8];
  // live-ray budget per initial ray that the last splitting optb_trace_host call needed (its grow loop starts there)
  int64_t live_per_ray_hint;
  // NCCL communicator for optb_monitor_merge (library loaded at run time)
  void* nccl_lib; void* nccl_comm; int comm_rank, comm_size; long long* d_merge;  // d_merge: device scratch of the merge
};

struct optb_scene {
  unsigned char* d_blob; size_t blob_cap; uint32_t blob_bytes; SceneOff off;
  int n_nodes, n_leaves, n_mats, n_mons, n_caps; long long n_aux;
  int max_children; int has_boxes; int has_asph; int has_grid; int has_pass;
  bool in_smem; bool hist_smem; uint32_t smem_bytes;
  // recorded on the stream of every trace that reads the blob: releasing the scene waits for this event only,
  // not for the whole device (other streams, NCCL and unrelated kernels keep running)
  cudaEvent_t last_use; bool used;
  std::vector<unsigned char>* cull;  // cullable bit per node as uploaded (optb_scene_update_nodes keeps it current)
  int n_cfg; uint32_t cfg_stride;    // sweep scenes: configurations, bytes per configuration blob (0, 0 otherwise)
};

// histograms a trace of the scene fills: [n_cfg][n_mons] for a sweep
static int hist_mons(const optb_scene* s) { return s->n_mons * std::max(s->n_cfg, 1); }

static int fail(optb_ctx* ctx, int code, const char* what, cudaError_t e = cudaSuccess) {
  // A refused runtime call may also leave its error as the runtime's last error: clear it, so that a later
  // cudaGetLastError check (the end of trace_impl) cannot report it a second time.
  if (e != cudaSuccess) cudaGetLastError();
  if (ctx) {
    if (e != cudaSuccess) snprintf(ctx->err, sizeof ctx->err, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(ctx->err, sizeof ctx->err, "%s", what);
  }
  return code;
}
#define CK(call, what) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(ctx, -10, what, e__); } while (0)

extern "C" int optb_abi_version(void) { return OPTB_ABI_VERSION; }
extern "C" int optb_comm_destroy(optb_ctx* ctx);
extern "C" int64_t optb_sort_workspace_bytes(int64_t n_rows);
static int sort_rows_dev(optb_ctx* ctx, const optb_result* res, const optb_result* dst, int64_t n_seg, int64_t n_hit,
                         const unsigned long long* d_counters, void* workspace, int64_t workspace_bytes, cudaStream_t st,
                         int end_bit);
static cudaError_t smem_static_max(size_t* out);

extern "C" int optb_ctx_create(int device, optb_ctx** out) {
  if (!out) return -1;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || device < 0 || device >= ndev) return -2;
  optb_ctx* ctx = new (std::nothrow) optb_ctx();
  if (!ctx) return -3;
  memset(ctx, 0, sizeof *ctx);
  ctx->device = device;
  int sm = 0, optin = 0;
  if (cudaSetDevice(device) != cudaSuccess ||
      cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
      cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess ||
      cudaMallocHost((void**)&ctx->h_counters, sizeof(unsigned long long) * OPTB_C_COUNT) != cudaSuccess ||
      cudaMallocHost((void**)&ctx->h_hdr, sizeof(Header)) != cudaSuccess ||
      smem_static_max(&ctx->smem_static) != cudaSuccess) {
    cudaGetLastError();
    optb_ctx_destroy(ctx);
    return -10;
  }
  ctx->sm_count = sm;
  ctx->smem_optin = (size_t)optin;
  *out = ctx;
  return 0;
}

extern "C" int optb_ctx_destroy(optb_ctx* ctx) {
  if (!ctx) return 0;
  cudaSetDevice(ctx->device);
  optb_comm_destroy(ctx);
  if (ctx->arena) cudaFree(ctx->arena);
  for (auto& b : ctx->pool) if (b.p) cudaFree(b.p);
  if (ctx->h_counters) cudaFreeHost(ctx->h_counters);
  if (ctx->h_hdr) cudaFreeHost(ctx->h_hdr);
  if (ctx->h_chunk) cudaFreeHost(ctx->h_chunk);
  if (ctx->s_h2d) { cudaStreamDestroy(ctx->s_h2d); cudaStreamDestroy(ctx->s_run); cudaStreamDestroy(ctx->s_d2h); }
  delete ctx;
  return 0;
}

extern "C" const char* optb_last_error(const optb_ctx* ctx) { return ctx ? ctx->err : "null context"; }

// Which boxes may ALSO be used to dismiss a subtree by distance ("cullable"): a hit on a leaf always lies inside the
// leaf's geometric extent (planar: the aperture in the plane x = 0; curved: the local box that brackets the reference's
// root search, optical_component.py:197-233), so if the stored lab box contains that extent in the leaf's CURRENT pose,
// every hit on the leaf is at t >= the box's entry parameter, and a box entered beyond the closest hit found so far
// cannot change the result. The reference's boxes are cached and may be stale (SURVEY A.2: the flattener ships the
// object's own `.bbox`): a stale box is still TESTED like the reference does, but never used for dismissal. A group is
// cullable when its box contains the boxes of all its children, all of them cullable. Capped leaves count every
// geometric hit, closest or not (optical_component.py:359-362): never cullable, nor is any group above them.
// One node's bit: `nf` is node i's node_f row; a group reads its children's rows and bits through row_of(j) / cull_of(j)
// (node_i, which fixes the tree, comes from `d`).
template <class RowOf, class CullOf>
static bool cull_node(const optb_scene_desc* d, int i, const double* nf, RowOf row_of, CullOf cull_of) {
  auto contains = [](const double* outer, const double* inner) {
    for (int ax = 0; ax < 3; ax++) {
      const double tol = 1e-9 * std::max(1.0, std::max(fabs(inner[2 * ax]), fabs(inner[2 * ax + 1])));
      if (!(outer[2 * ax] <= inner[2 * ax] + tol && outer[2 * ax + 1] >= inner[2 * ax + 1] - tol)) return false;
    }
    return true;
  };
  const int32_t* ni = d->node_i + (size_t)i * OPTB_NI_STRIDE;
  if (!ni[OPTB_NI_AABB]) return false;
  const int g = ni[OPTB_NI_GEOM];
  if (g == OPTB_G_GROUP || g == OPTB_G_GRID) {
    bool ok = true;
    for (int j = i + 1; j < ni[OPTB_NI_SKIP] && ok; j = d->node_i[(size_t)j * OPTB_NI_STRIDE + OPTB_NI_SKIP])
      ok = cull_of(j) && contains(nf + OPTB_NF_AABB, row_of(j) + OPTB_NF_AABB);
    return ok && ni[OPTB_NI_SKIP] > i + 1;
  }
  if (ni[OPTB_NI_CAPSLOT] >= 0) return false;
  const double* p = nf + OPTB_NF_P;
  double e[6];  // geometric extent of the hittable points in the local frame
  switch (g) {
    case OPTB_G_CIRCLE: e[0] = e[1] = 0; e[2] = e[4] = -p[0]; e[3] = e[5] = p[0]; break;
    case OPTB_G_RECT: e[0] = e[1] = 0; e[2] = -p[0]; e[3] = p[0]; e[4] = -p[1]; e[5] = p[1]; break;
    case OPTB_G_SPHERE: for (int k = 0; k < 6; k++) e[k] = p[2 + k]; break;
    case OPTB_G_ASPHERE: e[0] = p[6]; e[1] = p[7]; e[2] = e[4] = -p[0]; e[3] = e[5] = p[0]; break;
    case OPTB_G_CYL: e[0] = e[2] = -p[0]; e[1] = e[3] = p[0]; e[4] = -p[1] / 2; e[5] = p[1] / 2; break;
    default: return false;  // polygons, composite apertures: boxes are tested, not used for dismissal
  }
  if (!(e[0] <= e[1] && e[2] <= e[3] && e[4] <= e[5])) return false;
  const double* T = nf + OPTB_NF_T;
  const double* c = nf + OPTB_NF_ORIGIN;
  double lab[6] = {INFINITY, -INFINITY, INFINITY, -INFINITY, INFINITY, -INFINITY};
  for (int corner = 0; corner < 8; corner++) {
    const double x = e[corner & 1], y = e[2 + ((corner >> 1) & 1)], z = e[4 + ((corner >> 2) & 1)];
    for (int ax = 0; ax < 3; ax++) {
      const double v = T[3 * ax] * x + T[3 * ax + 1] * y + T[3 * ax + 2] * z + c[ax];
      lab[2 * ax] = std::min(lab[2 * ax], v); lab[2 * ax + 1] = std::max(lab[2 * ax + 1], v);
    }
  }
  // (a curved leaf finds roots up to 1e-9 outside its bracket; the tolerance of `contains` covers that)
  return contains(nf + OPTB_NF_AABB, lab);
}

static void cull_bits(const optb_scene_desc* d, std::vector<unsigned char>& cull) {
  const int n = d->n_nodes;
  cull.assign(n, 0);
  auto row_of = [d](int j) { return d->node_f + (size_t)j * OPTB_NF_STRIDE; };
  auto cull_of = [&cull](int j) { return cull[j] != 0; };
  for (int i = n - 1; i >= 0; i--)  // children before parents (pre-order table, reverse scan)
    cull[i] = cull_node(d, i, row_of(i), row_of, cull_of);
}

// Device-side extras of an asphere row: k1 of the sign / Newton functor (AsphF) in the FOCAL slot, which a refractive
// leaf does not use. Same expressions, same IEEE operations as the device used to evaluate per test.
static void asphere_constants(double* nf, const int32_t* ni) {
  if (ni[OPTB_NI_GEOM] != OPTB_G_ASPHERE) return;
  const double* c = nf + OPTB_NF_P + 1;
  if (ni[OPTB_NI_AUX] == OPTB_ASPH_PARAMETRIC) nf[OPTB_NF_FOCAL] = (1.0 + c[1]) / (c[0] * c[0]);
  else nf[OPTB_NF_FOCAL] = (c[1] + 1.0) / ((c[1] - 1.0) * c[0] * c[0]);
}

// The kernels index the tables without bounds checks: reject anything that could walk out of them. Node i with the
// rows `ni` / `nf` (d's own, or a sweep configuration's replacement of them) in the tables of `d`.
static int validate_node(optb_ctx* ctx, const optb_scene_desc* d, int i, const int32_t* ni, const double* nf) {
  const int g = ni[OPTB_NI_GEOM];
  if (ni[OPTB_NI_SKIP] <= i || ni[OPTB_NI_SKIP] > d->n_nodes) return fail(ctx, -5, "scene: node skip pointer out of range");
  if (g < OPTB_G_GROUP || g > OPTB_G_GRID) return fail(ctx, -5, "scene: unknown geometry kind");
  if (g == OPTB_G_GRID) {  // lattice descriptor: inside the aux pool, every listed child a leaf of this subtree
    const long long off = ni[OPTB_NI_AUX];
    if (off < 0 || off + OPTB_GRID_CELLS > d->n_aux) return fail(ctx, -5, "scene: lattice descriptor out of range");
    const double* gd = d->aux + off;
    const double cells = gd[OPTB_GRID_NOUTER] * gd[OPTB_GRID_NINNER] + gd[OPTB_GRID_NEXT];
    if (!(gd[OPTB_GRID_NOUTER] >= 1 && gd[OPTB_GRID_NINNER] >= 1 && gd[OPTB_GRID_NEXT] >= 0 && cells <= 1e8) ||
        off + OPTB_GRID_CELLS + (long long)cells > d->n_aux)
      return fail(ctx, -5, "scene: lattice descriptor out of range");
    for (long long k = 0; k < (long long)cells; k++) {
      const double c = gd[OPTB_GRID_CELLS + k];
      if (!(c > i && c < ni[OPTB_NI_SKIP]) || d->node_i[(size_t)c * OPTB_NI_STRIDE + OPTB_NI_GEOM] == OPTB_G_GROUP ||
          d->node_i[(size_t)c * OPTB_NI_STRIDE + OPTB_NI_GEOM] == OPTB_G_GRID)
        return fail(ctx, -5, "scene: lattice child is not a leaf of the group's subtree");
    }
  }
  if (g == OPTB_G_GROUP || g == OPTB_G_GRID) return 0;
  if (ni[OPTB_NI_SKIP] != i + 1) return fail(ctx, -5, "scene: a leaf must skip to the next node");
  if (ni[OPTB_NI_INTER] < OPTB_I_MIRROR || ni[OPTB_NI_INTER] > OPTB_I_PASS) return fail(ctx, -5, "scene: unknown interaction kind");
  if (ni[OPTB_NI_MAT1] < 0 || ni[OPTB_NI_MAT1] >= d->n_materials || ni[OPTB_NI_MAT2] < 0 || ni[OPTB_NI_MAT2] >= d->n_materials)
    return fail(ctx, -5, "scene: material index out of range");
  if (ni[OPTB_NI_CAPSLOT] >= d->n_capslots) return fail(ctx, -5, "scene: cap slot out of range");
  if (ni[OPTB_NI_LEAF] < 0 || ni[OPTB_NI_LEAF] >= d->n_leaves) return fail(ctx, -5, "scene: leaf index out of range");
  auto poly_ok = [&](long long off) {
    if (off < 0 || off + OPTB_POLY_HEADER > d->n_aux) return false;
    const double nv = d->aux[off];
    return nv >= 3 && nv <= 1e6 && off + OPTB_POLY_HEADER + 2 * (long long)nv <= d->n_aux;
  };
  const double* p = nf + OPTB_NF_P;
  if ((g == OPTB_G_POLY2D || g == OPTB_G_POLY3D) && !poly_ok(ni[OPTB_NI_AUX])) return fail(ctx, -5, "scene: polygon record out of range");
  if (g == OPTB_G_ASPHERE && ni[OPTB_NI_AUX] != OPTB_ASPH_PARAMETRIC && ni[OPTB_NI_AUX] != OPTB_ASPH_EXACT_SPH)
    return fail(ctx, -5, "scene: unknown asphere form");
  if (g == OPTB_G_CSG && (int)p[0] == 2) {  // nested composite: a well-formed postfix program in the aux pool
    const long long off = ni[OPTB_NI_AUX];
    if (off < 0 || off + 1 > d->n_aux) return fail(ctx, -5, "scene: CSG program out of range");
    const double nt = d->aux[off];
    if (!(nt >= 3 && nt <= 4096) || off + 1 + 3 * (long long)nt > d->n_aux) return fail(ctx, -5, "scene: CSG program out of range");
    int depth = 0;
    for (int k = 0; k < (int)nt; k++) {
      const int code = (int)d->aux[off + 1 + 3 * k];
      if (code == OPTB_G_CIRCLE || code == OPTB_G_RECT || code == OPTB_G_POLY2D) {
        if (code == OPTB_G_POLY2D && !poly_ok((long long)d->aux[off + 2 + 3 * k])) return fail(ctx, -5, "scene: CSG polygon out of range");
        if (++depth > OPTB_CSG_MAX_DEPTH) return fail(ctx, -5, "scene: CSG program nests too deep");
      } else if (code == OPTB_CSG_SUBTRACT || code == OPTB_CSG_UNION) {
        if (depth < 2) return fail(ctx, -5, "scene: malformed CSG program");
        depth--;
      } else {
        return fail(ctx, -5, "scene: bad CSG token");
      }
    }
    if (depth != 1) return fail(ctx, -5, "scene: malformed CSG program");
  } else if (g == OPTB_G_CSG) {
    if ((int)p[0] != 0 && (int)p[0] != 1) return fail(ctx, -5, "scene: bad CSG op");
    for (int q = 0; q < 2; q++) {
      const int k = (int)p[1 + 3 * q];
      if (k != OPTB_G_CIRCLE && k != OPTB_G_RECT && k != OPTB_G_POLY2D) return fail(ctx, -5, "scene: bad CSG operand");
      if (k == OPTB_G_POLY2D && !poly_ok((long long)p[2 + 3 * q])) return fail(ctx, -5, "scene: CSG polygon out of range");
    }
  }
  return 0;
}

static int validate_desc(optb_ctx* ctx, const optb_scene_desc* d) {
  if (d->abi_version != OPTB_ABI_VERSION) return fail(ctx, -4, "scene ABI version mismatch");
  if (d->n_nodes < 0 || d->n_materials < 1) return fail(ctx, -5, "bad scene counts");
  for (int i = 0; i < d->n_nodes; i++)
    if (int rc = validate_node(ctx, d, i, d->node_i + (size_t)i * OPTB_NI_STRIDE, d->node_f + (size_t)i * OPTB_NF_STRIDE)) return rc;
  return 0;
}

// Byte layout of one scene blob; returns its size.
static size_t blob_layout(const optb_scene_desc* d, SceneOff& off) {
  size_t b_nf = (size_t)d->n_nodes * OPTB_NF_STRIDE * 8, b_ni = (size_t)d->n_nodes * OPTB_NI_STRIDE * 4;
  size_t b_mk = (size_t)d->n_materials * 4, b_mf = (size_t)d->n_materials * OPTB_MF_STRIDE * 8;
  size_t b_mon = (size_t)std::max(d->n_monitors, 1) * kMonBlobStride * 8, b_aux = (size_t)std::max<long long>(d->n_aux, 1) * 8;
  size_t o = 0;
  const size_t b_trav = (size_t)std::max(d->n_nodes, 1) * 64;
  off.trav = (uint32_t)o; o = align_up(o + b_trav, 16);
  off.nf = (uint32_t)o; o = align_up(o + b_nf, 16);
  off.ni = (uint32_t)o; o = align_up(o + b_ni, 16);
  off.matk = (uint32_t)o; o = align_up(o + b_mk, 16);
  off.matf = (uint32_t)o; o = align_up(o + b_mf, 16);
  off.mon = (uint32_t)o; o = align_up(o + b_mon, 16);
  off.aux = (uint32_t)o; o = align_up(o + b_aux, 16);
  return o;
}

// Parent of every node, from the skip pointers (pre-order: the innermost open group that still covers i).
static std::vector<int32_t> node_parents(const optb_scene_desc* d) {
  std::vector<int32_t> parent(d->n_nodes, -1), open;
  for (int i = 0; i < d->n_nodes; i++) {
    const int32_t* ni = d->node_i + (size_t)i * OPTB_NI_STRIDE;
    while (!open.empty() && d->node_i[(size_t)open.back() * OPTB_NI_STRIDE + OPTB_NI_SKIP] <= i) open.pop_back();
    parent[i] = open.empty() ? -1 : open.back();
    if (ni[OPTB_NI_GEOM] == OPTB_G_GROUP || ni[OPTB_NI_GEOM] == OPTB_G_GRID) open.push_back(i);
  }
  return parent;
}

// Box word of a traversal record: bit 0 = test the box (component_group.py:98-107), bit 1 = the box may dismiss by
// distance (cull_bits).
static int32_t box_word(const int32_t* ni, bool cull) { return (ni[OPTB_NI_AABB] ? 1 : 0) | (cull ? 2 : 0); }

// Blob record of one monitor: the ABI record + the histogram constants derived from it (kMonBlobStride).
static void mon_record(double* mf, const double* rec) {
  memcpy(mf, rec, OPTB_MON_STRIDE * 8);
  const double w = mf[OPTB_MON_HW] - (-mf[OPTB_MON_HW]), h = mf[OPTB_MON_HH] - (-mf[OPTB_MON_HH]);  // hi - lo as hist_bin forms it
  mf[OPTB_MON_STRIDE] = OPTB_HIST_BINS / w; mf[OPTB_MON_STRIDE + 1] = w / OPTB_HIST_BINS;
  mf[OPTB_MON_STRIDE + 2] = OPTB_HIST_BINS / h; mf[OPTB_MON_STRIDE + 3] = h / OPTB_HIST_BINS;
}

// Host image of one scene blob (zeroed `host`, blob_layout bytes); `cull` receives the cullable bit of every node.
static void fill_blob(const optb_scene_desc* d, const SceneOff& off, unsigned char* host, std::vector<unsigned char>& cull) {
  const size_t b_nf = (size_t)d->n_nodes * OPTB_NF_STRIDE * 8, b_ni = (size_t)d->n_nodes * OPTB_NI_STRIDE * 4;
  if (d->n_nodes) {
    memcpy(host + off.nf, d->node_f, b_nf);
    memcpy(host + off.ni, d->node_i, b_ni);
    const std::vector<int32_t> parent = node_parents(d);
    cull_bits(d, cull);
    for (int i = 0; i < d->n_nodes; i++) {  // compact traversal records
      unsigned char* tv = host + off.trav + (size_t)i * kTravBytes;
      const int32_t* ni = d->node_i + (size_t)i * OPTB_NI_STRIDE;
      memcpy(tv, d->node_f + (size_t)i * OPTB_NF_STRIDE + OPTB_NF_AABB, 48);
      const int32_t pack[4] = {ni[OPTB_NI_GEOM], ni[OPTB_NI_SKIP], box_word(ni, cull[i]), parent[i]};
      memcpy(tv + 48, pack, 16);
    }
  }
  memcpy(host + off.matk, d->mat_kind, (size_t)d->n_materials * 4);
  memcpy(host + off.matf, d->mat_f, (size_t)d->n_materials * OPTB_MF_STRIDE * 8);
  for (int m = 0; m < d->n_monitors; m++)
    mon_record((double*)(host + off.mon) + (size_t)m * kMonBlobStride, d->mon_f + (size_t)m * OPTB_MON_STRIDE);
  for (int i = 0; i < d->n_nodes; i++) asphere_constants((double*)(host + off.nf) + (size_t)i * OPTB_NF_STRIDE,
                                                         d->node_i + (size_t)i * OPTB_NI_STRIDE);
  if (d->n_aux) memcpy(host + off.aux, d->aux, (size_t)d->n_aux * 8);
}

// Most rays one interaction of a node can emit.
static int node_children(const int32_t* ni, const double* nf) {
  switch (ni[OPTB_NI_INTER]) {
    case OPTB_I_MIRROR: return (nf[OPTB_NF_REFL] > 0) + (nf[OPTB_NF_TRANS] > 0);
    case OPTB_I_REFRACT: return nf[OPTB_NF_REFL] > 0 ? 2 : 1;
    case OPTB_I_THINLENS: case OPTB_I_PASS: return 1;
    default: return 0;
  }
}

// Scene-wide properties that pick the kernel variant. max_children: most children one interaction can emit (decides
// whether the wavefront machinery is needed).
struct SceneProps { int max_children, has_boxes, has_asph, has_grid, has_pass; };
static SceneProps scene_props(const optb_scene_desc* d) {
  SceneProps p{0, 0, 0, 0, 0};
  for (int i = 0; i < d->n_nodes; i++) {
    const int32_t* ni = d->node_i + (size_t)i * OPTB_NI_STRIDE;
    if (ni[OPTB_NI_AABB]) p.has_boxes = 1;
    if (ni[OPTB_NI_GEOM] == OPTB_G_ASPHERE) p.has_asph = 1;
    if (ni[OPTB_NI_GEOM] == OPTB_G_GRID) p.has_grid = 1;
    if (ni[OPTB_NI_INTER] == OPTB_I_PASS) p.has_pass = 1;
    p.max_children = std::max(p.max_children, node_children(ni, d->node_f + (size_t)i * OPTB_NF_STRIDE));
  }
  return p;
}

// First node_i column other than OPTB_NI_ORTHO in which two rows differ, or -1. The configurations of a sweep may differ
// in that column only: a leaf index, skip pointer, material and cap slot mean the same in every configuration.
static int ni_row_differs(const int32_t* a, const int32_t* b) {
  for (int c = 0; c < OPTB_NI_STRIDE; c++)
    if (c != OPTB_NI_ORTHO && a[c] != b[c]) return c;
  return -1;
}

// Device buffer of at least `bytes`: the smallest retired blob that is large enough, else a new allocation.
static cudaError_t blob_acquire(optb_ctx* ctx, size_t bytes, unsigned char** p, size_t* cap) {
  int pick = -1;
  for (int k = 0; k < 8; k++)
    if (ctx->pool[k].p && ctx->pool[k].cap >= bytes && (pick < 0 || ctx->pool[k].cap < ctx->pool[pick].cap)) pick = k;
  if (pick >= 0) {
    *p = ctx->pool[pick].p; *cap = ctx->pool[pick].cap;
    ctx->pool[pick].p = nullptr; ctx->pool[pick].cap = 0;
    return cudaSuccess;
  }
  *cap = (bytes + 65535) & ~(size_t)65535;
  return cudaMalloc((void**)p, *cap);
}

// Retire a device buffer that no kernel reads any more: into a free pool slot when it is small enough, else freed.
static void blob_release(optb_ctx* ctx, unsigned char* p, size_t cap) {
  int slot = -1;
  if (ctx && cap <= ((size_t)64 << 20))
    for (int k = 0; k < 8 && slot < 0; k++) if (!ctx->pool[k].p) slot = k;
  if (slot >= 0) {
    ctx->pool[slot].p = p; ctx->pool[slot].cap = cap;
  } else {
    cudaFree(p);
  }
}

// Handle of one scene (n_cfg = 0) or of a sweep of n_cfg configurations with the sizes of `d`: layout, shared-memory
// plan and a device blob of n_cfg configuration blobs back to back (contents and kernel-selection properties are the
// caller's to fill).
static int scene_alloc(optb_ctx* ctx, const optb_scene_desc* d, int n_cfg, optb_scene** out) {
  const int K = std::max(n_cfg, 1);
  cudaSetDevice(ctx->device);
  optb_scene* s = new (std::nothrow) optb_scene();
  if (!s) return -3;
  memset(s, 0, sizeof *s);
  s->n_nodes = d->n_nodes; s->n_leaves = d->n_leaves; s->n_mats = d->n_materials; s->n_mons = d->n_monitors;
  s->n_caps = d->n_capslots; s->n_aux = d->n_aux;
  s->n_cfg = n_cfg;
  const size_t stride = blob_layout(d, s->off);
  const size_t o = stride * K;
  if (o > 0xfff00000ull) { delete s; return fail(ctx, -6, "scene too large"); }
  s->blob_bytes = (uint32_t)o; s->cfg_stride = (uint32_t)stride;
  size_t hist_bytes = (size_t)K * d->n_monitors * OPTB_HIST_BINS * (OPTB_HIST_BINS + 1) * 4;
  // dynamic + static shared memory of a block may not exceed the opt-in limit. The budget takes the largest static
  // size of the shared-memory kernels, not the one the scene's first trace selects: a later trace of the same scene
  // with flag_ambiguity, reference_roots or a family column runs a general kind, which has the largest.
  size_t budget = ctx->smem_optin > ctx->smem_static ? ctx->smem_optin - ctx->smem_static : 0;
  s->in_smem = !n_cfg && (o <= budget);  // sweep kernels read the tables from global memory (L1/L2)
  size_t used = s->in_smem ? o : 0;
  s->hist_smem = (hist_bytes > 0 && used + hist_bytes <= std::min<size_t>(budget, used + 65536));
  s->smem_bytes = (uint32_t)(used + (s->hist_smem ? hist_bytes : 0));
  if (d->n_nodes) s->cull = new std::vector<unsigned char>();
  cudaError_t e = blob_acquire(ctx, o, &s->d_blob, &s->blob_cap);
  if (e != cudaSuccess) { delete s->cull; delete s; return fail(ctx, -10, "cudaMalloc(scene)", e); }
  e = cudaEventCreateWithFlags(&s->last_use, cudaEventDisableTiming);
  if (e != cudaSuccess) { optb_scene_destroy(ctx, s); return fail(ctx, -10, "cudaEventCreate(scene)", e); }
  *out = s;
  return 0;
}

// One scene (n_cfg = 0) or a sweep of n_cfg configurations of one topology (descs checked by the caller): the
// configuration blobs lie back to back at a stride of one blob.
static int scene_upload(optb_ctx* ctx, const optb_scene_desc* ds, int n_cfg, optb_scene** out) {
  const int K = std::max(n_cfg, 1);
  for (int k = 0; k < K; k++)
    if (int rc = validate_desc(ctx, &ds[k])) return rc;
  optb_scene* s = nullptr;
  if (int rc = scene_alloc(ctx, &ds[0], n_cfg, &s)) return rc;
  const size_t stride = s->cfg_stride;
  std::vector<unsigned char> host(s->blob_bytes, 0);
  for (int k = 0; k < K; k++) {
    std::vector<unsigned char> cull_k;  // (cull bits are per configuration; the scene keeps the first one's)
    fill_blob(&ds[k], s->off, host.data() + stride * k, k == 0 && s->cull ? *s->cull : cull_k);
    const SceneProps p = scene_props(&ds[k]);
    s->max_children = std::max(s->max_children, p.max_children);
    s->has_boxes |= p.has_boxes; s->has_asph |= p.has_asph; s->has_grid |= p.has_grid; s->has_pass |= p.has_pass;
  }
  cudaError_t e = cudaMemcpy(s->d_blob, host.data(), s->blob_bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { optb_scene_destroy(ctx, s); return fail(ctx, -10, "cudaMemcpy(scene)", e); }
  *out = s;
  return 0;
}

extern "C" int optb_scene_upload(optb_ctx* ctx, const optb_scene_desc* d, optb_scene** out) {
  if (!ctx || !d || !out) return -1;
  return scene_upload(ctx, d, 0, out);
}

extern "C" int optb_scene_upload_sweep(optb_ctx* ctx, const optb_scene_desc* descs, int32_t n_configs, optb_scene** out) {
  if (!ctx || !descs || !out) return -1;
  if (n_configs < 1) return fail(ctx, -5, "optb_scene_upload_sweep: n_configs must be >= 1");
  const optb_scene_desc* d0 = &descs[0];
  char msg[160];
  for (int k = 1; k < n_configs; k++) {
    const optb_scene_desc* d = &descs[k];
    if (d->n_nodes != d0->n_nodes || d->n_leaves != d0->n_leaves || d->n_materials != d0->n_materials ||
        d->n_monitors != d0->n_monitors || d->n_capslots != d0->n_capslots || d->n_aux != d0->n_aux) {
      snprintf(msg, sizeof msg, "optb_scene_upload_sweep: configuration %d differs from configuration 0 in its table sizes", k);
      return fail(ctx, -5, msg);
    }
    for (int i = 0; i < d0->n_nodes; i++) {
      const int c = ni_row_differs(d->node_i + (size_t)i * OPTB_NI_STRIDE, d0->node_i + (size_t)i * OPTB_NI_STRIDE);
      if (c >= 0) {
        snprintf(msg, sizeof msg, "optb_scene_upload_sweep: configuration %d differs from configuration 0 in node_i row %d column %d", k, i, c);
        return fail(ctx, -5, msg);
      }
    }
    if (memcmp(d->mat_kind, d0->mat_kind, (size_t)d0->n_materials * 4)) {
      snprintf(msg, sizeof msg, "optb_scene_upload_sweep: configuration %d differs from configuration 0 in its material kinds", k);
      return fail(ctx, -5, msg);
    }
  }
  return scene_upload(ctx, descs, n_configs, out);
}

extern "C" int optb_scene_upload_sweep_rows(optb_ctx* ctx, const optb_scene_desc* base, int32_t n_configs,
                                            const int32_t* nodes, int32_t n_var_nodes, const double* node_f,
                                            const int32_t* node_i, const int32_t* monitors, int32_t n_var_monitors,
                                            const double* mon_f, optb_scene** out) {
  if (!ctx || !base || !out || n_var_nodes < 0 || n_var_monitors < 0 || (n_var_nodes && (!nodes || !node_f || !node_i)) ||
      (n_var_monitors && (!monitors || !mon_f)))
    return -1;
  const optb_scene_desc* d = base;
  char msg[768];
  if (n_configs < 1) return fail(ctx, -5, "optb_scene_upload_sweep_rows: n_configs must be >= 1");
  if (int rc = validate_desc(ctx, d)) return rc;
  const int K = n_configs, N = d->n_nodes, M = d->n_monitors;
  std::vector<int32_t> var_of(N, -1), mon_slot(std::max(M, 1), -1);
  for (int v = 0; v < n_var_nodes; v++) {
    const int i = nodes[v];
    if (i < 0 || i >= N || var_of[i] >= 0) {
      snprintf(msg, sizeof msg, "optb_scene_upload_sweep_rows: varied node %d (entry %d) is out of range or repeated", i, v);
      return fail(ctx, -5, msg);
    }
    var_of[i] = v;
  }
  for (int w = 0; w < n_var_monitors; w++) {
    const int m = monitors[w];
    if (m < 0 || m >= M || mon_slot[m] >= 0) {
      snprintf(msg, sizeof msg, "optb_scene_upload_sweep_rows: varied monitor %d (entry %d) is out of range or repeated", m, w);
      return fail(ctx, -5, msg);
    }
    mon_slot[m] = w;
  }
  auto row_i = [&](int k, int v) { return node_i + ((size_t)k * n_var_nodes + v) * OPTB_NI_STRIDE; };
  auto row_f = [&](int k, int v) { return node_f + ((size_t)k * n_var_nodes + v) * OPTB_NF_STRIDE; };
  for (int k = 0; k < K; k++)
    for (int v = 0; v < n_var_nodes; v++) {
      const int i = nodes[v];
      const int c = ni_row_differs(row_i(k, v), d->node_i + (size_t)i * OPTB_NI_STRIDE);
      if (c >= 0) {
        snprintf(msg, sizeof msg, "optb_scene_upload_sweep_rows: configuration %d differs from the base in node_i row %d column %d", k, i, c);
        return fail(ctx, -5, msg);
      }
      if (validate_node(ctx, d, i, row_i(k, v), row_f(k, v))) {
        snprintf(msg, sizeof msg, "optb_scene_upload_sweep_rows: configuration %d, node %d: %s", k, i, ctx->err);
        return fail(ctx, -5, msg);
      }
    }
  optb_scene* s = nullptr;
  if (int rc = scene_alloc(ctx, d, K, &s)) return rc;
  // Rows sent per configuration: the varied nodes and all their ancestors (slots in pre-order), whose cull bits follow
  // their children's boxes and bits; every other node keeps the base's rows and bit. Then the varied monitors.
  const std::vector<int32_t> parent = node_parents(d);
  std::vector<int32_t> node_slot(std::max(N, 1), -1), U;
  for (int v = 0; v < n_var_nodes; v++)
    for (int i = nodes[v]; i >= 0 && node_slot[i] < 0; i = parent[i]) node_slot[i] = 0;
  for (int i = 0; i < N; i++)
    if (node_slot[i] >= 0) { node_slot[i] = (int32_t)U.size(); U.push_back(i); }
  const size_t stride = s->cfg_stride, n_u = U.size();
  const size_t maps_at = stride, rows_at = maps_at + align_up((node_slot.size() + mon_slot.size()) * 4, 16);
  const size_t mon_rows_at = n_u * kVarNodeBytes, cfg_bytes = mon_rows_at + (size_t)n_var_monitors * kMonBytes;
  // staging: base blob, slot maps, configuration rows
  std::vector<unsigned char> host(rows_at + K * cfg_bytes, 0);
  std::vector<unsigned char> cull_tmp;
  std::vector<unsigned char>& cull = s->cull ? *s->cull : cull_tmp;
  fill_blob(d, s->off, host.data(), cull);
  memcpy(host.data() + maps_at, node_slot.data(), node_slot.size() * 4);
  memcpy(host.data() + maps_at + node_slot.size() * 4, mon_slot.data(), mon_slot.size() * 4);
  const SceneProps p = scene_props(d);  // kinds, boxes and interactions live in node_i: the same in every configuration
  s->has_boxes = p.has_boxes; s->has_asph = p.has_asph; s->has_grid = p.has_grid; s->has_pass = p.has_pass;
  for (int i = 0; i < N; i++)
    if (var_of[i] < 0) s->max_children = std::max(s->max_children, node_children(d->node_i + (size_t)i * OPTB_NI_STRIDE, d->node_f + (size_t)i * OPTB_NF_STRIDE));
  std::vector<unsigned char> cull_k(n_u);
  for (int k = 0; k < K; k++) {
    unsigned char* cfg = host.data() + rows_at + k * cfg_bytes;
    auto nf_of = [&](int j) { return var_of[j] >= 0 ? row_f(k, var_of[j]) : d->node_f + (size_t)j * OPTB_NF_STRIDE; };
    auto ni_of = [&](int j) { return var_of[j] >= 0 ? row_i(k, var_of[j]) : d->node_i + (size_t)j * OPTB_NI_STRIDE; };
    auto cull_of = [&](int j) { return (node_slot[j] >= 0 ? cull_k[node_slot[j]] : cull[j]) != 0; };
    for (size_t u = n_u; u-- > 0;) {  // children before parents
      const int i = U[u];
      cull_k[u] = cull_node(d, i, nf_of(i), nf_of, cull_of);
      unsigned char* r = cfg + u * kVarNodeBytes;
      memcpy(r, host.data() + s->off.trav + (size_t)i * kTravBytes, kTravBytes);  // kind, skip, parent: the base's
      memcpy(r, nf_of(i) + OPTB_NF_AABB, 48);
      const int32_t word = box_word(ni_of(i), cull_k[u]);
      memcpy(r + 56, &word, 4);
      memcpy(r + kTravBytes, nf_of(i), kNfBytes);
      asphere_constants((double*)(r + kTravBytes), ni_of(i));
      memcpy(r + kTravBytes + kNfBytes, ni_of(i), kNiBytes);
    }
    for (int v = 0; v < n_var_nodes; v++) s->max_children = std::max(s->max_children, node_children(row_i(k, v), row_f(k, v)));
    for (int w = 0; w < n_var_monitors; w++)
      mon_record((double*)(cfg + mon_rows_at + (size_t)w * kMonBytes), mon_f + ((size_t)k * n_var_monitors + w) * OPTB_MON_STRIDE);
  }
  // one copy of the staging, one kernel writing every configuration blob (legacy default stream: after the copy)
  unsigned char* stage = nullptr;
  size_t stage_cap = 0;
  cudaError_t e = blob_acquire(ctx, host.size(), &stage, &stage_cap);
  if (e == cudaSuccess) e = cudaMemcpy(stage, host.data(), host.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    const uint32_t total = s->blob_bytes / 16;
    const int grid = (int)std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 8);
    sweep_build_kernel<<<std::max(grid, 1), 256>>>((uint4*)s->d_blob, (const uint4*)stage, stage + rows_at,
                                                   (const int32_t*)(stage + maps_at), (const int32_t*)(stage + maps_at) + node_slot.size(),
                                                   s->off, N, M, (uint32_t)(stride / 16), total, (uint32_t)cfg_bytes,
                                                   (uint32_t)mon_rows_at);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  if (stage) blob_release(ctx, stage, stage_cap);
  if (e != cudaSuccess) { optb_scene_destroy(ctx, s); return fail(ctx, -10, "optb_scene_upload_sweep_rows: building the configurations", e); }
  *out = s;
  return 0;
}

extern "C" int optb_scene_update_nodes(optb_ctx* ctx, optb_scene* s, const optb_scene_desc* d, const int32_t* nodes,
                                       int32_t n, void* stream_v) {
  if (!ctx || !s || !d || (n > 0 && !nodes)) return -1;
  if (s->n_cfg) return fail(ctx, -7, "optb_scene_update_nodes: not available on a sweep scene (upload the configurations again)");
  if (d->n_nodes != s->n_nodes || d->n_leaves != s->n_leaves || d->n_materials != s->n_mats || d->n_aux != s->n_aux ||
      d->n_capslots != s->n_caps)
    return fail(ctx, -5, "optb_scene_update_nodes: the tables no longer have the shape of the uploaded scene");
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream_v;
  for (int k = 0; k < n; k++) {
    const int i = nodes[k];
    if (i < 0 || i >= d->n_nodes) return fail(ctx, -5, "optb_scene_update_nodes: node index out of range");
    const int32_t* ni = d->node_i + (size_t)i * OPTB_NI_STRIDE;
    const double* nf = d->node_f + (size_t)i * OPTB_NF_STRIDE;
    double row[OPTB_NF_STRIDE];
    memcpy(row, nf, sizeof row);
    asphere_constants(row, ni);
    // (pageable source: the call returns once `row` has been copied to the driver's staging memory)
    CK(cudaMemcpyAsync(s->d_blob + s->off.nf + (size_t)i * OPTB_NF_STRIDE * 8, row, OPTB_NF_STRIDE * 8, cudaMemcpyHostToDevice, st), "update node_f");
    CK(cudaMemcpyAsync(s->d_blob + s->off.ni + (size_t)i * OPTB_NI_STRIDE * 4, ni, OPTB_NI_STRIDE * 4, cudaMemcpyHostToDevice, st), "update node_i");
    CK(cudaMemcpyAsync(s->d_blob + s->off.trav + (size_t)i * 64, nf + OPTB_NF_AABB, 48, cudaMemcpyHostToDevice, st), "update box");
  }
  // a moved node may change which boxes are allowed to dismiss by distance, up to the root: recompute, send the changes
  if (s->cull) {
    std::vector<unsigned char> now;
    cull_bits(d, now);
    for (int i = 0; i < d->n_nodes; i++) {
      if (now[i] == (*s->cull)[i]) continue;
      const int32_t word = box_word(d->node_i + (size_t)i * OPTB_NI_STRIDE, now[i]);
      CK(cudaMemcpyAsync(s->d_blob + s->off.trav + (size_t)i * 64 + 56, &word, 4, cudaMemcpyHostToDevice, st), "update box word");
    }
    s->cull->swap(now);
  }
  // scene-wide properties that pick the kernel variant follow the new rows
  const SceneProps p = scene_props(d);
  s->max_children = p.max_children; s->has_boxes = p.has_boxes; s->has_asph = p.has_asph; s->has_pass = p.has_pass;
  return 0;
}

extern "C" int optb_scene_destroy(optb_ctx* ctx, optb_scene* s) {
  if (!s) return 0;
  if (ctx) cudaSetDevice(ctx->device);
  if (s->d_blob) {
    if (s->used) cudaEventSynchronize(s->last_use);  // no kernel may still be reading the blob
    blob_release(ctx, s->d_blob, s->blob_cap);
  }
  if (s->last_use) cudaEventDestroy(s->last_use);
  delete s->cull;
  delete s;
  return 0;
}

namespace {
struct WsLayout {
  size_t hdr, w, c, nchild, gen_first, gen_last, sums, iota, perm, key_sorted, key_dense, slot_a, slot_b, cub, cub_bytes, total;
  long long cap;  // wavefront capacity (rays)
};
size_t raybuf_bytes(long long cap) { return align_up((size_t)cap * sizeof(RayRec), 256) + 2 * align_up((size_t)cap * 8, 256); }
WsLayout ws_layout(long long n_rays, long long max_live, bool split) {
  WsLayout L{};
  size_t o = 0;
  L.hdr = o; o += align_up(sizeof(Header), 256);
  L.cap = split ? std::max(max_live, n_rays) : 0;
  if (split) {
    L.w = o; o += raybuf_bytes(2 * L.cap);  // two sparse child buffers, used alternately as source and destination
    L.c = o; o += raybuf_bytes(2 * L.cap);
    L.slot_a = o; o += align_up((size_t)L.cap * 4, 256);
    L.slot_b = o; o += align_up((size_t)L.cap * 4, 256);
    L.key_dense = o; o += align_up((size_t)L.cap * 4, 256);
    L.nchild = o; o += align_up((size_t)L.cap, 256);
    L.gen_first = o; o += align_up((size_t)n_rays * 4, 256);
    L.gen_last = o; o += align_up((size_t)n_rays * 4, 256);
    L.sums = o; o += align_up(((size_t)L.cap / kTile + 2) * 4, 256);
    L.iota = o; o += align_up((size_t)L.cap * 4, 256);
    L.perm = o; o += align_up((size_t)L.cap * 4, 256);
    L.key_sorted = o; o += align_up((size_t)L.cap * 4, 256);
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)std::min<long long>(L.cap, 0x7fffffffll), 0, 32);
    L.cub = o; L.cub_bytes = align_up(tb + 256, 256); o += L.cub_bytes;
  }
  L.total = o;
  return L;
}
RayBuf make_raybuf(unsigned char* base, long long cap) {
  RayBuf b;
  b.rec = (RayRec*)base;
  b.key = (uint2*)(base + align_up((size_t)cap * sizeof(RayRec), 256));
  b.rk = (uint2*)(base + align_up((size_t)cap * sizeof(RayRec), 256) + align_up((size_t)cap * 8, 256));
  return b;
}
bool needs_wavefront(const optb_scene* s, const optb_params* p) {
  return s->max_children > 1 || p->chain_len > 0 || p->flag_ambiguity || p->reference_roots || s->has_pass;  // (these run the SPLIT variants)
}
// Interact caps make the result depend on the reference's sequential order as soon as two rays of one family can
// be in flight: splitting scenes, or several initial rays sharing an `_id` (family column given).
bool needs_serial(const optb_scene* s, const optb_rays* r, const optb_params* p) {
  return s->n_caps > 0 && !p->caps_slack && (s->max_children > 1 || r->family != nullptr);
}
struct SerialLayout { size_t hdr, off, cursor, roots, ring, total; };
SerialLayout serial_layout(long long n_rays, long long n_fam, long long ring_entries) {
  SerialLayout L{};
  size_t o = 0;
  L.hdr = o; o += align_up(sizeof(Header), 256);
  L.off = o; o += align_up((size_t)(n_fam + 2) * 4, 256);
  L.cursor = o; o += align_up((size_t)(n_fam + 1) * 4, 256);
  L.roots = o; o += align_up((size_t)std::max<long long>(n_rays, 1) * 4, 256);
  L.ring = o; o += raybuf_bytes(std::max<long long>(ring_entries, 1));
  L.total = o;
  return L;
}

using Kern = void (*)(const TraceArgs);
// One trace_kernel instantiation and its template arguments as OPTB_PLAN_* bits (what optb_trace_plan reports)
struct KernPick { Kern kern; uint32_t bits; };
template <bool SMEM, bool SERIAL, int BOXES, bool ASPH, bool SPLIT, bool FLAG = false, bool BRENT = false, bool PASSK = false,
          bool SWEEP = false>
KernPick pick() {
  return {trace_kernel<SMEM, SERIAL, BOXES, ASPH, SPLIT, FLAG, BRENT, PASSK, SWEEP>,
          (SMEM ? OPTB_PLAN_SMEM : 0u) | (SERIAL ? OPTB_PLAN_SERIAL : 0u) | ((uint32_t)BOXES << OPTB_PLAN_BOX_SHIFT) |
              (ASPH ? OPTB_PLAN_ASPH : 0u) | (SPLIT ? OPTB_PLAN_SPLIT : 0u) | (FLAG ? OPTB_PLAN_FLAG : 0u) |
              (BRENT ? OPTB_PLAN_BRENT : 0u) | (PASSK ? OPTB_PLAN_PASSK : 0u) | (SWEEP ? OPTB_PLAN_SWEEP : 0u)};
}
// The parallel-path kinds, indexed by [box mode][aspheres][split]; SWEEP: each lane on its root's configuration
template <bool SMEM, bool SWEEP = false>
KernPick parallel_kernel(int boxmode, bool asph, bool split) {
#define OPTB_K(B, A, P) pick<SMEM, false, B, A, P, false, false, false, SWEEP>()
#define OPTB_KROW(B) {{OPTB_K(B, false, false), OPTB_K(B, false, true)}, {OPTB_K(B, true, false), OPTB_K(B, true, true)}}
  static const KernPick k[3][2][2] = {OPTB_KROW(0), OPTB_KROW(1), OPTB_KROW(2)};
#undef OPTB_KROW
#undef OPTB_K
  return k[boxmode][asph ? 1 : 0][split ? 1 : 0];
}
// The general kind (box walk, aspheres, split) with one of the options only it carries
template <bool SERIAL, bool FLAG, bool BRENT, bool PASSK>
KernPick general_kernel(bool smem) {
  return smem ? pick<true, SERIAL, 1, true, true, FLAG, BRENT, PASSK>() : pick<false, SERIAL, 1, true, true, FLAG, BRENT, PASSK>();
}
// The trace_kernel instantiation that runs a trace. Sweep scenes read their tables from global memory. The
// family-serial path, the two diagnostics modes (params.reference_roots: brentq_dev roots; params.flag_ambiguity: the
// A.9 pass at every pop) and pass-through leaves (OPTB_I_PASS) only exist in the general kind.
KernPick select_kernel(const optb_scene* scene, const optb_params* prm, bool serial, bool split) {
  // box mode: 0 none, 1 pre-order walk with culling, 2 walk + lattice windows (scenes with OPTB_G_GRID groups)
  const int boxmode = !scene->has_boxes ? 0 : (scene->has_grid ? 2 : 1);
  const bool smem = scene->in_smem, asph = scene->has_asph;
  if (scene->n_cfg && serial) return pick<false, true, 1, true, true, false, false, false, true>();
  if (scene->n_cfg)
    return scene->has_pass ? pick<false, false, 1, true, true, false, false, true, true>()
                           : parallel_kernel<false, true>(boxmode, asph, split);
  if (prm->reference_roots)
    return serial ? general_kernel<true, false, true, false>(smem) : general_kernel<false, false, true, false>(smem);
  if (prm->flag_ambiguity) return general_kernel<false, true, false, false>(smem);
  if (serial) return general_kernel<true, false, false, false>(smem);
  if (scene->has_pass) return general_kernel<false, false, false, true>(smem);
  return smem ? parallel_kernel<true>(boxmode, asph, split) : parallel_kernel<false>(boxmode, asph, split);
}

// What a trace launches: the kernel, its OPTB_PLAN_* bits, the dynamic shared memory of every launch and the
// resident CTAs per SM at that size. trace_impl and optb_trace_plan both take it from launch_plan.
struct LaunchPlan { KernPick k; uint32_t smem; int occ; };
}  // namespace

// Largest static shared memory over the trace kernels that stage the blob in shared memory (every kind a scene that
// scene_alloc puts in shared memory can be traced with) and the family-serial sweep kind: the part of the opt-in window
// that is not the blob's or the histograms'.
static cudaError_t smem_static_max(size_t* out) {
  std::vector<Kern> ks;
  for (int b = 0; b < 3; b++)
    for (int a = 0; a < 2; a++)
      for (int p = 0; p < 2; p++) ks.push_back(parallel_kernel<true>(b, a, p).kern);
  ks.push_back(general_kernel<false, false, true, false>(true).kern);
  ks.push_back(general_kernel<true, false, true, false>(true).kern);
  ks.push_back(general_kernel<false, true, false, false>(true).kern);
  ks.push_back(general_kernel<true, false, false, false>(true).kern);
  ks.push_back(general_kernel<false, false, false, true>(true).kern);
  ks.push_back(pick<false, true, 1, true, true, false, false, false, true>().kern);
  size_t m = 0;
  for (Kern k : ks) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, (const void*)k);
    if (e != cudaSuccess) return e;
    m = std::max(m, fa.sharedSizeBytes);
  }
  *out = m;
  return cudaSuccess;
}

// The kernel of a trace with these options and its launch configuration. Sets the kernel's dynamic shared-memory
// attribute (a host call; nothing is enqueued): a plan CUDA refuses fails here, in the query as in the trace.
static int launch_plan(optb_ctx* ctx, const optb_scene* scene, const optb_params* prm, bool serial, bool split,
                       bool hist_smem, LaunchPlan* lp) {
  lp->k = select_kernel(scene, prm, serial, split);
  if (hist_smem) lp->k.bits |= OPTB_PLAN_HIST_SMEM;
  lp->smem = scene->in_smem ? scene->smem_bytes : (hist_smem ? scene->smem_bytes : 0);
  const Kern kern = lp->k.kern;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<uint32_t>(lp->smem, 1024)), "smem attr");
  lp->occ = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&lp->occ, kern, kBlock, lp->smem), "occupancy");
  if (lp->occ < 1) lp->occ = 1;
  return 0;
}

// The checks of a trace's arguments that do not read the result buffers (optb_trace_plan runs them too).
static int check_trace_args(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* prm) {
  if (rays->n >= 0xffffffffll) return fail(ctx, -7, "at most 2^32-1 rays per call");
  // a sweep scene traces every ray through every configuration: root k * rays.n + r = ray r in configuration k
  const long long n_roots = scene->n_cfg ? rays->n * scene->n_cfg : rays->n;
  if (scene->n_cfg) {
    if (n_roots >= 0xffffffffll) return fail(ctx, -7, "sweep: n_configs * rays.n must stay below 2^32");
    // the family-serial sweep: a family column on a scene whose caps may bind
    const bool serial_sweep = rays->family && scene->n_caps > 0 && !prm->caps_slack;
    if (needs_serial(scene, rays, prm) && !serial_sweep)
      return fail(ctx, -7, "sweep: the scene has interact caps; set params.caps_slack, or give rays.family for the "
                           "family-serial sweep");
    if (prm->flag_ambiguity || prm->reference_roots)
      return fail(ctx, -7, "sweep: flag_ambiguity and reference_roots are not available on sweep scenes");
    if (rays->family && !serial_sweep) return fail(ctx, -7, "sweep: rays.family must be NULL (every root is its own family)");
    if (serial_sweep && (long long)prm->n_families * scene->n_cfg >= 0x7fffffffll)
      return fail(ctx, -7, "sweep: n_configs * n_families must stay below 2^31");
  }
  // cap_counts is [n_capslots][n_families]; without a family column every initial ray is its own family (column
  // index = ray index), so the table must have a column per ray
  if (scene->n_caps > 0 && prm->n_families < 1) return fail(ctx, -7, "scene has interact caps: cap_counts/n_families required");
  if (scene->n_caps > 0 && !rays->family && (long long)prm->n_families < n_roots)
    return fail(ctx, -7, "scene has interact caps and rays.family is NULL: n_families must be >= rays.n (times n_configs for a sweep)");
  if (needs_serial(scene, rays, prm) && prm->flag_ambiguity)
    return fail(ctx, -7, "flag_ambiguity is not available on the family-serial path (binding interact caps)");
  if (prm->reference_roots && prm->flag_ambiguity) return fail(ctx, -7, "reference_roots and flag_ambiguity are separate diagnostics modes");
  return 0;
}

extern "C" int64_t optb_workspace_bytes(const optb_scene* scene, int64_t n_rays, int64_t max_live) {
  if (!scene || n_rays < 0) return -1;
  if (scene->n_cfg) n_rays *= scene->n_cfg;  // sweep: n_rays per configuration, one root per (configuration, ray)
  // the caller may later pass chain_len > 0, so always size for the wavefront when asked for max_live > 0
  bool split = scene->max_children > 1 || max_live > 0 || scene->has_pass;
  int64_t need = (int64_t)ws_layout(n_rays, std::max<int64_t>(max_live, n_rays), split).total;
  if (scene->n_caps > 0)  // family-serial mode: max_live = total FIFO entries over all families
    need = std::max<int64_t>(need, (int64_t)serial_layout(n_rays, n_rays, std::max<int64_t>(max_live, 8 * n_rays)).total);
  return need;
}

static int trace_impl(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* prm,
                      optb_result* out, void* workspace, int64_t workspace_bytes, cudaStream_t st, uint32_t root_base,
                      bool zero_hist);

extern "C" int optb_trace(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* prm,
                          optb_result* out, void* workspace, int64_t workspace_bytes, void* stream_v) {
  if (!ctx || !scene || !rays || !prm || !out) return -1;
  return trace_impl(ctx, scene, rays, prm, out, workspace, workspace_bytes, (cudaStream_t)stream_v, 0u, true);
}

extern "C" int optb_trace_plan(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* prm,
                               int64_t out[5]) {
  if (!ctx || !scene || !rays || !prm || !out) return -1;
  cudaSetDevice(ctx->device);
  if (int rc = check_trace_args(ctx, scene, rays, prm)) return rc;
  const bool serial = needs_serial(scene, rays, prm), split = !serial && needs_wavefront(scene, prm);
  LaunchPlan lp;
  if (int rc = launch_plan(ctx, scene, prm, serial, split, prm->record_hist && scene->n_mons > 0 && scene->hist_smem, &lp))
    return rc;
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, (const void*)lp.k.kern), "kernel attributes");
  out[0] = lp.k.bits; out[1] = scene->blob_bytes; out[2] = lp.smem; out[3] = (int64_t)fa.sharedSizeBytes;
  out[4] = (int64_t)ctx->smem_optin;
  return 0;
}

static int trace_impl(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* prm,
                      optb_result* out, void* workspace, int64_t workspace_bytes, cudaStream_t st, uint32_t root_base,
                      bool zero_hist) {
  cudaSetDevice(ctx->device);
  if (!out->counters) return fail(ctx, -7, "result.counters is required");
  if (int rc = check_trace_args(ctx, scene, rays, prm)) return rc;
  const long long n_roots = scene->n_cfg ? rays->n * scene->n_cfg : rays->n;
  if (prm->record_hits && out->hit_capacity > 0 && !out->hit_monitor && !out->hit_key) return fail(ctx, -7, "record_hits needs hit_monitor or hit_key");
  if (prm->record_hits && out->hit_key && (prm->max_trace_num > (1ll << 24) || scene->n_mons > 256))
    return fail(ctx, -7, "hit_key packs pop into 24 bits and the monitor into 8: max_trace_num <= 2^24 and <= 256 monitors");
  if (prm->flag_ambiguity && !out->root_flags) return fail(ctx, -7, "flag_ambiguity needs result.root_flags [rays.n]");
  if (scene->n_caps > 0 && !out->cap_counts) return fail(ctx, -7, "scene has interact caps: cap_counts/n_families required");
  const bool serial = needs_serial(scene, rays, prm);
  if (prm->record_hist && scene->n_mons && (!out->hist_y || (zero_hist && !out->hist_yz)))
    return fail(ctx, -7, "record_hist needs hist_y and hist_yz");
  const bool split = !serial && needs_wavefront(scene, prm);
  WsLayout L = ws_layout(n_roots, 0, false);
  long long cap = 0;
  SerialLayout SL{};
  long long n_fam = 0, qcap = 0;
  if (serial) {
    // a sweep has n_families families in each configuration: global family k * n_families + f
    n_fam = rays->family ? (long long)prm->n_families * std::max(scene->n_cfg, 1) : rays->n;
    if (n_fam < 1) return fail(ctx, -7, "n_families must be >= 1");
    const long long want = std::min<long long>(prm->max_trace_num + 2, 1ll << 20);
    const size_t fixed = serial_layout(n_roots, n_fam, 1).total;
    if ((size_t)workspace_bytes <= fixed) return fail(ctx, -8, "workspace too small (see optb_workspace_bytes)");
    long long lo = 1, hi = std::max<long long>(want, 2) * n_fam;
    while (lo < hi) {
      long long mid = lo + (hi - lo + 1) / 2;
      if ((int64_t)serial_layout(n_roots, n_fam, mid).total <= workspace_bytes) lo = mid; else hi = mid - 1;
    }
    qcap = std::min<long long>(lo / n_fam, want);
    if (qcap < 4) return fail(ctx, -8, "workspace too small for the per-family FIFO (see optb_workspace_bytes)");
    SL = serial_layout(n_roots, n_fam, qcap * n_fam);
    L.hdr = SL.hdr;
  } else if (split) {
    // find the largest wavefront capacity the given workspace supports
    if (workspace_bytes < (int64_t)ws_layout(n_roots, n_roots, true).total) return fail(ctx, -8, "workspace too small (see optb_workspace_bytes)");
    // upper end of the search: what the workspace could hold at ~100 B per live ray (far above the real cost of
    // ~540 B), so the capacity is set by the caller's workspace and never by the size of the batch: one initial ray
    // through cascaded beam splitters may need thousands of live rays (the reference allows 2000 pops)
    long long lo = n_roots, hi = std::max<long long>(n_roots, (long long)(workspace_bytes / 100));
    hi = std::min<long long>(hi, 0x7ffffff0ll);
    while (lo < hi) {
      long long mid = lo + (hi - lo + 1) / 2;
      if ((int64_t)ws_layout(n_roots, mid, true).total <= workspace_bytes) lo = mid; else hi = mid - 1;
    }
    cap = lo;
    L = ws_layout(n_roots, cap, true);
  } else if (workspace_bytes < (int64_t)L.total) {
    return fail(ctx, -8, "workspace too small (see optb_workspace_bytes)");
  }
  unsigned char* ws = (unsigned char*)workspace;
  Header* hdr = (Header*)(ws + L.hdr);

  CK(cudaMemsetAsync(out->counters, 0, sizeof(int64_t) * OPTB_C_COUNT, st), "memset counters");
  CK(cudaMemsetAsync(hdr, 0, sizeof(Header), st), "memset header");
  if (prm->record_hist && scene->n_mons && zero_hist) {
    CK(cudaMemsetAsync(out->hist_y, 0, sizeof(int64_t) * OPTB_HIST_BINS * hist_mons(scene), st), "memset hist");
    CK(cudaMemsetAsync(out->hist_yz, 0, sizeof(int64_t) * OPTB_HIST_BINS * OPTB_HIST_BINS * hist_mons(scene), st), "memset hist");
  }

  if (prm->flag_ambiguity) CK(cudaMemsetAsync(out->root_flags, 0, sizeof(uint32_t) * (size_t)rays->n, st), "memset root flags");
  TraceArgs a;
  memset(&a, 0, sizeof a);
  a.blob = scene->d_blob; a.blob_bytes = scene->blob_bytes; a.off = scene->off;
  a.n_nodes = scene->n_nodes; a.n_mons = scene->n_mons;
  a.in0 = *rays; a.gen0 = 1; a.n_in = n_roots; a.n_in_dev = nullptr;
  if (scene->n_cfg) { a.blob_bytes = scene->cfg_stride; a.sweep_n = (uint32_t)rays->n; a.hist_mons = hist_mons(scene); }
  a.max_trace = prm->max_trace_num; a.unit = prm->unit;
  a.rec_seg = prm->record_segments; a.rec_hit = prm->record_hits; a.rec_hist = prm->record_hist && scene->n_mons > 0;
  a.chain_len = prm->chain_len; a.n_families = prm->n_families;
  a.fam_shared = (rays->family != nullptr) || prm->caps_slack;
  a.hist_smem = a.rec_hist && scene->hist_smem;
  a.out = *out;
  a.counters = (unsigned long long*)out->counters;
  a.hdr = hdr;
  a.root_base = root_base;
  a.has_boxes = scene->has_boxes;
  if (split) {
    a.w = make_raybuf(ws + L.w, 2 * cap);
    a.c = make_raybuf(ws + L.c, 2 * cap);
    a.nchild = ws + L.nchild;
    a.gen_first = (uint32_t*)(ws + L.gen_first);
    a.gen_last = (uint32_t*)(ws + L.gen_last);
  }
  LaunchPlan lp;
  if (int rc = launch_plan(ctx, scene, prm, serial, split, a.hist_smem, &lp)) return rc;
  const Kern kern = lp.k.kern;
  const uint32_t smem = lp.smem;
  const int full_grid = ctx->sm_count * lp.occ;

  unsigned long long gens = 0, launches = 0;
  long long n_in = n_roots;
  if (serial && n_in > 0) {
    unsigned int* off = (unsigned int*)(ws + SL.off);
    unsigned int* cursor = (unsigned int*)(ws + SL.cursor);
    uint32_t* roots = (uint32_t*)(ws + SL.roots);
    CK(cudaMemsetAsync(off, 0, (size_t)(n_fam + 2) * 4, st), "memset family offsets");
    CK(cudaMemsetAsync(cursor, 0, (size_t)(n_fam + 1) * 4, st), "memset family cursors");
    const int g = (int)std::min<long long>(full_grid * 4, (n_in + 255) / 256);
    const uint32_t n_cfg_rays = (uint32_t)rays->n;
    if (scene->n_cfg) fam_count_sweep_kernel<<<g, 256, 0, st>>>(rays->family, n_in, n_cfg_rays, prm->n_families, off);
    else fam_count_kernel<<<g, 256, 0, st>>>(rays->family, n_in, off);
    scan_sums_kernel<<<1, 1024, 0, st>>>(off, (int)(n_fam + 1), hdr, a.counters, 0xffffffffu);  // exclusive, in place
    if (scene->n_cfg) fam_scatter_sweep_kernel<<<g, 256, 0, st>>>(rays->family, n_in, n_cfg_rays, prm->n_families, off, cursor, roots);
    else fam_scatter_kernel<<<g, 256, 0, st>>>(rays->family, n_in, off, cursor, roots);
    a.fam_off = off; a.fam_roots = roots; a.qcap = (uint32_t)qcap;
    if (scene->n_cfg) a.n_families = (int)n_fam;  // cap_counts [n_capslots][n_configs * n_families]
    a.w = make_raybuf(ws + SL.ring, qcap * n_fam);
    a.fam_shared = 0;
    a.n_in = n_fam;
    void* kargs[] = {(void*)&a};
    int grid = (int)std::min<long long>(full_grid, (n_fam + kBlock - 1) / kBlock);
    CK(cudaLaunchKernel((const void*)kern, dim3(grid), dim3(kBlock), kargs, smem, st), "launch trace_kernel (family-serial)");
    launches += 4; gens = 1;
    n_in = 0;
  }
  int key_bits = 1;
  while ((1ll << key_bits) < 2ll * std::max(scene->n_leaves, 1)) key_bits++;
  while (n_in > 0) {
    if (split && !a.gen0 && n_in >= 2048 && n_in < 0x7fffffffll) {
      uint32_t* iota = (uint32_t*)(ws + L.iota);
      uint32_t* perm = (uint32_t*)(ws + L.perm);
      uint32_t* key_dense = (uint32_t*)(ws + L.key_dense);
      sort_prep_kernel<<<std::min(full_grid * 4, (int)((n_in + 255) / 256)), 256, 0, st>>>(iota, key_dense, a.w.key, a.w.rk, a.slot, n_in, key_bits);
      size_t tb = L.cub_bytes;
      CK(cub::DeviceRadixSort::SortPairs(ws + L.cub, tb, (const uint32_t*)key_dense, (uint32_t*)(ws + L.key_sorted),
                                         (const uint32_t*)iota, perm, (int)n_in, 0, key_bits + 1, st), "radix sort");
      a.perm = perm;
      launches += 4;
    } else {
      a.perm = nullptr;
    }
    // Small wavefronts: the host round trip per generation (read the header, synchronise) costs more than the
    // generation itself, so up to kUnseen further generations are enqueued without knowing their size. They take
    // it from the header (at most twice the previous one, which bounds the grids) and are no-ops once the
    // wavefront has died. Sorting needs the size on the host; the bound keeps these below the sort threshold.
    constexpr int kUnseen = 8;
    int unseen_left = 0;
    if (split) {
      long long bound = n_in;
      while (unseen_left < kUnseen && 2 * bound < 2048 && 2 * bound <= cap) { bound *= 2; unseen_left++; }
    }
    long long bound = n_in;
    for (int u = 0; u <= unseen_left; u++) {
      const bool unseen = u > 0;
      if (unseen) { bound *= 2; a.perm = nullptr; }
      long long want = (bound + kBlock - 1) / kBlock;
      int grid = (int)std::min<long long>(full_grid, want);
      a.n_in = bound;
      a.n_in_dev = unseen ? &hdr->n_next : nullptr;
      void* kargs[] = {(void*)&a};
      CK(cudaLaunchKernel((const void*)kern, dim3(grid), dim3(kBlock), kargs, smem, st), "launch trace_kernel");
      launches++; gens++;
      if (!split) break;
      int ntiles = (int)((bound + kTile - 1) / kTile);
      unsigned int* sums = (unsigned int*)(ws + L.sums);
      tile_sums_kernel<<<ntiles, kScanBlock, 0, st>>>(a.nchild, bound, sums, unseen ? hdr : nullptr);
      scan_sums_kernel<<<1, 1024, 0, st>>>(sums, ntiles, hdr, a.counters, (unsigned int)std::min<long long>(cap, 0xffffffffll), unseen);
      // the children just written to a.c become the next generation's source; the other buffer is free again
      uint32_t* slot_next = (uint32_t*)(ws + ((gens & 1) ? L.slot_a : L.slot_b));
      slots_kernel<<<ntiles, kScanBlock, 0, st>>>(a.nchild, bound, sums, slot_next, hdr, unseen);
      const int mgrid = std::min(full_grid * 2, std::max(1, (int)((2 * bound + 255) / 256)));
      mark_kernel<<<mgrid, 256, 0, st>>>(a.c.key, slot_next, hdr, (uint32_t*)a.gen_first, (uint32_t*)a.gen_last);
      rank_kernel<<<mgrid, 256, 0, st>>>(a.c.key, a.c.rk, slot_next, hdr, a.gen_first, a.gen_last);
      std::swap(a.w, a.c);
      a.slot = slot_next;
      launches += 5;
      a.gen0 = 0;
    }
    if (!split) break;
    a.n_in_dev = nullptr;
    CK(cudaMemcpyAsync(ctx->h_hdr, hdr, sizeof(Header), cudaMemcpyDeviceToHost, st), "read header");
    CK(cudaStreamSynchronize(st), "sync generation");
    n_in = ((Header*)ctx->h_hdr)->n_next;
  }
  if (prm->flag_ambiguity && rays->n > 0) {
    count_flags_kernel<<<(int)std::min<long long>((rays->n + 255) / 256, (long long)full_grid * 4), 256, 0, st>>>(out->root_flags, rays->n, a.counters);
    launches++;
  }
  finish_kernel<<<1, 1, 0, st>>>(a.counters, gens, launches + 1, hdr);
  CK(cudaGetLastError(), "kernel launch");
  cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &capturing);
  if (capturing == cudaStreamCaptureStatusNone) {  // (a captured event could not be waited on when the scene is released;
    CK(cudaEventRecord(scene->last_use, st), "record scene use");  //  the owner of a graph synchronises before that)
    const_cast<optb_scene*>(scene)->used = true;
  }
  return 0;
}

namespace {
// Bump allocator over the optb_trace_host arena. With no base it only measures: the same carve run once without a
// base and once over an arena of the measured size takes the same offsets.
struct ArenaCursor {
  unsigned char* base; size_t off;
  void* take(size_t bytes) { size_t o = align_up(off, 256); off = o + bytes; return base ? base + o : nullptr; }
};
}  // namespace

// optb_trace_host in chunks of `chunk` rays over three streams: the host->device copy of chunk c+1, the trace of
// chunk c and the device->host copy of chunk c-1 overlap (PCIe is full duplex). Rows of chunk c land behind the rows
// of chunks < c; row keys stay global through root_base. chunk >= rays.n is the one-shot trace: one result set of the
// caller's capacity, nothing overlapped. `live`: the live-ray budget of a splitting scene. Returns 1 when one of
// several chunks overflowed its (estimated) share of the result capacity: the caller then repeats the whole batch as
// one chunk.
static int trace_host(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* prm,
                      optb_result* out, int64_t chunk, int64_t live) {
  cudaSetDevice(ctx->device);
  const int64_t n = rays->n, n_roots = n * std::max(scene->n_cfg, 1);
  const int nch = chunk >= n ? 1 : (int)((n + chunk - 1) / chunk);
  const bool chunked = nch > 1;
  const int64_t segcap = prm->record_segments ? out->seg_capacity : 0, hitcap = prm->record_hits ? out->hit_capacity : 0;
  auto chunk_cap = [&](int64_t total) { return chunked && total ? std::min<int64_t>(total, (int64_t)((double)total * chunk / n * 1.25) + 4096) : total; };
  const int64_t cseg = chunk_cap(segcap), chit = chunk_cap(hitcap);
  const bool serial = needs_serial(scene, rays, prm), split = needs_wavefront(scene, prm) || serial;
  const int64_t croots = std::min(chunk, n) * std::max(scene->n_cfg, 1);  // roots of the largest chunk
  const int64_t wsb = serial ? optb_workspace_bytes(scene, n, 16 * std::max<int64_t>(live, 64))
                             : (int64_t)ws_layout(croots, split ? std::max(live, croots) : 0, split).total;
  // sorted_rows: one chunk is sorted in place once its row counts are known; several chunks are each gathered into a
  // sorted copy right behind their trace, so that the copy back never waits for a later chunk's trace
  const bool sorted = prm->sorted_rows != 0, gather = sorted && chunked;
  const int64_t sortb = sorted ? optb_sort_workspace_bytes(std::max(cseg, chit)) : 0;
  const bool hist = prm->record_hist && scene->n_mons;
  const size_t hy = (size_t)hist_mons(scene) * OPTB_HIST_BINS * 8, hyz = hy * OPTB_HIST_BINS;
  // the family-serial sweep: [n_capslots][n_configs * n_families]
  const size_t capb = (size_t)scene->n_caps * std::max(prm->n_families, 1) * (rays->family ? std::max(scene->n_cfg, 1) : 1) * 4;
  if (!ctx->s_h2d) {
    CK(cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking), "stream");
    CK(cudaStreamCreateWithFlags(&ctx->s_run, cudaStreamNonBlocking), "stream");
    CK(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking), "stream");
  }
  if (ctx->h_chunk_n < (size_t)nch) {
    if (ctx->h_chunk) cudaFreeHost(ctx->h_chunk);
    ctx->h_chunk = nullptr; ctx->h_chunk_n = 0;
    CK(cudaMallocHost((void**)&ctx->h_chunk, sizeof(unsigned long long) * OPTB_C_COUNT * nch), "pinned counters");
    ctx->h_chunk_n = nch;
  }
  // full-length device input columns (chunks are slices of them); dev: the result sets the traces of even / odd
  // chunks append to; srt: their sorted copies
  optb_rays dr = *rays;
  const double* const* src_f = &rays->ox;
  const double** dst_f = &dr.ox;
  struct Col { void* dev[2]; void* srt[2]; unsigned char* host; size_t elt; int kind; };  // kind 0 seg, 1 hit
  std::vector<Col> cols;
  optb_result dv[2] = {*out, *out}, sv[2] = {*out, *out};
  int64_t *d_hy = nullptr, *d_hyz = nullptr;
  int32_t* d_caps = nullptr;
  void* ws[2] = {nullptr, nullptr};
  void* sort_ws = nullptr;
  for (int pass = 0; pass < 2; pass++) {  // pass 0 measures the carve, pass 1 takes it from an arena of that size
    ArenaCursor ac{pass ? (unsigned char*)ctx->arena : nullptr, 0};
    for (int f = 0; f < kRayF64; f++)
      dst_f[f] = src_f[f] ? (const double*)ac.take((((rays->broadcast >> f) & 1u) ? 1 : (size_t)n) * 8) : nullptr;
    if (rays->flags) dr.flags = (const uint32_t*)ac.take((size_t)n * 4);
    if (rays->family) dr.family = (const int32_t*)ac.take((size_t)n * 4);
    cols.clear();
    auto add = [&](size_t field_off, void* host_ptr, size_t elt, int64_t capn, int kind) {
      Col c{{nullptr, nullptr}, {nullptr, nullptr}, (unsigned char*)host_ptr, elt, kind};
      const bool want = host_ptr && capn;
      for (int s = 0; s < (chunked ? 2 : 1) && want; s++) {
        c.dev[s] = ac.take((size_t)capn * elt);
        if (gather) c.srt[s] = ac.take((size_t)capn * elt);
      }
      for (int s = 0; s < 2; s++) {
        *(void**)((unsigned char*)&dv[s] + field_off) = c.dev[s];
        *(void**)((unsigned char*)&sv[s] + field_off) = c.srt[s];
      }
      if (want) cols.push_back(c);
    };
#define OPTB_FIELD(name) offsetof(optb_result, name), (void*)out->name
    const size_t seg0 = offsetof(optb_result, seg_ox), hit0 = offsetof(optb_result, hit_px);
    double* const* seg_h = &out->seg_ox; double* const* hit_h = &out->hit_px;
    for (int f = 0; f < 13; f++) add(seg0 + 8 * f, seg_h[f], 8, cseg, 0);
    add(OPTB_FIELD(seg_flags), 4, cseg, 0); add(OPTB_FIELD(seg_root), 4, cseg, 0);
    add(OPTB_FIELD(seg_pop), 4, cseg, 0); add(OPTB_FIELD(seg_leaf), 4, cseg, 0);
    add(OPTB_FIELD(hit_monitor), 4, chit, 1); add(OPTB_FIELD(hit_root), 4, chit, 1); add(OPTB_FIELD(hit_pop), 4, chit, 1);
    for (int f = 0; f < 10; f++) add(hit0 + 8 * f, hit_h[f], 8, chit, 1);
    add(OPTB_FIELD(hit_key), 8, chit, 1);
#undef OPTB_FIELD
    if (hist) { d_hy = (int64_t*)ac.take(hy); d_hyz = (int64_t*)ac.take(hyz); }
    if (capb) d_caps = (int32_t*)ac.take(capb);
    for (int s = 0; s < (chunked ? 2 : 1); s++) {
      dv[s].seg_capacity = cseg; dv[s].hit_capacity = chit;
      dv[s].hist_y = d_hy; dv[s].hist_yz = d_hyz; dv[s].cap_counts = d_caps; dv[s].root_flags = nullptr;
      dv[s].counters = (int64_t*)ac.take(OPTB_C_COUNT * 8);
      ws[s] = ac.take((size_t)wsb);
    }
    if (sortb) sort_ws = ac.take((size_t)sortb);
    if (pass == 0 && ctx->arena_bytes < ac.off) {
      if (ctx->arena) cudaFree(ctx->arena);
      ctx->arena = nullptr; ctx->arena_bytes = 0;
      CK(cudaMalloc(&ctx->arena, ac.off), "cudaMalloc(arena)");
      ctx->arena_bytes = ac.off;
    }
  }
  int end_bit = 33;  // keys are root << 32 | ...: sort only the bits a root index of this batch can occupy
  while (end_bit < 64 && (1ull << (end_bit - 32)) <= (unsigned long long)n_roots) end_bit++;
  struct Events {  // destroyed on every exit path
    std::vector<cudaEvent_t> v;
    explicit Events(int n) : v(n) { for (auto& e : v) cudaEventCreateWithFlags(&e, cudaEventDisableTiming); }
    ~Events() { for (auto& e : v) cudaEventDestroy(e); }
    cudaEvent_t& operator[](int i) { return v[i]; }
  } ev_in(1), ev_h2d(nch), ev_run(nch), ev_d2h(nch);
  // the call comes after the caller's earlier work on the legacy default stream and on every blocking stream
  CK(cudaEventRecord(ev_in[0], 0), "event");
  CK(cudaStreamWaitEvent(ctx->s_h2d, ev_in[0], 0), "wait");
  CK(cudaStreamWaitEvent(ctx->s_run, ev_in[0], 0), "wait");
  if (hist) {
    CK(cudaMemsetAsync(d_hy, 0, hy, ctx->s_run), "memset hist");
    CK(cudaMemsetAsync(d_hyz, 0, hyz, ctx->s_run), "memset hist");
  }
  if (capb && out->cap_counts) CK(cudaMemcpyAsync(d_caps, out->cap_counts, capb, cudaMemcpyHostToDevice, ctx->s_h2d), "H2D caps");
  else if (capb) CK(cudaMemsetAsync(d_caps, 0, capb, ctx->s_h2d), "memset caps");  // no table given: every family starts at zero
  unsigned long long tot[OPTB_C_COUNT] = {0};
  int64_t seg_off = 0, hit_off = 0;
  bool chunk_overflow = false;
  int rc = 0;
  auto drain = [&](int k) -> int {
    CK(cudaEventSynchronize(ev_run[k]), "sync chunk");
    const unsigned long long* hc = ctx->h_chunk + (size_t)k * OPTB_C_COUNT;
    if (chunked && (hc[OPTB_C_STATUS] & (OPTB_ST_SEG_OVERFLOW | OPTB_ST_HIT_OVERFLOW))) chunk_overflow = true;
    int64_t rows[2] = {std::min<int64_t>((int64_t)hc[OPTB_C_SEGMENTS], cseg), std::min<int64_t>((int64_t)hc[OPTB_C_HITS], chit)};
    int64_t room[2] = {segcap - seg_off, hitcap - hit_off};
    for (int kind = 0; kind < 2; kind++)
      if (rows[kind] > room[kind]) { rows[kind] = std::max<int64_t>(room[kind], 0); tot[OPTB_C_STATUS] |= kind ? OPTB_ST_HIT_OVERFLOW : OPTB_ST_SEG_OVERFLOW; }
    if (sorted && !gather)
      if (int src = sort_rows_dev(ctx, &dv[0], nullptr, rows[0], rows[1], nullptr, sort_ws, sortb, ctx->s_d2h, end_bit)) return src;
    for (auto& c : cols) {
      const int64_t r = rows[c.kind], off = c.kind ? hit_off : seg_off;
      if (r > 0) CK(cudaMemcpyAsync(c.host + (size_t)off * c.elt, gather ? c.srt[k & 1] : c.dev[k & 1], (size_t)r * c.elt, cudaMemcpyDeviceToHost, ctx->s_d2h), "D2H rows");
    }
    CK(cudaEventRecord(ev_d2h[k], ctx->s_d2h), "event");
    seg_off += rows[0];
    hit_off += rows[1];
    for (int q = 0; q < OPTB_C_COUNT; q++)
      tot[q] = q == OPTB_C_STATUS ? tot[q] | hc[q] : q == OPTB_C_GENERATIONS ? std::max(tot[q], hc[q]) : tot[q] + hc[q];
    return 0;
  };
  for (int c = 0; c < nch && !rc; c++) {
    const int64_t lo = (int64_t)c * chunk, m = std::min<int64_t>(chunk, n - lo);
    optb_rays cr = dr;
    cr.n = m;
    const double** cf = &cr.ox;
    for (int f = 0; f < kRayF64; f++) {
      if (!src_f[f]) continue;
      const bool bc = (rays->broadcast >> f) & 1u;  // one value for all rays: staged with the first chunk
      if (!bc) cf[f] += lo;
      if (!bc || c == 0) CK(cudaMemcpyAsync((void*)cf[f], src_f[f] + (bc ? 0 : lo), (bc ? 1 : (size_t)m) * 8, cudaMemcpyHostToDevice, ctx->s_h2d), "H2D rays");
    }
    if (cr.flags) { cr.flags += lo; CK(cudaMemcpyAsync((void*)cr.flags, rays->flags + lo, (size_t)m * 4, cudaMemcpyHostToDevice, ctx->s_h2d), "H2D flags"); }
    if (cr.family) { cr.family += lo; CK(cudaMemcpyAsync((void*)cr.family, rays->family + lo, (size_t)m * 4, cudaMemcpyHostToDevice, ctx->s_h2d), "H2D family"); }
    CK(cudaEventRecord(ev_h2d[c], ctx->s_h2d), "event");
    CK(cudaStreamWaitEvent(ctx->s_run, ev_h2d[c], 0), "wait");
    if (c >= 2 && !gather) CK(cudaStreamWaitEvent(ctx->s_run, ev_d2h[c - 2], 0), "wait");  // the result set is free again
    rc = trace_impl(ctx, scene, &cr, prm, &dv[c & 1], ws[c & 1], wsb, ctx->s_run, (uint32_t)lo, false);
    if (rc) break;
    if (gather) {
      // reference order inside the chunk (chunks follow each other in ray order): keys + radix sort + one gather of
      // all columns into the sorted set, on the trace stream right behind the trace. The row counts stay on the
      // device (rows beyond them sort to the end), so nothing here waits for the host.
      if (c >= 2) CK(cudaStreamWaitEvent(ctx->s_run, ev_d2h[c - 2], 0), "wait");  // the sorted set is free again
      rc = sort_rows_dev(ctx, &dv[c & 1], &sv[c & 1], cseg, chit, (const unsigned long long*)dv[c & 1].counters, sort_ws,
                         sortb, ctx->s_run, end_bit);
      if (rc) break;
    }
    CK(cudaMemcpyAsync(ctx->h_chunk + (size_t)c * OPTB_C_COUNT, dv[c & 1].counters, OPTB_C_COUNT * 8, cudaMemcpyDeviceToHost, ctx->s_run), "D2H counters");
    CK(cudaEventRecord(ev_run[c], ctx->s_run), "event");
    if (c >= 1) rc = drain(c - 1);
  }
  if (!rc) rc = drain(nch - 1);
  if (!rc && hist) {
    if (out->hist_y) CK(cudaMemcpyAsync(out->hist_y, d_hy, hy, cudaMemcpyDeviceToHost, ctx->s_d2h), "D2H hist");
    if (out->hist_yz) CK(cudaMemcpyAsync(out->hist_yz, d_hyz, hyz, cudaMemcpyDeviceToHost, ctx->s_d2h), "D2H hist");
  }
  if (!rc && capb && out->cap_counts) CK(cudaMemcpyAsync(out->cap_counts, d_caps, capb, cudaMemcpyDeviceToHost, ctx->s_d2h), "D2H caps");
  cudaStreamSynchronize(ctx->s_h2d); cudaStreamSynchronize(ctx->s_run);
  cudaError_t e = cudaStreamSynchronize(ctx->s_d2h);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(ctx, -10, "host trace", e);
  if (chunk_overflow) return 1;
  memcpy(ctx->h_counters, tot, sizeof tot);
  if (out->counters) memcpy(out->counters, tot, sizeof tot);
  return 0;
}

extern "C" int optb_trace_host(optb_ctx* ctx, const optb_scene* scene, const optb_rays* rays, const optb_params* prm,
                               optb_result* out) {
  if (!ctx || !scene || !rays || !prm || !out) return -1;
  constexpr int64_t kChunk = 1 << 20;  // rays per chunk
  if (!needs_wavefront(scene, prm) && scene->n_caps == 0 && !scene->n_cfg && rays->n >= (3ll << 20)) {
    int rc = trace_host(ctx, scene, rays, prm, out, kChunk, 0);
    if (rc <= 0) return rc;  // 1 = a chunk outgrew its estimated share of the result capacity: rerun as one chunk
  }
  // The live ray set of a splitting scene is not known in advance: grow the workspace until it fits. A root pops at
  // most max_trace_num rays and every pop queues at most two, so 2 n max_trace_num live rays always suffice.
  const int64_t n_roots = rays->n * std::max(scene->n_cfg, 1);
  const double bound_d = 2.0 * (double)std::max<int64_t>(n_roots, 1) * (double)std::max<int64_t>(prm->max_trace_num, 1);
  const int64_t bound = bound_d > 4e9 ? (int64_t)4e9 : (int64_t)bound_d;
  const int64_t per_ray = std::max<int64_t>(4, ctx->live_per_ray_hint);
  for (int64_t live = std::min<int64_t>(std::max<int64_t>(per_ray * n_roots, 1024), std::max<int64_t>(bound, 1024));;
       live = std::min<int64_t>(live * 2, bound)) {
    int rc = trace_host(ctx, scene, rays, prm, out, rays->n, live);
    if (rc) return rc;
    if (!(ctx->h_counters[OPTB_C_STATUS] & OPTB_ST_WORK_OVERFLOW)) {
      if (n_roots > 0 && needs_wavefront(scene, prm)) ctx->live_per_ray_hint = (live + n_roots - 1) / n_roots;
      return 0;
    }
    if (live >= bound) break;
  }
  return fail(ctx, -8, "live ray set exceeds 2 * n * max_trace_num: workspace overflow");
}

extern "C" int optb_measure_fp64_peak(optb_ctx* ctx, double* tflops_out) {
  if (!ctx || !tflops_out) return -1;
  cudaSetDevice(ctx->device);
  const int blocks = ctx->sm_count * 8, threads = 256, iters = 1 << 16;
  double* d = nullptr;
  CK(cudaMalloc((void**)&d, sizeof(double) * blocks * threads), "cudaMalloc");
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  dfma_kernel<<<blocks, threads>>>(d, 1024);
  float best = 1e30f;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0);
    dfma_kernel<<<blocks, threads>>>(d, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    best = std::min(best, ms);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaError_t e = cudaGetLastError();
  cudaFree(d);
  if (e != cudaSuccess) return fail(ctx, -10, "dfma kernel", e);
  double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
  *tflops_out = flops / (best * 1e-3) / 1e12;
  return 0;
}


// ---- rows into reference order ------------------------------------------------------------------------------------
namespace {
// `d_count` (optional): the number of valid rows lives on the device (a counter of the trace that just ran on the same
// stream); rows beyond it get the largest key and sort to the end, so the host need not know the count to enqueue the sort
__global__ void seg_keys_kernel(const uint32_t* __restrict__ root, const uint32_t* __restrict__ pop, long long n,
                                const unsigned long long* __restrict__ d_count,
                                unsigned long long* __restrict__ key, uint32_t* __restrict__ idx) {
  const long long valid = d_count ? (long long)min(*d_count, (unsigned long long)n) : n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    key[i] = i < valid ? (((unsigned long long)root[i] << 32) | pop[i]) : ~0ull;
    idx[i] = (uint32_t)i;
  }
}
__global__ void hit_keys_kernel(const unsigned long long* __restrict__ packed, const uint32_t* __restrict__ root,
                                const int32_t* __restrict__ mon, const uint32_t* __restrict__ pop, long long n,
                                const unsigned long long* __restrict__ d_count,
                                unsigned long long* __restrict__ key, uint32_t* __restrict__ idx) {
  const long long valid = d_count ? (long long)min(*d_count, (unsigned long long)n) : n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    key[i] = i >= valid ? ~0ull
             : packed   ? packed[i]
                        : (((unsigned long long)root[i] << 32) | ((unsigned long long)(uint32_t)mon[i] << 24) | pop[i]);
    idx[i] = (uint32_t)i;
  }
}
// all columns of a row set in one pass: dst[c][i] = src[c][order[i]]
struct GatherCols { const void* src[20]; void* dst[20]; int elt[20]; int ncol; };
__global__ void __launch_bounds__(256) gather_rows_kernel(const GatherCols g, const uint32_t* __restrict__ order, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t j = order[i];
    for (int c = 0; c < g.ncol; c++) {
      if (g.elt[c] == 8) ((unsigned long long*)g.dst[c])[i] = ((const unsigned long long*)g.src[c])[j];
      else ((uint32_t*)g.dst[c])[i] = ((const uint32_t*)g.src[c])[j];
    }
  }
}
struct SortLayout { size_t key_a, key_b, idx_a, idx_b, tmp, cub, cub_bytes, total; };
SortLayout sort_layout(long long n) {
  SortLayout L{};
  n = std::max<long long>(n, 1);
  size_t o = 0;
  L.key_a = o; o += align_up((size_t)n * 8, 256);
  L.key_b = o; o += align_up((size_t)n * 8, 256);
  L.idx_a = o; o += align_up((size_t)n * 4, 256);
  L.idx_b = o; o += align_up((size_t)n * 4, 256);
  L.tmp = o; o += align_up((size_t)n * 8, 256);
  size_t tb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tb, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)std::min<long long>(n, 0x7fffffffll), 0, 64);
  L.cub = o; L.cub_bytes = align_up(tb + 256, 256); o += L.cub_bytes;
  L.total = o;
  return L;
}
}  // namespace

extern "C" int64_t optb_sort_workspace_bytes(int64_t n_rows) { return n_rows < 0 ? -1 : (int64_t)sort_layout(n_rows).total; }

// Sort the first n_seg / n_hit rows of `src` by their keys. dst == nullptr: in place (column by column through a
// scratch column); else every present column of src is gathered into the same column of dst in one pass.
// d_counters (optional): device counters of the trace that produced the rows; then n_seg / n_hit are capacities.
static int sort_rows_dev(optb_ctx* ctx, const optb_result* res, const optb_result* dst, int64_t n_seg, int64_t n_hit,
                         const unsigned long long* d_counters, void* workspace, int64_t workspace_bytes, cudaStream_t st,
                         int end_bit) {
  const long long nmax = std::max<long long>(n_seg, n_hit);
  if (nmax <= 0) return 0;
  if (nmax >= 0x7fffffffll) return fail(ctx, -7, "optb_sort_rows: at most 2^31-1 rows");
  const SortLayout L = sort_layout(nmax);
  if (!workspace || workspace_bytes < (int64_t)L.total) return fail(ctx, -8, "optb_sort_rows: workspace too small (optb_sort_workspace_bytes)");
  unsigned char* ws = (unsigned char*)workspace;
  unsigned long long* key_a = (unsigned long long*)(ws + L.key_a);
  unsigned long long* key_b = (unsigned long long*)(ws + L.key_b);
  uint32_t* idx_a = (uint32_t*)(ws + L.idx_a);
  uint32_t* idx_b = (uint32_t*)(ws + L.idx_b);
  void* tmp = ws + L.tmp;
  for (int pass = 0; pass < 2; pass++) {
    const long long n = pass == 0 ? n_seg : n_hit;
    if (n <= 1 && !d_counters) continue;
    if (n <= 0) continue;
    const int grid = (int)std::min<long long>((n + 255) / 256, (long long)ctx->sm_count * 16);
    if (pass == 0) {
      if (!res->seg_root || !res->seg_pop) return fail(ctx, -7, "optb_sort_rows: seg_root and seg_pop are the segment key");
      seg_keys_kernel<<<grid, 256, 0, st>>>(res->seg_root, res->seg_pop, n, d_counters ? d_counters + OPTB_C_SEGMENTS : nullptr, key_a, idx_a);
    } else {
      if (!res->hit_key && !(res->hit_root && res->hit_pop && res->hit_monitor))
        return fail(ctx, -7, "optb_sort_rows: hit_key, or hit_root + hit_monitor + hit_pop, is the monitor-row key");
      hit_keys_kernel<<<grid, 256, 0, st>>>((const unsigned long long*)res->hit_key, res->hit_root, res->hit_monitor, res->hit_pop, n,
                                            d_counters ? d_counters + OPTB_C_HITS : nullptr, key_a, idx_a);
    }
    size_t tb = L.cub_bytes;
    CK(cub::DeviceRadixSort::SortPairs(ws + L.cub, tb, (const unsigned long long*)key_a, key_b, (const uint32_t*)idx_a, idx_b,
                                       (int)n, 0, end_bit, st), "radix sort of the row keys");
    const optb_result* to = dst ? dst : res;
    GatherCols g;
    g.ncol = 0;
    auto col = [&](const void* sp, void* dp, int elt) { if (sp && dp) { g.src[g.ncol] = sp; g.dst[g.ncol] = dp; g.elt[g.ncol] = elt; g.ncol++; } };
    if (pass == 0) {
      double* const* f = &res->seg_ox; double* const* fd = &to->seg_ox;
      for (int c = 0; c < 13; c++) col(f[c], fd[c], 8);
      col(res->seg_flags, to->seg_flags, 4); col(res->seg_root, to->seg_root, 4);
      col(res->seg_pop, to->seg_pop, 4); col(res->seg_leaf, to->seg_leaf, 4);
    } else {
      double* const* f = &res->hit_px; double* const* fd = &to->hit_px;
      for (int c = 0; c < 10; c++) col(f[c], fd[c], 8);
      col(res->hit_monitor, to->hit_monitor, 4); col(res->hit_root, to->hit_root, 4);
      col(res->hit_pop, to->hit_pop, 4); col(res->hit_key, to->hit_key, 8);
    }
    if (dst) {
      if (g.ncol) gather_rows_kernel<<<grid, 256, 0, st>>>(g, idx_b, n);
      continue;
    }
    for (int c = 0; c < g.ncol; c++) {  // in place: each column through the scratch column
      GatherCols one;
      one.src[0] = g.src[c]; one.dst[0] = tmp; one.elt[0] = g.elt[c]; one.ncol = 1;
      gather_rows_kernel<<<grid, 256, 0, st>>>(one, idx_b, n);
      CK(cudaMemcpyAsync(g.dst[c], tmp, (size_t)n * g.elt[c], cudaMemcpyDeviceToDevice, st), "reorder column");
    }
  }
  CK(cudaGetLastError(), "optb_sort_rows");
  return 0;
}

extern "C" int optb_sort_rows(optb_ctx* ctx, const optb_result* res, int64_t n_seg, int64_t n_hit, void* workspace,
                              int64_t workspace_bytes, void* stream_v) {
  if (!ctx || !res) return -1;
  cudaSetDevice(ctx->device);
  return sort_rows_dev(ctx, res, nullptr, n_seg, n_hit, nullptr, workspace, workspace_bytes, (cudaStream_t)stream_v, 64);
}

// ---- monitor analytics on the rows in HBM ---------------------------------------------------------------------------
namespace {
// What the Monitor accessors derive for row j in frame f: y, z (local point . lab tangent), tY, tZ and the signed waist
// distance (NaN without hit_dx..dz, resp. hit_q_re); returns the row's bin of the 30-bin histogram of y (-1 outside).
// One definition for the grouped statistics kernels and abcd_matrix_kernel, so that the per-row values they use agree
// bit for bit.
template <class Cols>
OPTB_DEV int eval_row(const Cols& a, long long j, const optb_monitor_frame& f, double& y, double& z, double& ty,
                      double& tz, double& wd) {
  const double Px = a.px[j], Py = a.py[j], Pz = a.pz[j];
  y = dot3(Px, Py, Pz, f.tangent_y[0], f.tangent_y[1], f.tangent_y[2]);
  z = dot3(Px, Py, Pz, f.tangent_z[0], f.tangent_z[1], f.tangent_z[2]);
  ty = NAN; tz = NAN; wd = NAN;
  if (a.dx) {
    const double dx = a.dx[j], dy = a.dy[j], dz = a.dz[j];
    ty = dot3(dx, dy, dz, f.tangent_y[0], f.tangent_y[1], f.tangent_y[2]);
    tz = dot3(dx, dy, dz, f.tangent_z[0], f.tangent_z[1], f.tangent_z[2]);
    if (a.qre) {
      const double dist = a.qre[j] + a.t[j];  // Re(q_at_z(t)) = distance to the waist plane (ray.py:17-25)
      wd = dot3(dx, dy, dz, f.normal[0], f.normal[1], f.normal[2]) > 0.0 ? -dist : dist;
    }
  }
  return hist_bin(y, -f.half_width, f.half_width);
}
}  // namespace

// ---- grouped monitor analytics: every (configuration, monitor) of a result in one call, deterministically ---------
// Rows are sorted by group (stable radix sort of (group, row index)), each group's run is cut into tiles of kGroupTile
// rows, a block reduces one tile in a fixed order and a warp combines a group's tile partials in tile order. Nothing
// depends on the grid or the SM count, so the same rows in the same order give the same bits on every call.
namespace {
constexpr int kGroupThreads = 256;
constexpr int kGroupTile = kGroupThreads * 16;
constexpr long long kMaxGroups = 1ll << 20;
struct GroupArgs {
  const double *px, *py, *pz, *I, *t, *dx, *dy, *dz, *qre;
  const uint32_t* root; const int32_t* mon; const unsigned long long* key;
  long long first, n, per_config; int n_configs, n_monitors, n_groups;
  const optb_monitor_frame* frames;
  double *stats, *y, *z, *ty, *tz, *wd;
  uint32_t *key_a, *key_b, *idx_a, *idx_b, *start, *ntiles, *tile_first;
  double* part; long long part_stride;  // tile partials, slot-major: part[slot * part_stride + tile]
};
struct GroupLayout { size_t key_a, key_b, idx_a, idx_b, start, ntiles, tile_first, part, cub, cub_bytes, total;
                     long long tiles_cap; int end_bit; };
GroupLayout group_layout(long long n, int G) {
  GroupLayout L{};
  const long long nn = std::max<long long>(n, 1);
  // sum over groups of ceil(count / tile) <= floor(n / tile) + (number of non-empty groups)
  L.tiles_cap = n / kGroupTile + std::min<long long>(G, n) + 1;
  L.end_bit = 32 - __builtin_clz((unsigned)G);  // keys 0..G (G: the row belongs to no group)
  size_t o = 0;
  L.key_a = o; o += align_up((size_t)nn * 4, 256);
  L.key_b = o; o += align_up((size_t)nn * 4, 256);
  L.idx_a = o; o += align_up((size_t)nn * 4, 256);
  L.idx_b = o; o += align_up((size_t)nn * 4, 256);
  L.start = o; o += align_up((size_t)(G + 1) * 4, 256);
  L.ntiles = o; o += align_up((size_t)(G + 1) * 4, 256);
  L.tile_first = o; o += align_up((size_t)(G + 1) * 4, 256);
  L.part = o; o += align_up((size_t)L.tiles_cap * OPTB_MS_STRIDE * 8, 256);
  size_t tb_sort = 0, tb_scan = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tb_sort, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, (int)std::min<long long>(nn, 0x7fffffffll), 0, L.end_bit);
  cub::DeviceScan::ExclusiveSum(nullptr, tb_scan, (const uint32_t*)nullptr, (uint32_t*)nullptr, G + 1);
  L.cub = o; L.cub_bytes = align_up(std::max(tb_sort, tb_scan) + 256, 256); o += L.cub_bytes;
  L.total = o;
  return L;
}
OPTB_DEV bool slot_is_min(int q) { return q == OPTB_MS_MIN_Y || q == OPTB_MS_MIN_Z; }
OPTB_DEV bool slot_is_max(int q) { return q == OPTB_MS_MAX_Y || q == OPTB_MS_MAX_Z; }
// group of every row (n_groups: none; its per-row outputs are NaN here, the passes never see it) and the identity
// permutation for the sort
__global__ void group_keys_kernel(const GroupArgs a) {
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < a.n; k += (long long)gridDim.x * blockDim.x) {
    const long long j = a.first + k;
    const int m = a.mon ? a.mon[j] : (int)((a.key[j] >> 24) & 0xffu);
    long long cfg = 0;
    if (a.per_config > 0) cfg = (long long)(a.root ? a.root[j] : (uint32_t)(a.key[j] >> 32)) / a.per_config;
    const bool ok = m >= 0 && m < a.n_monitors && cfg < a.n_configs;
    a.key_a[k] = ok ? (uint32_t)(cfg * a.n_monitors + m) : (uint32_t)a.n_groups;
    a.idx_a[k] = (uint32_t)k;
    if (!ok) {
      if (a.y) a.y[k] = NAN;
      if (a.z) a.z[k] = NAN;
      if (a.ty) a.ty[k] = NAN;
      if (a.tz) a.tz[k] = NAN;
      if (a.wd) a.wd[k] = NAN;
    }
  }
}
OPTB_DEV uint32_t lower_bound_u32(const uint32_t* v, uint32_t n, uint32_t x) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (v[mid] < x) lo = mid + 1; else hi = mid; }
  return lo;
}
// start[g] = first sorted row of group g (start[G] = rows in some group); ntiles[g] = tiles of its run (ntiles[G] = 0)
__global__ void group_bounds_kernel(const GroupArgs a) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g > a.n_groups) return;
  const uint32_t s0 = lower_bound_u32(a.key_b, (uint32_t)a.n, (uint32_t)g);
  a.start[g] = s0;
  if (g == a.n_groups) { a.ntiles[g] = 0; return; }
  const uint32_t s1 = lower_bound_u32(a.key_b, (uint32_t)a.n, (uint32_t)g + 1);
  a.ntiles[g] = (s1 - s0 + kGroupTile - 1) / kGroupTile;
}
// the tile this block reduces: its group (the last g with tile_first[g] <= tile) and its sorted rows [row0, row1)
OPTB_DEV bool find_tile(const GroupArgs& a, long long tile, int& g, uint32_t& row0, uint32_t& row1) {
  if (tile >= a.tile_first[a.n_groups]) return false;
  int lo = 0, hi = a.n_groups;  // invariant: tile_first[lo] <= tile < tile_first[hi]
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (a.tile_first[mid] <= tile) lo = mid; else hi = mid; }
  g = lo;
  row0 = a.start[g] + (uint32_t)(tile - a.tile_first[g]) * kGroupTile;
  row1 = min(row0 + (uint32_t)kGroupTile, a.start[g + 1]);
  return true;
}
// first pass over one tile: the sums, extrema and histogram of the OPTB_MS_* slots, and the per-row outputs
__global__ void __launch_bounds__(kGroupThreads) group_stats_kernel(const GroupArgs a) {
  __shared__ unsigned int s_hist[OPTB_HIST_BINS];
  __shared__ double s_red[OPTB_MS_M2_Y][kGroupThreads / 32];
  int g; uint32_t row0, row1;
  const long long tile = blockIdx.x;
  if (!find_tile(a, tile, g, row0, row1)) return;
  if (threadIdx.x < OPTB_HIST_BINS) s_hist[threadIdx.x] = 0u;
  __syncthreads();
  const optb_monitor_frame f = a.frames[g];
  double v[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // count, I, y, yy, z, zz, waist, tY, tYtY
  double ymin = INFINITY, ymax = -INFINITY, zmin = INFINITY, zmax = -INFINITY;
  for (uint32_t i = row0 + threadIdx.x; i < row1; i += kGroupThreads) {
    const uint32_t k = a.idx_b[i];
    const long long j = a.first + k;
    double y, z, ty, tz, wd;
    const int b = eval_row(a, j, f, y, z, ty, tz, wd);
    v[0] += 1.0; v[1] += a.I[j]; v[2] += y; v[3] = fma(y, y, v[3]); v[4] += z; v[5] = fma(z, z, v[5]);
    ymin = fmin(ymin, y); ymax = fmax(ymax, y); zmin = fmin(zmin, z); zmax = fmax(zmax, z);
    if (b >= 0) atomicAdd(&s_hist[b], 1u);  // integer counts: the order of the atomics does not matter
    if (a.dx) {
      v[7] += ty; v[8] = fma(ty, ty, v[8]);
      if (a.qre) v[6] += wd;
    }
    if (a.y) a.y[k] = y;
    if (a.z) a.z[k] = z;
    if (a.ty) a.ty[k] = ty;
    if (a.tz) a.tz[k] = tz;
    if (a.wd) a.wd[k] = wd;
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int q = 0; q < 9; q++) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    ymin = fmin(ymin, __shfl_xor_sync(0xffffffffu, ymin, o)); ymax = fmax(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
    zmin = fmin(zmin, __shfl_xor_sync(0xffffffffu, zmin, o)); zmax = fmax(zmax, __shfl_xor_sync(0xffffffffu, zmax, o));
  }
  if (lane == 0) {  // s_red is indexed by stats slot: these are slots 0..12
    s_red[OPTB_MS_COUNT][wid] = v[0]; s_red[OPTB_MS_SUM_I][wid] = v[1]; s_red[OPTB_MS_SUM_Y][wid] = v[2];
    s_red[OPTB_MS_SUM_YY][wid] = v[3]; s_red[OPTB_MS_SUM_Z][wid] = v[4]; s_red[OPTB_MS_SUM_ZZ][wid] = v[5];
    s_red[OPTB_MS_SUM_WD][wid] = v[6]; s_red[OPTB_MS_SUM_TY][wid] = v[7]; s_red[OPTB_MS_SUM_TYTY][wid] = v[8];
    s_red[OPTB_MS_MIN_Y][wid] = ymin; s_red[OPTB_MS_MAX_Y][wid] = ymax; s_red[OPTB_MS_MIN_Z][wid] = zmin; s_red[OPTB_MS_MAX_Z][wid] = zmax;
  }
  __syncthreads();
  if (threadIdx.x < 13) {
    const int q = threadIdx.x;
    const bool mn = slot_is_min(q), mx = slot_is_max(q);
    double tot = s_red[q][0];
    for (int w = 1; w < kGroupThreads / 32; w++) tot = mn ? fmin(tot, s_red[q][w]) : mx ? fmax(tot, s_red[q][w]) : tot + s_red[q][w];
    a.part[q * a.part_stride + tile] = tot;
  }
  if (threadIdx.x < OPTB_HIST_BINS) a.part[(OPTB_MS_HIST + threadIdx.x) * a.part_stride + tile] = (double)s_hist[threadIdx.x];
  // the slots this pass does not fill (M2_*: the second pass; the two after the histogram: unused) combine to zero
  if (threadIdx.x >= 32 && threadIdx.x < 37) {
    const int r = threadIdx.x - 32;
    a.part[(r < 3 ? OPTB_MS_M2_Y + r : OPTB_MS_HIST + OPTB_HIST_BINS + r - 3) * a.part_stride + tile] = 0.0;
  }
}
// second pass over one tile: sums of squares about the group's means
__global__ void __launch_bounds__(kGroupThreads) group_m2_kernel(const GroupArgs a) {
  __shared__ double s_red[3][kGroupThreads / 32];
  int g; uint32_t row0, row1;
  const long long tile = blockIdx.x;
  if (!find_tile(a, tile, g, row0, row1)) return;
  const optb_monitor_frame f = a.frames[g];
  const double* s = a.stats + (long long)g * OPTB_MS_STRIDE;
  const double n = s[OPTB_MS_COUNT];
  const double my = s[OPTB_MS_SUM_Y] / n, mz = s[OPTB_MS_SUM_Z] / n, mty = s[OPTB_MS_SUM_TY] / n;
  double v[3] = {0.0, 0.0, 0.0};
  for (uint32_t i = row0 + threadIdx.x; i < row1; i += kGroupThreads) {
    const long long j = a.first + a.idx_b[i];
    double y, z, ty, tz, wd;
    eval_row(a, j, f, y, z, ty, tz, wd);
    y -= my; z -= mz;
    v[0] = fma(y, y, v[0]); v[1] = fma(z, z, v[1]);
    if (a.dx) {
      ty -= mty;
      v[2] = fma(ty, ty, v[2]);
    }
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < 3; q++) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    if (lane == 0) s_red[q][wid] = v[q];
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double tot = s_red[threadIdx.x][0];
    for (int w = 1; w < kGroupThreads / 32; w++) tot += s_red[threadIdx.x][w];
    a.part[(OPTB_MS_M2_Y + threadIdx.x) * a.part_stride + tile] = tot;
  }
}
// one warp per group: slots [q0, q1) of stats[g] from the group's tile partials, in tile order (lane l takes tiles
// l, l + 32, ...; then a fixed shuffle tree). A group without rows gets zeros, min +inf and max -inf.
__global__ void group_combine_kernel(const GroupArgs a, int q0, int q1) {
  const long long g = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (g >= a.n_groups) return;
  const int lane = threadIdx.x & 31;
  const uint32_t t0 = a.tile_first[g], t1 = a.tile_first[g + 1];
  for (int q = q0; q < q1; q++) {
    const bool mn = slot_is_min(q), mx = slot_is_max(q);
    double v = mn ? INFINITY : mx ? -INFINITY : 0.0;
    for (uint32_t t = t0 + lane; t < t1; t += 32) {
      const double p = a.part[q * a.part_stride + t];
      v = mn ? fmin(v, p) : mx ? fmax(v, p) : v + p;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double w = __shfl_xor_sync(0xffffffffu, v, o);
      v = mn ? fmin(v, w) : mx ? fmax(v, w) : v + w;
    }
    if (lane == 0) a.stats[g * OPTB_MS_STRIDE + q] = v;
  }
}
}  // namespace

extern "C" int64_t optb_monitor_stats_grouped_workspace_bytes(int64_t n_rows, int32_t n_groups) {
  if (n_rows < 0 || n_rows >= 0x7fffffffll || n_groups < 1 || n_groups > kMaxGroups) return -1;
  return (int64_t)group_layout(n_rows, n_groups).total;
}

extern "C" int optb_monitor_stats_grouped(optb_ctx* ctx, const optb_result* rows, int64_t first, int64_t n,
                                          int64_t rays_per_config, int32_t n_configs, int32_t n_monitors,
                                          const optb_monitor_frame* frames, double* stats, double* y, double* z,
                                          double* ty, double* tz, double* waist, void* workspace,
                                          int64_t workspace_bytes, void* stream_v) {
  if (!ctx || !rows || !frames || !stats || first < 0 || n < 0 || rays_per_config < 0 || n_configs < 1 || n_monitors < 1)
    return -1;
  if (!rows->hit_px || !rows->hit_py || !rows->hit_pz || !rows->hit_intensity || !rows->hit_t)
    return fail(ctx, -7, "optb_monitor_stats_grouped: hit_px/py/pz, hit_intensity and hit_t are required");
  if (!rows->hit_monitor && !rows->hit_key)
    return fail(ctx, -7, "optb_monitor_stats_grouped: the monitor of a row needs hit_monitor or hit_key");
  if (rays_per_config > 0 && !rows->hit_root && !rows->hit_key)
    return fail(ctx, -7, "optb_monitor_stats_grouped: the configuration of a row needs hit_root or hit_key");
  if ((ty || tz || waist) && !(rows->hit_dx && rows->hit_dy && rows->hit_dz)) return fail(ctx, -7, "optb_monitor_stats_grouped: slopes / waist distances need hit_dx, hit_dy, hit_dz");
  if (waist && !rows->hit_q_re) return fail(ctx, -7, "optb_monitor_stats_grouped: waist distances need hit_q_re");
  if (n_monitors > 256) return fail(ctx, -7, "optb_monitor_stats_grouped: at most 256 monitors");
  if ((long long)n_configs * n_monitors > kMaxGroups) return fail(ctx, -7, "optb_monitor_stats_grouped: n_configs * n_monitors must be at most 2^20");
  if (n >= 0x7fffffffll) return fail(ctx, -7, "optb_monitor_stats_grouped: at most 2^31-1 rows");
  const int G = n_configs * n_monitors;
  const GroupLayout L = group_layout(n, G);
  if (!workspace || workspace_bytes < (int64_t)L.total)
    return fail(ctx, -7, "optb_monitor_stats_grouped: workspace too small (optb_monitor_stats_grouped_workspace_bytes)");
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream_v;
  unsigned char* ws = (unsigned char*)workspace;
  GroupArgs a;
  a.px = rows->hit_px; a.py = rows->hit_py; a.pz = rows->hit_pz; a.I = rows->hit_intensity; a.t = rows->hit_t;
  a.dx = rows->hit_dx && rows->hit_dy && rows->hit_dz ? rows->hit_dx : nullptr; a.dy = rows->hit_dy; a.dz = rows->hit_dz;
  a.qre = rows->hit_q_re;
  a.root = rows->hit_root; a.mon = rows->hit_monitor; a.key = (const unsigned long long*)rows->hit_key;
  a.first = first; a.n = n; a.per_config = rays_per_config; a.n_configs = n_configs; a.n_monitors = n_monitors; a.n_groups = G;
  a.frames = frames;
  a.stats = stats; a.y = y; a.z = z; a.ty = ty; a.tz = tz; a.wd = waist;
  a.key_a = (uint32_t*)(ws + L.key_a); a.key_b = (uint32_t*)(ws + L.key_b);
  a.idx_a = (uint32_t*)(ws + L.idx_a); a.idx_b = (uint32_t*)(ws + L.idx_b);
  a.start = (uint32_t*)(ws + L.start); a.ntiles = (uint32_t*)(ws + L.ntiles); a.tile_first = (uint32_t*)(ws + L.tile_first);
  a.part = (double*)(ws + L.part); a.part_stride = L.tiles_cap;
  if (n > 0) {
    const int grid = (int)std::min<long long>((n + 255) / 256, (long long)ctx->sm_count * 16);
    group_keys_kernel<<<grid, 256, 0, st>>>(a);
    size_t tb = L.cub_bytes;
    CK(cub::DeviceRadixSort::SortPairs(ws + L.cub, tb, (const uint32_t*)a.key_a, a.key_b, (const uint32_t*)a.idx_a, a.idx_b,
                                       (int)n, 0, L.end_bit, st), "radix sort of the row groups");
  }
  group_bounds_kernel<<<(G + 1 + 255) / 256, 256, 0, st>>>(a);
  size_t tb = L.cub_bytes;
  CK(cub::DeviceScan::ExclusiveSum(ws + L.cub, tb, (const uint32_t*)a.ntiles, a.tile_first, G + 1, st), "scan of the tile counts");
  const long long gw = ((long long)G * 32 + 255) / 256;
  group_stats_kernel<<<(unsigned)L.tiles_cap, kGroupThreads, 0, st>>>(a);
  group_combine_kernel<<<(unsigned)gw, 256, 0, st>>>(a, 0, OPTB_MS_STRIDE);
  group_m2_kernel<<<(unsigned)L.tiles_cap, kGroupThreads, 0, st>>>(a);
  group_combine_kernel<<<(unsigned)gw, 256, 0, st>>>(a, OPTB_MS_M2_Y, OPTB_MS_HIST);
  CK(cudaGetLastError(), "optb_monitor_stats_grouped");
  return 0;
}

// ---- ABCD matrices of a sweep: the rows of (trace, configuration, ray) joined through a slot table -------------------
// Slot s = (trace * K + k) * N + r counts the rows of ray r of configuration k at the monitor in one trace and keeps the
// index of the first row it saw. A slot is read only when its count is 1, so the row it holds is the only one, whatever
// order the atomics ran in: the results depend on the rows, not on their order.
namespace {
struct AbcdRows {
  const double *px, *py, *pz, *dx, *dy, *dz, *qre, *t;  // what eval_row reads (qre = NULL: no waist distance)
  const uint32_t* root; const int32_t* mon; const unsigned long long* key;
};
struct AbcdLayout { size_t count, row, total; };
AbcdLayout abcd_layout(long long slots) {
  AbcdLayout L{};
  L.count = 0;
  L.row = align_up((size_t)slots * 4, 256);
  L.total = L.row + align_up((size_t)slots * 4, 256);
  return L;
}
AbcdRows abcd_rows(const optb_result* r) {
  AbcdRows a;
  a.px = r->hit_px; a.py = r->hit_py; a.pz = r->hit_pz; a.dx = r->hit_dx; a.dy = r->hit_dy; a.dz = r->hit_dz;
  a.qre = nullptr; a.t = r->hit_t;
  a.root = r->hit_root; a.mon = r->hit_monitor; a.key = (const unsigned long long*)r->hit_key;
  return a;
}
// the checks both entry points share; returns 0 or the fail() code
int abcd_check(optb_ctx* ctx, const char* fn, const optb_result* r, bool slopes, int monitor, long long n,
               long long n_rays, int n_configs) {
  char msg[160];
  const char* why = nullptr;
  if (!r->hit_root && !r->hit_key) why = "the configuration and ray of a row need hit_root or hit_key";
  else if (!r->hit_monitor && !r->hit_key) why = "the monitor of a row needs hit_monitor or hit_key";
  else if (!r->hit_px || !r->hit_py || !r->hit_pz) why = "hit_px/py/pz are required";
  else if (slopes && !(r->hit_dx && r->hit_dy && r->hit_dz)) why = "hit_dx/dy/dz are required";
  else if (monitor < 0 || monitor > 255) why = "monitor index outside [0, 256)";
  else if (2 * (long long)n_configs * n_rays >= (1ll << 32)) why = "2 * n_configs * n_rays must stay below 2^32";
  else if (n >= 0x7fffffffll) why = "at most 2^31-1 rows";
  if (!why) return 0;
  snprintf(msg, sizeof msg, "%s: %s", fn, why);
  return fail(ctx, -7, msg);
}
// slot of every row of `monitor` in a trace of `per_config` roots per configuration, `first_trace` the slot trace of
// root offset 0 (sweep A: nominal 0, shifted 1 with per_config = 2N; sweep B: 2 with per_config = N); `n_traces` limits
// the traces kept (the pivots keep only the nominal rows)
__global__ void abcd_scatter_kernel(const AbcdRows a, long long n, int monitor, long long n_rays, int n_configs,
                                    long long per_config, int first_trace, int n_traces, uint32_t* count, uint32_t* row) {
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    const int m = a.mon ? a.mon[j] : (int)((a.key[j] >> 24) & 0xffu);
    if (m != monitor) continue;
    const long long root = a.root ? (long long)a.root[j] : (long long)(a.key[j] >> 32);
    const long long k = root / per_config, rr = root - k * per_config;
    const int tr = first_trace + (int)(rr / n_rays);
    if (k >= n_configs || tr >= n_traces) continue;
    const long long s = ((long long)tr * n_configs + k) * n_rays + rr % n_rays;
    if (atomicAdd(&count[s], 1u) == 0u) row[s] = (uint32_t)j;
  }
}
OPTB_DEV unsigned long long f64_bits(double v) { return (unsigned long long)__double_as_longlong(v); }
__global__ void abcd_pivots_kernel(const AbcdRows a, long long n_rays, int n_configs, const uint32_t* count,
                                   const uint32_t* row, double* pivots, unsigned long long* first_bad) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // k * N + r
  if (i >= (long long)n_configs * n_rays) return;
  const long long r = i % n_rays;
  const bool one = count[i] == 1u, ref = count[r] == 1u;
  bool bad = !one;
  if (i < n_rays) {
    double P[3] = {NAN, NAN, NAN};
    if (one) {
      const uint32_t j = row[i];
      P[0] = a.px[j]; P[1] = a.py[j]; P[2] = a.pz[j];
    }
    pivots[3 * r + 0] = P[0]; pivots[3 * r + 1] = P[1]; pivots[3 * r + 2] = P[2];
  } else if (one && ref) {
    const uint32_t j = row[i], j0 = row[r];
    bad = f64_bits(a.px[j]) != f64_bits(a.px[j0]) || f64_bits(a.py[j]) != f64_bits(a.py[j0]) ||
          f64_bits(a.pz[j]) != f64_bits(a.pz[j0]);
  }
  if (bad) atomicMin(first_bad, (unsigned long long)i);   // -1 (all ones) loses to every index
}
__global__ void abcd_matrix_kernel(const AbcdRows a, const AbcdRows b, long long n_rays, int n_configs,
                                   const optb_monitor_frame* frames, double disp, double rot, const uint32_t* count,
                                   const uint32_t* row, double* abcd, int32_t* counts) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // k * N + r
  const long long KN = (long long)n_configs * n_rays;
  if (i >= KN) return;
  const uint32_t c0 = count[i], c1 = count[KN + i], c2 = count[2 * KN + i];
  counts[3 * i + 0] = (int32_t)c0; counts[3 * i + 1] = (int32_t)c1; counts[3 * i + 2] = (int32_t)c2;
  double* M = abcd + 4 * i;
  if (c0 != 1u || c1 != 1u || c2 != 1u) {
    M[0] = NAN; M[1] = NAN; M[2] = NAN; M[3] = NAN;
    return;
  }
  const optb_monitor_frame f = frames[i / n_rays];
  double y0, y1, y2, t0, t1, t2, z, tz, wd;
  eval_row(a, (long long)row[i], f, y0, z, t0, tz, wd);
  eval_row(a, (long long)row[KN + i], f, y1, z, t1, tz, wd);
  eval_row(b, (long long)row[2 * KN + i], f, y2, z, t2, tz, wd);
  M[0] = __ddiv_rn(__dsub_rn(y1, y0), disp); M[1] = __ddiv_rn(__dsub_rn(y2, y0), rot);
  M[2] = __ddiv_rn(__dsub_rn(t1, t0), disp); M[3] = __ddiv_rn(__dsub_rn(t2, t0), rot);
}
}  // namespace

extern "C" int64_t optb_sweep_abcd_workspace_bytes(int64_t n_rays, int32_t n_configs) {
  if (n_rays < 1 || n_configs < 1 || 2 * (long long)n_configs * n_rays >= (1ll << 32)) return -1;
  return (int64_t)abcd_layout(3ll * n_configs * n_rays).total;
}

extern "C" int optb_sweep_abcd_pivots(optb_ctx* ctx, const optb_result* rows, int64_t n, int64_t n_rays,
                                      int32_t n_configs, int32_t mon0, double* pivots, int64_t* first_bad,
                                      void* workspace, int64_t workspace_bytes, void* stream_v) {
  if (!ctx || !rows || !pivots || !first_bad || n < 0 || n_rays < 1 || n_configs < 1) return -1;
  if (int rc = abcd_check(ctx, "optb_sweep_abcd_pivots", rows, false, mon0, n, n_rays, n_configs)) return rc;
  const long long KN = (long long)n_configs * n_rays;
  const AbcdLayout L = abcd_layout(KN);
  if (!workspace || workspace_bytes < (int64_t)L.total)
    return fail(ctx, -7, "optb_sweep_abcd_pivots: workspace too small (optb_sweep_abcd_workspace_bytes)");
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream_v;
  unsigned char* ws = (unsigned char*)workspace;
  uint32_t *count = (uint32_t*)(ws + L.count), *row = (uint32_t*)(ws + L.row);
  const AbcdRows a = abcd_rows(rows);
  CK(cudaMemsetAsync(count, 0, (size_t)KN * 4, st), "optb_sweep_abcd_pivots: clearing the slots");
  CK(cudaMemsetAsync(first_bad, 0xff, sizeof(int64_t), st), "optb_sweep_abcd_pivots: clearing first_bad");
  if (n > 0) {
    const int grid = (int)std::min<long long>((n + 255) / 256, (long long)ctx->sm_count * 16);
    abcd_scatter_kernel<<<grid, 256, 0, st>>>(a, n, mon0, n_rays, n_configs, 2 * n_rays, 0, 1, count, row);
  }
  abcd_pivots_kernel<<<(unsigned)((KN + 255) / 256), 256, 0, st>>>(a, n_rays, n_configs, count, row, pivots,
                                                                    (unsigned long long*)first_bad);
  CK(cudaGetLastError(), "optb_sweep_abcd_pivots");
  return 0;
}

extern "C" int optb_sweep_abcd(optb_ctx* ctx, const optb_result* rows_a, int64_t n_a, const optb_result* rows_b,
                               int64_t n_b, int64_t n_rays, int32_t n_configs, int32_t mon1,
                               const optb_monitor_frame* frames, double disp, double rot, double* abcd, int32_t* counts,
                               void* workspace, int64_t workspace_bytes, void* stream_v) {
  if (!ctx || !rows_a || !rows_b || !frames || !abcd || !counts || n_a < 0 || n_b < 0 || n_rays < 1 || n_configs < 1)
    return -1;
  if (int rc = abcd_check(ctx, "optb_sweep_abcd", rows_a, true, mon1, n_a, n_rays, n_configs)) return rc;
  if (int rc = abcd_check(ctx, "optb_sweep_abcd", rows_b, true, mon1, n_b, n_rays, n_configs)) return rc;
  const long long KN = (long long)n_configs * n_rays;
  const AbcdLayout L = abcd_layout(3 * KN);
  if (!workspace || workspace_bytes < (int64_t)L.total)
    return fail(ctx, -7, "optb_sweep_abcd: workspace too small (optb_sweep_abcd_workspace_bytes)");
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream_v;
  unsigned char* ws = (unsigned char*)workspace;
  uint32_t *count = (uint32_t*)(ws + L.count), *row = (uint32_t*)(ws + L.row);
  const AbcdRows a = abcd_rows(rows_a), b = abcd_rows(rows_b);
  CK(cudaMemsetAsync(count, 0, (size_t)(3 * KN) * 4, st), "optb_sweep_abcd: clearing the slots");
  if (n_a > 0) {
    const int grid = (int)std::min<long long>((n_a + 255) / 256, (long long)ctx->sm_count * 16);
    abcd_scatter_kernel<<<grid, 256, 0, st>>>(a, n_a, mon1, n_rays, n_configs, 2 * n_rays, 0, 2, count, row);
  }
  if (n_b > 0) {
    const int grid = (int)std::min<long long>((n_b + 255) / 256, (long long)ctx->sm_count * 16);
    abcd_scatter_kernel<<<grid, 256, 0, st>>>(b, n_b, mon1, n_rays, n_configs, n_rays, 2, 3, count, row);
  }
  abcd_matrix_kernel<<<(unsigned)((KN + 255) / 256), 256, 0, st>>>(a, b, n_rays, n_configs, frames, disp, rot, count,
                                                                    row, abcd, counts);
  CK(cudaGetLastError(), "optb_sweep_abcd");
  return 0;
}

// ---- multi-GPU monitor merge over NCCL (loaded at run time: no link-time dependency) ------------------------------
namespace {
// the few NCCL entry points used, with the ABI of nccl.h (ncclResult_t = int, ncclUniqueId = 128 bytes by value)
struct NcclId { char internal[128]; };
struct NcclApi {
  int (*GetUniqueId)(NcclId*);
  int (*CommInitRank)(void**, int, NcclId, int);
  int (*CommDestroy)(void*);
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
  int (*GroupStart)();
  int (*GroupEnd)();
  const char* (*GetErrorString)(int);
};
constexpr int kNcclInt64 = 4, kNcclSum = 0, kNcclMax = 2;  // ncclDataType_t / ncclRedOp_t values of nccl.h
NcclApi g_nccl;
void* g_nccl_handle = nullptr;

int load_nccl(optb_ctx* ctx) {
  if (g_nccl_handle) return 0;
  void* h = nullptr;
  if (const char* p = getenv("OPTB_NCCL_LIB")) h = dlopen(p, RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);  // already in the process (e.g. torch's)
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return fail(ctx, -11, "NCCL not found: set OPTB_NCCL_LIB to libnccl.so.2");
  NcclApi a;
  a.GetUniqueId = (int (*)(NcclId*))dlsym(h, "ncclGetUniqueId");
  a.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(h, "ncclCommInitRank");
  a.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
  a.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
  a.GroupStart = (int (*)())dlsym(h, "ncclGroupStart");
  a.GroupEnd = (int (*)())dlsym(h, "ncclGroupEnd");
  a.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
  if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllReduce || !a.GroupStart || !a.GroupEnd)
    return fail(ctx, -11, "NCCL library lacks an expected symbol");
  g_nccl = a; g_nccl_handle = h;
  return 0;
}
int nccl_fail(optb_ctx* ctx, const char* what, int rc) {
  snprintf(ctx->err, sizeof ctx->err, "%s: NCCL error %d (%s)", what, rc, g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
  return -11;
}

// status word -> one slot per bit (so that a sum over ranks is an OR), generations -> their own slot (maximum)
constexpr int kMergeBits = 16;
__global__ void merge_prep_kernel(long long* counters, long long* scratch) {
  const int k = threadIdx.x;
  if (k < kMergeBits) scratch[k] = (counters[OPTB_C_STATUS] >> k) & 1;
  if (k == kMergeBits) scratch[kMergeBits] = counters[OPTB_C_GENERATIONS];
  __syncthreads();
  if (k == 0) { counters[OPTB_C_STATUS] = 0; counters[OPTB_C_GENERATIONS] = 0; }
}
__global__ void merge_post_kernel(long long* counters, const long long* scratch) {
  if (threadIdx.x == 0) {
    long long st = 0;
    for (int k = 0; k < kMergeBits; k++) if (scratch[k] > 0) st |= 1ll << k;
    counters[OPTB_C_STATUS] = st;
    counters[OPTB_C_GENERATIONS] = scratch[kMergeBits];
  }
}
}  // namespace

extern "C" int optb_comm_unique_id(optb_ctx* ctx, void* id128) {
  if (!ctx || !id128) return -1;
  if (int rc = load_nccl(ctx)) return rc;
  NcclId id;
  if (int rc = g_nccl.GetUniqueId(&id)) return nccl_fail(ctx, "ncclGetUniqueId", rc);
  memcpy(id128, &id, sizeof id);
  return 0;
}

extern "C" int optb_comm_init(optb_ctx* ctx, const void* id128, int rank, int nranks) {
  if (!ctx || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return -1;
  if (ctx->nccl_comm) return fail(ctx, -7, "communicator already initialised");
  if (int rc = load_nccl(ctx)) return rc;
  cudaSetDevice(ctx->device);
  NcclId id;
  memcpy(&id, id128, sizeof id);
  void* comm = nullptr;
  if (int rc = g_nccl.CommInitRank(&comm, nranks, id, rank)) return nccl_fail(ctx, "ncclCommInitRank", rc);
  CK(cudaMalloc((void**)&ctx->d_merge, sizeof(long long) * (kMergeBits + 1)), "cudaMalloc(merge scratch)");
  ctx->nccl_comm = comm; ctx->comm_rank = rank; ctx->comm_size = nranks;
  return 0;
}

extern "C" int optb_monitor_merge(optb_ctx* ctx, int64_t* hist_y, int64_t* hist_yz, int n_monitors, int64_t* counters,
                                  void* stream_v) {
  if (!ctx || n_monitors < 0) return -1;
  if (!ctx->nccl_comm) return fail(ctx, -7, "optb_monitor_merge: call optb_comm_init first");
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream_v;
  if (ctx->comm_size == 1) return 0;
  if (counters) merge_prep_kernel<<<1, 32, 0, st>>>((long long*)counters, ctx->d_merge);
  int rc = g_nccl.GroupStart();
  if (!rc && hist_y && n_monitors) rc = g_nccl.AllReduce(hist_y, hist_y, (size_t)n_monitors * OPTB_HIST_BINS, kNcclInt64, kNcclSum, ctx->nccl_comm, st);
  if (!rc && hist_yz && n_monitors) rc = g_nccl.AllReduce(hist_yz, hist_yz, (size_t)n_monitors * OPTB_HIST_BINS * OPTB_HIST_BINS, kNcclInt64, kNcclSum, ctx->nccl_comm, st);
  if (!rc && counters) rc = g_nccl.AllReduce(counters, counters, OPTB_C_COUNT, kNcclInt64, kNcclSum, ctx->nccl_comm, st);
  if (!rc && counters) rc = g_nccl.AllReduce(ctx->d_merge, ctx->d_merge, kMergeBits, kNcclInt64, kNcclSum, ctx->nccl_comm, st);
  if (!rc && counters) rc = g_nccl.AllReduce(ctx->d_merge + kMergeBits, ctx->d_merge + kMergeBits, 1, kNcclInt64, kNcclMax, ctx->nccl_comm, st);
  int rc2 = g_nccl.GroupEnd();
  if (rc || rc2) return nccl_fail(ctx, "ncclAllReduce", rc ? rc : rc2);
  if (counters) merge_post_kernel<<<1, 32, 0, st>>>((long long*)counters, ctx->d_merge);
  CK(cudaGetLastError(), "merge kernels");
  return 0;
}

extern "C" int optb_comm_destroy(optb_ctx* ctx) {
  if (!ctx) return -1;
  if (ctx->nccl_comm) {
    cudaSetDevice(ctx->device);
    g_nccl.CommDestroy(ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
  }
  if (ctx->d_merge) { cudaFree(ctx->d_merge); ctx->d_merge = nullptr; }
  return 0;
}
