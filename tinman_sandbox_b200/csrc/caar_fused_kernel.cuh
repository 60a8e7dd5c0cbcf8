// caar_fused_kernel.cuh — CAAR_MODE_FAST for every nlev <= 128 (an instance compiled for L levels serves any nlev <= L;
// the examples below are nlev = 72 / 128): the whole of compute_and_apply_rhs for one element in
// ONE kernel and one HBM pass (every input read once, every output written once; all 18 reference
// temporaries of PO/compute_and_apply_rhs.cpp:18-35 live in registers).
//
// Work decomposition: one THREAD-BLOCK CLUSTER per element. The column of nlev levels is cut into CL slabs, one
// CTA each (nlev = 72: three CTAs of 24 levels / 96 threads; nlev = 128: two CTAs of 64 levels / 256 threads).
// Thread t of a CTA owns level t/4 of the slab and GLL row igp = t%4, i.e. the 4 points jgp = 0..3: 32 contiguous
// bytes of every scalar level-field, 64 of (u,v). 128 registers per thread; 5 (nlev=72) or 2 (nlev=128) CTAs of
// different elements share an SM, each in its own phase.
//
// Data movement (per CTA):
//   * "early" inputs dp3d(n0), v(n0) — needed at once — are LDG.128'd straight into registers;
//   * T(n0), Qdp and the "late" inputs derived_vn0, pecnd, derived_omega_p, dp3d(nm1), T(nm1), v(nm1) are fetched by
//     ONE thread at kernel entry with eight 3-D tiled TMA copies (cp.async.bulk.tensor.3d, SASS UTMALDG.3D, 128-byte
//     swizzle) into shared memory and complete on three mbarriers while the CTA computes: no registers, no LSU, full
//     prefetch distance;
//   * every output is written IN PLACE over the late input that has the same shape
//     (vn0->vn0, pecnd->phi, omega_p->omega_p, dp3d(nm1)->dp3d(np1), T(nm1)->T(np1), v(nm1)->v(np1)) and
//     leaves the SM as six TMA tile stores (UTMASTG.3D): fully coalesced, asynchronous, no per-thread STG;
//   * the element's 2-D geometry (Dinv*rrearth, D, metdet, rmetdet, fcor, spheremp, phis: 1664 B) sits in
//     shared memory and is re-read (warp-broadcast) where used, instead of pinning 40 registers;
//   * thread 0 prefetches the early inputs and the geometry of a later element into L2 (cp.async.bulk.prefetch.L2).
//
// Math:
//   * sphere operators (PO/sphere_operators.cpp:9-129): derivative along jgp is thread-local (Dvv from the
//     constant bank); derivative along igp: one DMMA.8x8x4 per jgp column differentiates all 8 levels of the warp at
//     once and one 64-bit shuffle per value brings the (transposed) result home — see deriv_i.
//   * vertical integrals (PO:76-97, 280-312, 314-352) in scan form: warp-shuffle scans over the 8 levels of
//     a warp (lane stride 4); the per-warp totals are combined over the nlev/8 warps of the column — inside a CTA
//     through shared memory, between the CTAs of the cluster through distributed shared memory: a warp sends its
//     total row to the CTAs that need it with st.async ... mbarrier::complete_tx (SASS STAS) and the receiver
//     waits on its own mbarrier (no cluster barrier, no fence on the critical path). 3 __syncthreads in all.
//   * one reciprocal of p serves the four divisions by p (PO:219,300,333,336).
// Rounding differs from the reference by FMA contraction, scan ordering and the shared reciprocal
// (~1e-15 relative); tests/test_parity_gpu.py holds it to 1e-12 per field.
//
// EUL instances: the Eulerian vertical coordinate (rsplit == 0), see the comment at the kernel.
// Level counts up to 64 run with one CTA per element (CL = 1, at most 256 threads); see cluster_for().
#pragma once
#include <cstdio>
#include <cstdlib>

#include "caar_device.cuh"

namespace caar {
namespace {

constexpr unsigned FULL = 0xffffffffu;

// ---- TMA bulk copy + mbarrier primitives (sm_90+/sm_100a PTX) ---------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 3-D tiled TMA load: rows [row, row+box) x 16 doubles of slice `slice` of the array behind `map` -> swizzled smem
// tile. The arrays are described as [slice][row][16 doubles] (slice = element x time level ..., row = level, or level x
// component for (u,v)); rows beyond the slice's extent are zero-filled in shared memory and never read from HBM, which
// is what lets an instance compiled for L levels serve any nlev <= L.
__device__ __forceinline__ void tma_load(void* dst, const CUtensorMap* map, int row, int slice, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(0), "r"(row), "r"(slice), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
// 3-D tiled TMA store: swizzled smem tile -> rows [row, row+box) of slice `slice`; rows beyond the slice's extent
// are clipped (not written)
__device__ __forceinline__ void tma_store(const CUtensorMap* map, int row, int slice, const void* src) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(map), "r"(0),
               "r"(row), "r"(slice), "r"(smem_u32(src))
               : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ---- thread-block cluster primitives (CL = 2: the two halves of an element's column run as a CTA pair) ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init_cluster() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// Store a row into the same shared-memory location of CTA `rank` of this cluster (distributed shared memory) and
// credit its 32 bytes to that CTA's mbarrier `bar`: the receiver just waits on its own mbarrier — no cluster
// barrier, no fence on the sender (st.async ... mbarrier::complete_tx::bytes).
__device__ __forceinline__ void st_row_async_remote(const double* local, const uint64_t* bar, uint32_t rank,
                                                    const double (&x)[4]) {
  uint32_t dst, rbar;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(dst) : "r"(smem_u32(local)), "r"(rank));
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rbar) : "r"(smem_u32(bar)), "r"(rank));
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(dst),
               "d"(x[0]), "d"(x[1]), "r"(rbar)
               : "memory");
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(dst + 16),
               "d"(x[2]), "d"(x[3]), "r"(rbar)
               : "memory");
}

// 1/x to ~1 ulp: hardware 20-bit seed + two Newton steps (x is a positive, normal pressure / thickness)
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = fma(fma(-x, r, 1.0), r, r);
  r = fma(fma(-x, r, 1.0), r, r);
  return r;
}

// ---- register tiles -----------------------------------------------------------------------------------
struct Row {  // the 4 points (jgp = 0..3) of one GLL row of one level
  double x[4];
};
__device__ __forceinline__ Row ld_row(const double* p) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  Row r;
  r.x[0] = a.x; r.x[1] = a.y; r.x[2] = b.x; r.x[3] = b.y;
  return r;
}
__device__ __forceinline__ void st_row(double* p, const Row& r) {
  *reinterpret_cast<double2*>(p) = make_double2(r.x[0], r.x[1]);
  *reinterpret_cast<double2*>(p + 2) = make_double2(r.x[2], r.x[3]);
}
__device__ __forceinline__ void ld_row2(const double* p, Row& u, Row& w) {  // interleaved [jgp][2]
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double2 a = *reinterpret_cast<const double2*>(p + 2 * j);
    u.x[j] = a.x;
    w.x[j] = a.y;
  }
}
// Tiles written by TMA with SWIZZLE_128B: inside every 1024-byte block the 16-byte chunk index (address bits
// 4-6) is XORed with the 128-byte row index (bits 7-9). `sw` is this thread's byte offset of its first chunk;
// its other chunks are sw ^ 16, sw ^ 32, sw ^ 48. The 8 lanes of a quarter-warp hit 8 different chunk columns:
// conflict-free 128-bit accesses.
__device__ __forceinline__ Row ld_tile(const double* tile, uint32_t sw) {
  const char* b = reinterpret_cast<const char*>(tile);
  const double2 a = *reinterpret_cast<const double2*>(b + sw);
  const double2 c = *reinterpret_cast<const double2*>(b + (sw ^ 16));
  Row r;
  r.x[0] = a.x; r.x[1] = a.y; r.x[2] = c.x; r.x[3] = c.y;
  return r;
}
__device__ __forceinline__ void st_tile(double* tile, uint32_t sw, const Row& r) {
  char* b = reinterpret_cast<char*>(tile);
  *reinterpret_cast<double2*>(b + sw) = make_double2(r.x[0], r.x[1]);
  *reinterpret_cast<double2*>(b + (sw ^ 16)) = make_double2(r.x[2], r.x[3]);
}
__device__ __forceinline__ void ld_tile2(const double* tile, uint32_t sw, Row& u, Row& w) {  // interleaved (u,v)
  const char* b = reinterpret_cast<const char*>(tile);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double2 a = *reinterpret_cast<const double2*>(b + (sw ^ (j << 4)));
    u.x[j] = a.x;
    w.x[j] = a.y;
  }
}
__device__ __forceinline__ void st_tile2(double* tile, uint32_t sw, const Row& u, const Row& w) {
  char* b = reinterpret_cast<char*>(tile);
#pragma unroll
  for (int j = 0; j < 4; ++j) *reinterpret_cast<double2*>(b + (sw ^ (j << 4))) = make_double2(u.x[j], w.x[j]);
}

// shared-memory loads the compiler may not merge/hoist across uses (keeps the geometry out of registers)
__device__ __forceinline__ double2 lds2(const double* p) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(smem_u32(p)));
  return v;
}

// The igp derivative out[j] = sum_m Dvv[m][r] * s_m[j] (s_m: row m of this level) on the FP64 tensor core: for a
// fixed jgp j the eight levels of a warp form ONE 8x8x4 product D_j = A B_j with A[i'][m] = Dvv[m][i' & 3] (rows 4-7
// repeat rows 0-3) and B_j[m][n] = s of level n at (igp m, jgp j). In the mma.m8n8k4 fragment layout the thread
// lane = 4*level + igp holds exactly B_j[lane & 3][lane >> 2] = its own x[j], and one constant element of A. The
// result lands transposed: thread (q = lane >> 2, c = lane & 3) holds D_j[q][2c], D_j[q][2c+1] = the derivative at
// igp q & 3 of the levels 2c and 2c+1. Since the rows q and q + 4 are copies, the lanes with q < 4 hand out their even
// level and the lanes with q >= 4 their odd one, and every thread fetches its value with ONE 64-bit shuffle: 4 DMMA +
// 8 SHFL per call instead of 16 DFMA + 24 SHFL — a third of the shared-memory-pipe wavefronts of the derivative (the
// L1 data pipe is this kernel's co-limiter, DESIGN.md 5.1). A/B against the shuffle form on one box
// (profiles/r2u_mma_ab.jsonl): nlev 72 1.055 -> 1.065 of the measured peak at full clocks and 0.935 -> 1.014 on a
// power-capped GPU (~1.6 GHz), aliased time levels 0.88 -> 0.91-0.98, Eulerian nlev 72 / 128 0.931 -> 0.984 /
// 0.904 -> 0.952.
struct DerivMma {
  double a;   // A[lane >> 2][lane & 3] = Dvv[lane & 3][(lane >> 2) & 3]
  int src;    // lane that holds this thread's result
  bool odd;   // this lane hands out D[.][2c+1] (q >= 4), else D[.][2c]
};
__device__ __forceinline__ DerivMma deriv_mma_setup(const double* __restrict__ dvv, int lane) {
  DerivMma d;
  const int q = lane >> 2, c = lane & 3;
  d.a = dvv[c * 4 + (q & 3)];
  d.odd = q >= 4;
  // this thread = (level q, igp c): its row of D is c (level even) or c + 4 (level odd), its column pair is q >> 1
  d.src = ((((q & 1) ? c + 4 : c)) << 2) | (q >> 1);
  return d;
}
__device__ __forceinline__ Row deriv_i(const Row& s, const DerivMma& m) {
  Row o;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    double d0, d1;
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%4, %5};"
                 : "=d"(d0), "=d"(d1)
                 : "d"(m.a), "d"(s.x[j]), "d"(0.0), "d"(0.0));
    o.x[j] = __shfl_sync(FULL, m.odd ? d1 : d0, m.src);
  }
  return o;
}
// out[l] = sum_m Dvv[m][l] * s[m] (thread-local; Dvv from the constant bank)
__device__ __forceinline__ Row deriv_j(const Row& s, const double* __restrict__ dvv) {
  Row o;
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    double acc = dvv[0 * 4 + l] * s.x[0];
#pragma unroll
    for (int m = 1; m < 4; ++m) acc = fma(dvv[m * 4 + l], s.x[m], acc);
    o.x[l] = acc;
  }
  return o;
}

// gradient_sphere (PO/sphere_operators.cpp:9-48) for this thread's row; di = this row's Dinv*rrearth in smem,
// [jgp][2*a+b]
__device__ __forceinline__ void gradient(const Row& s, const double* di, const DerivMma& cx,
                                         const double* __restrict__ dvv, Row& g0, Row& g1) {
  const Row a = deriv_i(s, cx);   // v1[igp][jgp]
  const Row b = deriv_j(s, dvv);  // v2[igp][jgp]
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double2 d01 = lds2(di + j * 4), d23 = lds2(di + j * 4 + 2);
    g0.x[j] = fma(d01.x, a.x[j], d23.x * b.x[j]);
    g1.x[j] = fma(d01.y, a.x[j], d23.y * b.x[j]);
  }
}

// inclusive scans over the 8 levels of a warp (same igp => lane stride 4)
__device__ __forceinline__ double scan_down(double v, int lane) {  // towards larger k
#pragma unroll
  for (int d = 4; d < 32; d <<= 1) {
    const double t = __shfl_up_sync(FULL, v, d);
    if (lane >= d) v += t;
  }
  return v;
}
__device__ __forceinline__ double scan_up(double v, int lane) {  // towards smaller k
#pragma unroll
  for (int d = 4; d < 32; d <<= 1) {
    const double t = __shfl_down_sync(FULL, v, d);
    if (lane + d < 32) v += t;
  }
  return v;
}

// Sum over the warps ww in [lo, hi) of the per-warp scan totals tot[ww][r*4 + j], j = 0..3, delivered to every lane
// for its own GLL row r. Lane c (+16) sums column c of the rows lo, lo+2, ... (lo+1, lo+3, ...): one 256-byte LDS.64
// per pair of rows, the two halves meet in one xor-shuffle and every lane picks the four columns of its GLL row: about
// NWT + 10 shared-memory wavefronts per call against 40 for a butterfly over the lane bits 2..4 (which is what the
// LSU-bound Eulerian instances feel).
template <int NWT>
__device__ __forceinline__ void warp_totals(const double (*tot)[16], int lo, int hi, int lane, double (&out)[4]) {
  const int c = lane & 15, h = lane >> 4, r = lane & 3;
  double acc = 0.0, acc2 = 0.0;
#pragma unroll
  for (int k = 0; k < (NWT + 1) / 2; ++k) {  // every row is loaded (no branch between the loads), the range selects
    const int ww = 2 * k + h;
    const double x = tot[ww < NWT ? ww : NWT - 1][c];
    if (ww >= lo && ww < hi) {
      if (k & 1) acc2 += x;
      else acc += x;
    }
  }
  acc += acc2;
  acc += __shfl_xor_sync(FULL, acc, 16);
#pragma unroll
  for (int j = 0; j < 4; ++j) out[j] = __shfl_sync(FULL, acc, r * 4 + j);
}
// The same pass delivering two sums: rows [0, hi) (the carry of this warp) and all NWT rows (the column total that the
// Eulerian branch needs next): one set of loads instead of two calls. Used for columns of at most 96
// levels (NWT <= 12): A/B nlev 72 / 96 0.919 -> 0.932 / 0.930 of the measured peak, nlev 128 0.904 -> 0.899.
template <int NWT>
__device__ __forceinline__ void warp_totals_both(const double (*tot)[16], int hi, int lane, double (&pre)[4],
                                                 double (&all)[4]) {
  const int c = lane & 15, h = lane >> 4, r = lane & 3;
  double a0 = 0.0, a1 = 0.0, t0 = 0.0, t1 = 0.0;
#pragma unroll
  for (int k = 0; k < (NWT + 1) / 2; ++k) {
    const int ww = 2 * k + h;
    const double x = tot[ww < NWT ? ww : NWT - 1][c];
    if (ww < NWT) {
      if (k & 1) t1 += x;
      else t0 += x;
      if (ww < hi) {
        if (k & 1) a1 += x;
        else a0 += x;
      }
    }
  }
  a0 += a1;
  t0 += t1;
  a0 += __shfl_xor_sync(FULL, a0, 16);
  t0 += __shfl_xor_sync(FULL, t0, 16);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    pre[j] = __shfl_sync(FULL, a0, r * 4 + j);
    all[j] = __shfl_sync(FULL, t0, r * 4 + j);
  }
}

// Eulerian instances with at least this many levels per CTA issue the block's two global loads (dp3d re-read,
// eta_dot_dpdn) at its start: A/B nlev=128 (64 levels per CTA) 0.847 -> 0.861 of the measured peak, nlev=72 (24 per
// CTA) 0.878 -> 0.849 (the 16 live registers cost more there)
constexpr int EUL_HOIST_LEVELS = 56;

// CTAs per element (cluster size) for every level count with a compiled instance; 0 = none.
// Levels per CTA = nlev / cluster_for(nlev), a multiple of 8 (a warp scans 8 levels).
// nlev = 72: a cluster of three 96-thread CTAs (24 levels each); nlev = 128: a cluster of two 256-thread CTAs.
__host__ __device__ constexpr int cluster_for(int nlev) {
  return nlev == 72 ? 3 : nlev == 128 ? 2
         : (nlev >= 8 && nlev <= 64 && nlev % 8 == 0) ? 1
         : nlev == 80 ? 2 : nlev == 96 ? 3 : nlev == 112 ? 2 : nlev == 120 ? 3 : 0;
}
// The instance that serves a run-time level count: the smallest compiled level count >= nlev (0 = none: nlev > 128).
// The levels [nlev, instance) of the column are padding: their threads hold dp = 1, v = 0 and zero-filled tiles, so
// that every scan contribution from them is exactly 0, and their rows are neither read from nor written to HBM.
__host__ __device__ constexpr int instance_for(int nlev) {
  return nlev < 2 ? 0 : nlev <= 64 ? ((nlev + 7) / 8) * 8 : nlev <= 72 ? 72 : nlev <= 80 ? 80 : nlev <= 96 ? 96
         : nlev <= 112 ? 112 : nlev <= 120 ? 120 : nlev <= 128 ? 128 : 0;
}

// register budget per thread of every instance (CTAs of at most 256 threads: 5 x 96 or 2 x 256 threads per SM).
// A function of the block size because nvcc (12.9) rejects a literal __maxnreg__ next to __launch_bounds__ and takes
// both only when the cap depends on a template parameter.
constexpr int regs_for(int /*threads*/) { return 128; }

// L = levels held by this CTA, NWT = warps per element (scan totals of the whole column), EUL = Eulerian variant
template <int L, int NWT, bool EUL>
struct Smem {
  static constexpr int LF = L * PTS;  // doubles per scalar level-field (this CTA's slab)
  // late inputs, overwritten in place by the outputs of the same shape
  double vn0[2 * LF];      // derived_vn0           -> derived_vn0
  double vm1[2 * LF];      // v(nm1)                -> v(np1)
  double pec[LF];          // derived_pecnd         -> derived_phi
  double omp[LF];          // derived_omega_p       -> derived_omega_p
  double dpm[LF];          // dp3d(nm1)             -> dp3d(np1)
  double Tm1[LF];          // T(nm1)                -> T(np1)
  double Tn0[LF];          // T(n0)   (input only: keeps 8 registers free during the grad-p peak)
  double Qd[LF];           // Qdp     (input only)
  double vn[EUL ? 2 * LF : 2];  // Eulerian only (last tile: nothing behind it needs the 1024-byte tile alignment): v(n0) of the whole slab, for the k-1 / k+1 neighbours of preq_vertadv
  double tot[3][NWT][16];
  // 2x2 tensors: [igp] stride GS = 20 doubles (160 B) instead of 16 so that the four rows read by the
  // four igp-lanes of a level fall into different banks (conflict-free 128-bit broadcast loads)
  double dinv[4 * 20];     // Dinv * rrearth, [igp][jgp][2][2]
  double dmat[4 * 20];     // D
  double met[16], rmet[16], fcor[16], mp[16], phis[16];
  uint64_t bar[3];
  uint64_t xbar[3];  // CL > 1: arrival of the peer CTAs' scan totals tot[0], tot[1], tot[2]
};

// L = levels of the element, CL = CTAs per element (a thread-block cluster of CL CTAs, each holding L/CL levels).
// CL = 2 is used for nlev = 128: two 256-thread CTAs at 128 registers instead of one 512-thread CTA, so that two
// CTAs (of different elements, in different phases) share an SM; the vertical scans exchange their per-warp
// totals through distributed shared memory with st.async + mbarrier complete_tx (no cluster barrier on that path).
// EUL = the Eulerian vertical coordinate (rsplit == 0, F/routine_extracted.F90:227-262,325-334,515-517): after the
// divergence scan every thread also holds the column total S of div(v dp), hence eta_dot_dpdn at the two interfaces
// of its level (eta_hi = hybi[k+1]*S - prefix_k, eta_lo = hybi[k]*S - prefix_{k-1}, 0 at the top and the bottom);
// the levels k-1 and k+1 of T(n0), v(n0) needed by preq_vertadv (LV/CaarFunctor.hpp:504-547) are re-read from
// global memory (L1/L2 hits: neighbouring threads loaded them), derived_eta_dot_dpdn is updated in place, and the
// dp3d update moves behind the scan. +259 B per element*level of algorithmic traffic (the eta_dot_dpdn RMW).
template <int L, int CL, bool EUL>
__global__ void __launch_bounds__(4 * L / CL) __maxnreg__(regs_for(4 * L / CL))
caar_fused_kernel(const __grid_constant__ KernelArgs A, const __grid_constant__ TmaMaps M) {
  constexpr int LC = L / CL;        // levels per CTA
  constexpr int NW = LC / 8;        // warps per CTA
  constexpr int NWT = L / 8;        // warps per element
  constexpr int LF = LC * PTS;      // doubles per scalar level-field slab of this CTA
  constexpr int GS = 20;  // padded igp stride of the 2x2 tensors in shared memory
  constexpr unsigned FB = LF * sizeof(double);  // bytes of one scalar level-field slab
  static_assert(L % (8 * CL) == 0, "a warp holds 8 levels");
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // swizzled TMA tiles need 1024-byte alignment; the launch adds 1 KB of slack for this round-up
  Smem<LC, NWT, EUL>& S = *reinterpret_cast<Smem<LC, NWT, EUL>*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));

  const int t = threadIdx.x;
  const int lane = t & 31, w = t >> 5;
  const int r = t & 3;  // igp
  const uint32_t rank = (CL > 1) ? cluster_ctarank() : 0u;
  const int gw = (int)rank * NW + w;  // warp index within the element's column
  const int lev0 = (int)rank * LC;    // first level of this CTA
  const int ie = A.nets + (int)(blockIdx.x / CL);
  const size_t e = (size_t)ie;
  const int nl = A.nlev;               // levels of the column (<= L; the levels [nl, L) of this instance are padding)
  const size_t lf = (size_t)nl * PTS;  // doubles per scalar level-field of the whole element
  const int off = lev0 * PTS + t * 4;  // this thread's 4 points inside a scalar level-field of the element
  const bool live = lev0 + (t >> 2) < nl;  // this thread's level exists
  // this thread's first 16-byte chunk inside a swizzled scalar tile (row = level) / (u,v) tile (row = t/2)
  const uint32_t sw1 = (uint32_t)(t >> 2) * 128u + ((uint32_t)((2 * r) ^ ((t >> 2) & 7)) << 4);
  const uint32_t sw2 = (uint32_t)(t >> 1) * 128u + ((uint32_t)((4 * (r & 1)) ^ ((t >> 1) & 7)) << 4);
  // TMA coordinates: (row = level [x2 for (u,v)] inside the slice, slice = element [x time level])
  const int sl_n0 = ie * A.ntl + A.n0, sl_nm1 = ie * A.ntl + A.nm1, sl_np1 = ie * A.ntl + A.np1;

  // ---- kernel entry: one thread starts the TMA prefetch of the late inputs
  if (t == 0) {
    mbar_init(&S.bar[0], 1);
    mbar_init(&S.bar[1], 1);
    mbar_init(&S.bar[2], 1);
    if (CL > 1) {
      // the column is split over two CTAs: rank 1 receives rank 0's forward totals (pressure, divergence), rank 0
      // receives rank 1's reverse totals (geopotential): NW rows of 128 B each
      constexpr unsigned XB = NW * 16 * sizeof(double);
      mbar_init(&S.xbar[0], 1);
      mbar_init(&S.xbar[1], 1);
      mbar_init(&S.xbar[2], 1);
      fence_mbar_init_cluster();
      // forward totals (pressure, divergence) come from every lower rank, reverse totals (geopotential) from every
      // higher rank; Eulerian: the higher ranks' divergence totals too (column total)
      if (rank > 0) {
        mbar_expect_tx(&S.xbar[0], rank * XB);
        mbar_expect_tx(&S.xbar[2], rank * XB);
      }
      if (rank + 1 < CL) mbar_expect_tx(&S.xbar[1], (CL - 1 - rank) * (EUL ? 2 * XB : XB));
    }
    fence_proxy_async();
  }
  // "my mbarriers are initialised" — the peer may send to me once it has waited on this. Relaxed: the
  // fence.mbarrier_init above is the release; a releasing arrive placed after the TMA issue below would wait for
  // every outstanding bulk copy (measured: 22 % of all stall samples on ERRBAR / UCGABAR_ARV).
  if (CL > 1) cluster_arrive_relaxed();
  if (t == 0) {
    mbar_expect_tx(&S.bar[2], ((A.qn0 != -1 ? 2 : 1) + (EUL ? 2 : 0)) * FB);
    tma_load(S.Tn0, &M.T, lev0, sl_n0, &S.bar[2]);
    if (EUL) tma_load(S.vn, &M.v, lev0 * 2, sl_n0, &S.bar[2]);
    if (A.qn0 != -1) tma_load(S.Qd, &M.Qdp, lev0, (ie * A.qsize_d + 0) * 2 + A.qn0, &S.bar[2]);
    mbar_expect_tx(&S.bar[0], 4 * FB);
    tma_load(S.vn0, &M.vn0, lev0 * 2, ie, &S.bar[0]);
    tma_load(S.dpm, &M.dp3d, lev0, sl_nm1, &S.bar[0]);
    tma_load(S.pec, &M.pecnd, lev0, ie, &S.bar[0]);
    mbar_expect_tx(&S.bar[1], 4 * FB);
    tma_load(S.omp, &M.omega_p, lev0, ie, &S.bar[1]);
    tma_load(S.Tm1, &M.T, lev0, sl_nm1, &S.bar[1]);
    tma_load(S.vm1, &M.v, lev0 * 2, sl_nm1, &S.bar[1]);
    // pull the early inputs and the geometry of a later element (the one expected to run next on this SM slot) into L2, so
    // that its kernel-start loads see L2 latency instead of DRAM latency
    const int pe = ie + A.pf_dist;
    if (A.pf_dist > 0 && pe < A.nete && lev0 < nl) {
      const size_t pn0 = ((size_t)pe * A.ntl + A.n0) * lf + (size_t)lev0 * PTS;
      const unsigned PB = (nl - lev0 < LC) ? (unsigned)(nl - lev0) * PTS * sizeof(double) : FB;  // this slab, clipped to the column
      prefetch_l2(A.dp3d + pn0, PB);
      prefetch_l2(A.v + pn0 * 2, 2 * PB);
      prefetch_l2(A.T + pn0, PB);
      if (A.qn0 != -1) prefetch_l2(A.Qdp + (((size_t)pe * A.qsize_d + 0) * 2 + A.qn0) * lf + (size_t)lev0 * PTS, PB);
      if (rank == 0) {
        prefetch_l2(A.Dinv + (size_t)pe * 64, 512);
        prefetch_l2(A.D + (size_t)pe * 64, 512);
        prefetch_l2(A.metdet + (size_t)pe * 16, 128);
        prefetch_l2(A.rmetdet + (size_t)pe * 16, 128);
        prefetch_l2(A.fcor + (size_t)pe * 16, 128);
        prefetch_l2(A.spheremp + (size_t)pe * 16, 128);
        prefetch_l2(A.phis + (size_t)pe * 16, 128);
      }
    }
  }

  // ---- early inputs straight to registers
  const size_t on0 = (e * A.ntl + A.n0) * lf + off;
  Row dp, v1, v2;
  if (live) {
    dp = ld_row(A.dp3d + on0);
    ld_row2(A.v + on0 * 2, v1, v2);
  } else {  // padding level: a positive thickness and no wind make every scan contribution of this thread exactly 0
#pragma unroll
    for (int j = 0; j < 4; ++j) dp.x[j] = 1.0, v1.x[j] = 0.0, v2.x[j] = 0.0;
  }
  if (EUL && r == 0 && live)  // this level's derived_eta_dot_dpdn line is read-modify-written after the scans: pull it into L2
    asm volatile("prefetch.global.L2 [%0];" ::"l"(A.eta_dot_dpdn + e * (lf + PTS) + off));

  // ---- stage the element's geometry
  for (int g = t; g < 96; g += 4 * LC) {  // 96 staging slots; CTAs of fewer threads take several each
    if (g < 64) {
      S.dinv[(g >> 4) * GS + (g & 15)] = A.Dinv[e * 64 + g] * A.rrearth;
      S.dmat[(g >> 4) * GS + (g & 15)] = A.D[e * 64 + g];
    } else if (g < 80) {
      const int q = g - 64;
      S.met[q] = A.metdet[e * 16 + q];
      S.rmet[q] = A.rmetdet[e * 16 + q];
      S.fcor[q] = A.fcor[e * 16 + q];
    } else {
      const int q = g - 80;
      S.mp[q] = A.spheremp[e * 16 + q];
      S.phis[q] = A.phis[e * 16 + q];
    }
  }

  const DerivMma cx = deriv_mma_setup(A.dvv, lane);  // igp derivatives on the FP64 tensor core (see deriv_i)

  // ---- A: p = hyai0*ps0 + sum_{l<k} dp_l + dp_k/2   (PO:76-97)
  Row rp;
  {
    Row p;
#pragma unroll
    for (int j = 0; j < 4; ++j) p.x[j] = scan_down(dp.x[j], lane);
    if (CL > 1) cluster_wait();  // the peer CTA is running and has initialised its mbarriers
    if (lane >= 28) {
      st_row(&S.tot[0][gw][r * 4], p);
      if (CL > 1)
        for (uint32_t rr = rank + 1; rr < (uint32_t)CL; ++rr) st_row_async_remote(&S.tot[0][gw][r * 4], &S.xbar[0], rr, p.x);
    }
    __syncthreads();  // (1) tot[0], geometry, mbarrier init visible
    if (CL > 1 && rank > 0) mbar_wait(&S.xbar[0], 0);  // the lower ranks' totals have landed
    // The cluster and Eulerian instances combine the warp totals with warp_totals(). A/B: nlev=128 0.831 -> 0.844
    // (Eulerian 0.575 -> 0.674); nlev=72 on CTA triples 0.965 -> 0.993 (and no spills left). The single-CTA Lagrangian
    // instances (at most 8 warps) keep the plain loop; warp_totals() has not been measured there.
    constexpr bool LANE_CARRY = (CL > 1) || EUL;
    double carry[4] = {0, 0, 0, 0};
    if constexpr (LANE_CARRY) {
      warp_totals<NWT>(S.tot[0], 0, gw, lane, carry);
    } else {
#pragma unroll
      for (int ww = 0; ww < NWT - 1; ++ww)
        if (ww < gw) {
          const Row c = ld_row(&S.tot[0][ww][r * 4]);
#pragma unroll
          for (int j = 0; j < 4; ++j) carry[j] += c.x[j];
        }
    }
    const double ptop = A.hyai0 * A.ps0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      p.x[j] = ptop + ((carry[j] + p.x[j]) - 0.5 * dp.x[j]);
      rp.x[j] = fast_rcp(p.x[j]);
    }

    // ---- vorticity_sphere (PO/sphere_operators.cpp:91-129) first: it needs only v, and leaves one row (fv)
    Row fv;
    {
      Row vc0, vc1;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double2 d01 = lds2(S.dmat + r * GS + j * 4), d23 = lds2(S.dmat + r * GS + j * 4 + 2);
        vc0.x[j] = fma(d01.x, v1.x[j], d23.x * v2.x[j]);
        vc1.x[j] = fma(d01.y, v1.x[j], d23.y * v2.x[j]);
      }
      const Row dvdx = deriv_i(vc1, cx);
      const Row dudy = deriv_j(vc0, A.dvv);
      const Row rm = ld_row(S.rmet + r * 4), fc = ld_row(S.fcor + r * 4);
#pragma unroll
      for (int j = 0; j < 4; ++j) fv.x[j] = fma((dvdx.x[j] - dudy.x[j]) * rm.x[j], A.rrearth, fc.x[j]);
    }
    asm volatile("" ::: "memory");

    // ---- B1: grad_p; vgrad_p (PO:103-112); C: T_v (PO:126-156); glnps folded into the v tendencies
    Row gp0, gp1;
    // w = Dinv.v: v.grad(s) = a_s*w1 + b_s*w2 with (a_s,b_s) the raw igp/jgp derivatives of s
    // (PO/sphere_operators.cpp:21-47), and the divergence flux is metdet*dp*w (PO/sphere_operators.cpp:62-72): one
    // pass over Dinv serves -v.grad T (PO:200-209) and divergence_sphere(v*dp) (PO:122). In the cluster instances
    // the same pass also produces grad p, which saves 8 LDS.128; the single-CTA instances form w after grad p.
    // Whether they would gain from the fused pass has not been measured.
    constexpr bool FUSE_W = (CL > 1);
    Row w1, w2;
    if constexpr (FUSE_W) {
      const Row a = deriv_i(p, cx), b = deriv_j(p, A.dvv);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double2 d01 = lds2(S.dinv + r * GS + j * 4), d23 = lds2(S.dinv + r * GS + j * 4 + 2);
        gp0.x[j] = fma(d01.x, a.x[j], d23.x * b.x[j]);
        gp1.x[j] = fma(d01.y, a.x[j], d23.y * b.x[j]);
        w1.x[j] = fma(d01.x, v1.x[j], d01.y * v2.x[j]);
        w2.x[j] = fma(d23.x, v1.x[j], d23.y * v2.x[j]);
      }
    } else {
      gradient(p, S.dinv + r * GS, cx, A.dvv, gp0, gp1);
    }
    // from here on p is dead; only rp is kept
    mbar_wait(&S.bar[2], 0);  // T(n0), Qdp tiles
    Row Tv = ld_tile(S.Tn0, sw1);
    if (A.qn0 != -1) {
      const Row Qd = ld_tile(S.Qd, sw1);
      const double c = A.Rwv / A.Rgas - 1.0;
#pragma unroll
      for (int j = 0; j < 4; ++j) Tv.x[j] *= fma(c, Qd.x[j] * fast_rcp(dp.x[j]), 1.0);
    }
    // vgp <- v.grad_p ; vtens (without grad Ephi) = (+v2, -v1)*(fcor+vort) - Rgas*T_v/p * grad_p  (PO:219-228)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double vg = fma(v1.x[j], gp0.x[j], v2.x[j] * gp1.x[j]);
      const double gl = -A.Rgas * (Tv.x[j] * rp.x[j]);
      gp0.x[j] = fma(gl, gp0.x[j], v2.x[j] * fv.x[j]);
      gp1.x[j] = fma(gl, gp1.x[j], -v1.x[j] * fv.x[j]);
      p.x[j] = vg;  // p now holds vgrad_p
    }
    Row& vt1 = gp0;
    Row& vt2 = gp1;
    Row& vgp = p;
    asm volatile("" ::: "memory");

    if constexpr (!FUSE_W) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double2 d01 = lds2(S.dinv + r * GS + j * 4), d23 = lds2(S.dinv + r * GS + j * 4 + 2);
        w1.x[j] = fma(d01.x, v1.x[j], d01.y * v2.x[j]);
        w2.x[j] = fma(d23.x, v1.x[j], d23.y * v2.x[j]);
      }
    }
    Row ttp;
    {
      const Row T = ld_tile(S.Tn0, sw1);
      const Row a = deriv_i(T, cx), b = deriv_j(T, A.dvv);
#pragma unroll
      for (int j = 0; j < 4; ++j) ttp.x[j] = -fma(a.x[j], w1.x[j], b.x[j] * w2.x[j]);
    }
    if (EUL) st_tile(S.Qd, sw1, vt2);  // Eulerian: T(n0) stays in use (vertical neighbours), the Qdp slot is free

    // ---- late inputs, first batch (vn0, dp3d(nm1), pecnd) must have landed
    mbar_wait(&S.bar[0], 0);

    // ---- B2: derived_vn0 += eta_ave_w*v*dp (PO:114-118); divergence_sphere(v*dp) (PO/sphere_operators.cpp:50-89)
    Row divdp;
    {
      {
        Row a0, a1;
        ld_tile2(S.vn0, sw2, a0, a1);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          a0.x[j] = fma(A.eta_ave_w, v1.x[j] * dp.x[j], a0.x[j]);
          a1.x[j] = fma(A.eta_ave_w, v2.x[j] * dp.x[j], a1.x[j]);
        }
        st_tile2(S.vn0, sw2, a0, a1);
      }
      const Row met = ld_row(S.met + r * 4);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double md = met.x[j] * dp.x[j];
        w1.x[j] *= md;
        w2.x[j] *= md;
      }
      const Row dudx = deriv_i(w1, cx);
      const Row dvdy = deriv_j(w2, A.dvv);
      const Row rm = ld_row(S.rmet + r * 4);
#pragma unroll
      for (int j = 0; j < 4; ++j) divdp.x[j] = (dudx.x[j] + dvdy.x[j]) * rm.x[j];  // dinv carries rrearth
    }
    // dp3d(np1) = spheremp*(dp3d(nm1) - dt2*divdp)  (PO:254), in place over dp3d(nm1)
    Row dsave;  // Eulerian: div(v dp) of this level survives the scan (the vertical flux difference joins it later)
    if (EUL) {
      dsave = divdp;
    } else {
      const Row mp = ld_row(S.mp + r * 4);
      Row o = ld_tile(S.dpm, sw1);
#pragma unroll
      for (int j = 0; j < 4; ++j) o.x[j] = mp.x[j] * fma(-A.dt2, divdp.x[j], o.x[j]);
      st_tile(S.dpm, sw1, o);
    }
    fence_proxy_async();  // vn0 and dp3d(np1) tiles are final: make them visible to the TMA engine

    // ---- kinetic energy + pecnd (PO:196; phi is added after the scan)
    Row kep;
    {
      const Row pec = ld_tile(S.pec, sw1);
#pragma unroll
      for (int j = 0; j < 4; ++j) kep.x[j] = fma(0.5, fma(v1.x[j], v1.x[j], v2.x[j] * v2.x[j]), pec.x[j]);
      if (EUL) st_tile(S.pec, sw1, kep);  // Eulerian: waits in this thread's own (now dead) pecnd slot for phi
    }
    // v1, v2 are dead from here

    // ---- D+E: the two vertical integrals in scan form
    //   q_k = Rgas*T_v*dp/p ; phi_k = phis + sum_{l>k} q_l + q_k/2              (PO:280-312)
    //   omega_k = (vgrad_p - sum_{l<k} divdp_l - divdp_k/2) / p                 (PO:314-352)
    Row a, ph;
    {
      Row tq;
      const Row phis = ld_row(S.phis + r * 4);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double q = A.Rgas * Tv.x[j] * (dp.x[j] * rp.x[j]);
        const double sq = scan_up(q, lane);
        const double sd = scan_down(divdp.x[j], lane);
        ph.x[j] = phis.x[j] + (sq - 0.5 * q);
        a.x[j] = rp.x[j] * (vgp.x[j] - (sd - 0.5 * divdp.x[j]));
        tq.x[j] = sq;      // warp totals live in the end lanes
        divdp.x[j] = sd;
      }
      if (lane < 4) {
        st_row(&S.tot[1][gw][r * 4], tq);
        if (CL > 1)
          for (uint32_t rr = 0; rr < rank; ++rr) st_row_async_remote(&S.tot[1][gw][r * 4], &S.xbar[1], rr, tq.x);
      }
      if (lane >= 28) {
        st_row(&S.tot[2][gw][r * 4], divdp);
        if (CL > 1) {
          for (uint32_t rr = rank + 1; rr < (uint32_t)CL; ++rr)
            st_row_async_remote(&S.tot[2][gw][r * 4], &S.xbar[2], rr, divdp.x);
          if (EUL)
            for (uint32_t rr = 0; rr < rank; ++rr) st_row_async_remote(&S.tot[2][gw][r * 4], &S.xbar[1], rr, divdp.x);
        }
      }
    }
    // T tendency with the omega carry factored out: ttens = kappa*T_v*omega - v.gradT, omega = a - rp*carry
    Row tta, ttb;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double kt = A.kappa * Tv.x[j];
      tta.x[j] = fma(kt, a.x[j], ttp.x[j]);
      ttb.x[j] = kt * rp.x[j];
    }
    __syncthreads();  // (2) scan totals visible; vn0 / dp3d(np1) tiles complete
    if (CL > 1) {  // the peers' totals have landed
      if (rank + 1 < CL) mbar_wait(&S.xbar[1], 0);
      if (rank > 0) mbar_wait(&S.xbar[2], 0);
    }
    if (t == 0) {
      tma_store(&M.vn0, lev0 * 2, ie, S.vn0);
      if (!EUL) tma_store(&M.dp3d, lev0, sl_np1, S.dpm);
      bulk_commit();
    }
    double cq[4] = {0, 0, 0, 0}, cd[4] = {0, 0, 0, 0};
    double S4[4] = {0, 0, 0, 0};  // Eulerian: column total of div(v dp)
    if constexpr (LANE_CARRY) {
      warp_totals<NWT>(S.tot[1], gw + 1, NWT, lane, cq);
      if constexpr (EUL && NWT <= 12) warp_totals_both<NWT>(S.tot[2], gw, lane, cd, S4);
      else warp_totals<NWT>(S.tot[2], 0, gw, lane, cd);
    } else {
#pragma unroll
      for (int ww = 0; ww < NWT; ++ww) {
        if (ww > gw) {
          const Row c = ld_row(&S.tot[1][ww][r * 4]);
#pragma unroll
          for (int j = 0; j < 4; ++j) cq[j] += c.x[j];
        }
        if (ww < gw) {
          const Row c = ld_row(&S.tot[2][ww][r * 4]);
#pragma unroll
          for (int j = 0; j < 4; ++j) cd[j] += c.x[j];
        }
      }
    }

    // ---- late inputs, second batch (omega_p, T(nm1), v(nm1))
    mbar_wait(&S.bar[1], 0);
    const Row mp = ld_row(S.mp + r * 4);
    Row eta_old, dpk_early;  // Eulerian: the two global loads of this block, issued before the math that hides their latency
    constexpr bool HOIST = EUL && LC >= EUL_HOIST_LEVELS;
    if (EUL) {
      if (HOIST && live) {
        dpk_early = ld_row(A.dp3d + on0);
        if (lev0 + (t >> 2) > 0) eta_old = ld_row(A.eta_dot_dpdn + e * (lf + PTS) + off);
      }
      // finish what frees registers first (a, rp, ttb, ph, cq die here): omega_p, the T tendency without T_vadv,
      // phi and Ephi
      {
        Row om = ld_tile(S.omp, sw1);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          om.x[j] = fma(A.eta_ave_w, fma(-rp.x[j], cd[j], a.x[j]), om.x[j]);
          tta.x[j] = fma(-ttb.x[j], cd[j], tta.x[j]);
        }
        st_tile(S.omp, sw1, om);
      }
      kep = ld_tile(S.pec, sw1);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ph.x[j] += cq[j];
        kep.x[j] += ph.x[j];
      }
      st_tile(S.pec, sw1, ph);
      // column total S of div(v dp) and the vertical mass flux at this level's two interfaces
      // (F/routine_extracted.F90:233-254): eta(k+1) = hybi(k+1)*S - sum_{l<=k} divdp_l, 0 at the top and bottom
      if constexpr (NWT > 12) warp_totals<NWT>(S.tot[2], 0, NWT, lane, S4);  // else warp_totals_both delivered it
      const int kg = lev0 + (t >> 2);
      const double hb_lo = A.hybi[kg < nl ? kg : nl], hb_hi = A.hybi[kg < nl ? kg + 1 : nl];
      Row ehi, elo;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double P = cd[j] + divdp.x[j];  // inclusive prefix of div(v dp)
        ehi.x[j] = (kg >= nl - 1) ? 0.0 : fma(hb_hi, S4[j], -P);
        elo.x[j] = (kg == 0) ? 0.0 : fma(hb_lo, S4[j], -(P - dsave.x[j]));
      }
      {  // dp3d(np1) = spheremp*(dp3d(nm1) - dt2*(divdp + eta(k+1) - eta(k)))  (F/routine_extracted.F90:515-517)
        Row o = ld_tile(S.dpm, sw1);
#pragma unroll
        for (int j = 0; j < 4; ++j) o.x[j] = mp.x[j] * fma(-A.dt2, (dsave.x[j] + ehi.x[j]) - elo.x[j], o.x[j]);
        st_tile(S.dpm, sw1, o);
      }
      if (kg > 0 && live) {  // derived_eta_dot_dpdn(k) += eta_ave_w*eta(k) (F:270-277); interfaces 0 and L carry no flux
        double* pe = A.eta_dot_dpdn + e * (lf + PTS) + off;
        Row x = HOIST ? eta_old : ld_row(pe);
#pragma unroll
        for (int j = 0; j < 4; ++j) x.x[j] = fma(A.eta_ave_w, elo.x[j], x.x[j]);
        st_row(pe, x);
      }
      // preq_vertadv (LV/CaarFunctor.hpp:504-547): fac+ = eta(k+1)/(2 dp), fac- = eta(k)/(2 dp); the one-sided
      // forms at the top and bottom follow from eta = 0 there
      {
        Row dpk;  // re-read (L1/L2 hit) rather than 4 doubles live through the scans
        if (HOIST) dpk = dpk_early;
        else if (live) dpk = ld_row(A.dp3d + on0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double hr = live ? 0.5 * fast_rcp(dpk.x[j]) : 0.0;
          ehi.x[j] *= hr;
          elo.x[j] *= hr;
        }
      }
      // neighbouring levels come from the shared-memory tiles; only the first / last level of a split column
      // (CL = 2) reads its neighbour, which lives in the peer CTA, from global memory
      const int kl = t >> 2;  // level inside this CTA's slab
      {
        const Row Tk = ld_tile(S.Tn0, sw1);
        Row Tu = Tk, Td = Tk;
        if (kg + 1 < nl) {
          if (kl + 1 < LC) Tu = ld_tile(S.Tn0, (uint32_t)(kl + 1) * 128u + ((uint32_t)((2 * r) ^ ((kl + 1) & 7)) << 4));
          else Tu = ld_row(A.T + on0 + PTS);
        }
        if (kg > 0) {
          if (kl > 0) Td = ld_tile(S.Tn0, (uint32_t)(kl - 1) * 128u + ((uint32_t)((2 * r) ^ ((kl - 1) & 7)) << 4));
          else Td = ld_row(A.T + on0 - PTS);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)  // ttens = -T_vadv - v.gradT + kappa*T_v*omega (F:333)
          tta.x[j] -= fma(ehi.x[j], Tu.x[j] - Tk.x[j], elo.x[j] * (Tk.x[j] - Td.x[j]));
      }
      {
        Row uk, vk, uu, vu, ud, vd;
        ld_tile2(S.vn, sw2, uk, vk);
        uu = uk; vu = vk; ud = uk; vd = vk;
        const int tr = t >> 1;  // this thread's row in the (u,v) tile; a level spans two tile rows
        if (kg + 1 < nl) {
          if (kl + 1 < LC) ld_tile2(S.vn, (uint32_t)(tr + 2) * 128u + ((uint32_t)((4 * (r & 1)) ^ ((tr + 2) & 7)) << 4), uu, vu);
          else ld_row2(A.v + (on0 + PTS) * 2, uu, vu);
        }
        if (kg > 0) {
          if (kl > 0) ld_tile2(S.vn, (uint32_t)(tr - 2) * 128u + ((uint32_t)((4 * (r & 1)) ^ ((tr - 2) & 7)) << 4), ud, vd);
          else ld_row2(A.v + (on0 - PTS) * 2, ud, vd);
        }
        vt2 = ld_tile(S.Qd, sw1);  // parked there since the first half of the kernel
#pragma unroll
        for (int j = 0; j < 4; ++j) {  // vtens = -v_vadv + ... (F:325-331)
          vt1.x[j] -= fma(ehi.x[j], uu.x[j] - uk.x[j], elo.x[j] * (uk.x[j] - ud.x[j]));
          vt2.x[j] -= fma(ehi.x[j], vu.x[j] - vk.x[j], elo.x[j] * (vk.x[j] - vd.x[j]));
        }
      }
    }
    if constexpr (EUL) {  // T(np1) = spheremp*(T(nm1) + dt2*ttens); omega_p, phi and Ephi were done above
      Row Tn = ld_tile(S.Tm1, sw1);
#pragma unroll
      for (int j = 0; j < 4; ++j) Tn.x[j] = mp.x[j] * fma(A.dt2, tta.x[j], Tn.x[j]);
      st_tile(S.Tm1, sw1, Tn);
    } else {
      {  // derived_omega_p += eta_ave_w*omega (PO:173); T(np1) = spheremp*(T(nm1) + dt2*ttens) (PO:253)
        Row om = ld_tile(S.omp, sw1), Tn = ld_tile(S.Tm1, sw1);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double omega = fma(-rp.x[j], cd[j], a.x[j]);
          om.x[j] = fma(A.eta_ave_w, omega, om.x[j]);
          const double tt = fma(-ttb.x[j], cd[j], tta.x[j]);
          Tn.x[j] = mp.x[j] * fma(A.dt2, tt, Tn.x[j]);
        }
        st_tile(S.omp, sw1, om);
        st_tile(S.Tm1, sw1, Tn);
      }
      // phi (PO:294,303,309) in place over pecnd; Ephi = 0.5|v|^2 + phi + pecnd (PO:196)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ph.x[j] += cq[j];
        kep.x[j] += ph.x[j];
      }
      st_tile(S.pec, sw1, ph);
    }
    {  // v(np1) = spheremp*(v(nm1) + dt2*vtens) (PO:251-252), in place over v(nm1)
      Row g0, g1;
      gradient(kep, S.dinv + r * GS, cx, A.dvv, g0, g1);
      Row a0, a1;
      ld_tile2(S.vm1, sw2, a0, a1);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        a0.x[j] = mp.x[j] * fma(A.dt2, vt1.x[j] - g0.x[j], a0.x[j]);
        a1.x[j] = mp.x[j] * fma(A.dt2, vt2.x[j] - g1.x[j], a1.x[j]);
      }
      st_tile2(S.vm1, sw2, a0, a1);
    }
  }
  fence_proxy_async();
  // (3) all output tiles complete. Eulerian + split column + np1 == n0: the peer CTA reads my boundary level of
  // T(n0)/v(n0) from global memory, so my stores over that time level must wait for it as well
  if (CL > 1 && EUL && A.np1 == A.n0) {
    cluster_arrive();
    cluster_wait();
  } else {
    __syncthreads();
  }
  if (t == 0) {
    if (EUL) tma_store(&M.dp3d, lev0, sl_np1, S.dpm);
    tma_store(&M.omega_p, lev0, ie, S.omp);
    tma_store(&M.T, lev0, sl_np1, S.Tm1);
    tma_store(&M.phi, lev0, ie, S.pec);
    tma_store(&M.v, lev0 * 2, sl_np1, S.vm1);
    bulk_commit();
    bulk_wait_read_all();  // shared memory must stay alive until the TMA engine has read it
  }
}

template <int L, int CL, bool EUL>
cudaError_t launch_L(const KernelArgs& a, cudaStream_t s) {
  const int n = a.nete - a.nets;
  if (n <= 0) return cudaSuccess;
  constexpr int SMEM = (int)sizeof(Smem<L / CL, L / 8, EUL>) + 1024;
  static LaunchCache cache;
  int per_sm = 0;
  if (cudaError_t e = setup_launch(caar_fused_kernel<L, CL, EUL>, 4 * L / CL, SMEM, cache, &per_sm)) return e;
  if (!a.tma) return cudaErrorInvalidValue;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)n * CL, 1, 1);
  cfg.blockDim = dim3(4 * L / CL, 1, 1);
  cfg.dynamicSmemBytes = SMEM;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  // cluster scheduling policy: load balancing for the CTA triples (A/B at nlev=72: 1.037-1.040 of the measured peak vs
  // 0.995-1.014 with the default spread policy), spread for pairs (nlev=128: no difference)
  const bool balance = CL >= 3;
  attr[1].id = cudaLaunchAttributeClusterSchedulingPolicyPreference;
  attr[1].val.clusterSchedulingPolicyPreference =
      balance ? cudaClusterSchedulingPolicyLoadBalancing : cudaClusterSchedulingPolicySpread;
  cfg.attrs = attr;
  cfg.numAttrs = (CL > 1) ? 2 : 0;
  return cudaLaunchKernelEx(&cfg, caar_fused_kernel<L, CL, EUL>, a, *static_cast<const TmaMaps*>(a.tma));
}

// both vertical coordinates of one level count
template <int L>
cudaError_t launch_nlev(const KernelArgs& a, cudaStream_t s) {
  static_assert(cluster_for(L) > 0, "no fused instance for this level count");
  return a.rsplit == 0 ? launch_L<L, cluster_for(L), true>(a, s) : launch_L<L, cluster_for(L), false>(a, s);
}

}  // namespace
}  // namespace caar
