// caar_levelops.cu — the level-local operators around compute_and_apply_rhs (SURVEY §8f rank 4) on ONE skeleton:
//
//   OP_EULER           qtens[e][iq][k] = Qdp[e][iq][qn0][k] - dt * divergence_sphere(vstar[e][k] * Qdp[e][iq][qn0][k])
//                      EulerStepFunctor::operator() = divergence_sphere_update(alpha = -dt, beta = 1)
//                      (level_vectorized_ppscan/EulerStepFunctor.hpp:33-66, SphereOperators.hpp:362-403)
//   OP_DIVERGENCE_WK   out[e][k] = divergence_sphere_wk(vin[e][k])                  (SphereOperators.hpp:493-535)
//   OP_LAPLACE_SIMPLE  out[e][k] = divergence_sphere_wk(gradient_sphere(sin[e][k])) (SphereOperators.hpp:537-553)
//   OP_LAPLACE_TENSOR  out[e][k] = divergence_sphere_wk(tensorVisc[e] . gradient_sphere(sin[e][k]))
//                      (SphereOperators.hpp:555-636; "replace" = the same in place)
//
// in the pointers_only array conventions ([e]...[lev][igp][jgp]([c])). Levels are independent here (no vertical
// integral), so the unit of work is one group of 8 levels of one element for one streamed field = one WARP: lane = (level
// of the group, GLL row), 4 points each, as in the fused CAAR kernel.
//
// Data movement — the fused kernel's: every level-field array is a 3-D TMA tensor [slice][level][16 doubles]; the
// streamed input tiles (Qdp / vin / sin; 8 levels = 1 KB = one 128-byte-swizzle atom) arrive through an NS-deep ring of
// shared-memory stages PER WARP, filled by the warp's lane 0 with cp.async.bulk.tensor (UTMALDG) completing on the warp's
// own mbarriers, NS tiles ahead of the math; results leave as bulk tensor stores (UTMASTG) from a 2-deep ring of output
// tiles; vstar (OP_EULER) is a per-(element, group) tile, double-buffered and fetched two items ahead. Every warp of the
// persistent grid is an independent pipeline (__syncwarp only — the first version synchronised whole CTAs per tile and was
// latency-bound at 0.3-0.6 of the peak) over a contiguous range of the unit list (element, group, tracer), tracer
// fastest: the row's geometry is loaded once per element, the flux weights once per (element, group). Rows of a group
// beyond nlev are zero-filled on load and clipped on store: any nlev works.
//
// OP_EULER fast path per tracer and thread: the 16 values of the level's Qdp tile (8 conflict-free LDS.128 — the four
// threads of a level read the same 16 bytes) against 16 + 8 coefficients held in registers,
//   out(r,j) = q(r,j) + sum_m A(m,j) q(m,j) + c(r,j) sum_m Dvv[m][j] w2(r,m) q(r,m),
//   c(r,j) = -dt rmetdet(r,j) rrearth,  A(m,j) = c(r,j) Dvv[m][r] w1(m,j),  (w1,w2) = metdet Dinv vstar
//   — no shuffles and no geometry loads inside the tracer loop.
// divergence_sphere_wk (and the laplacians for nlev < 16) use the fused kernel's row decomposition: sums along jgp
// thread-local, sums along igp through three xor-shuffles per value; the laplacians proper run on laplace_flat_kernel
// below (one thread per level, tiles drawn from a global counter). Tried and rejected for the row-decomposed laplacians
// (profiles/README.md): exchanging the rows through the shared-memory
// tile instead of shuffles (80 fewer instructions per tile, two more __syncwarp round trips: 0.66 vs 0.70 for
// laplace_simple), and computing the per-element coefficients in a pre-pass kernel with a bulk-copy prefetch two elements
// ahead (the second launch costs more than the load chain it removes: 0.62 vs 0.70, tracer step 0.91 vs 0.97).
//
// Bound: HBM. Algorithmic bytes per element*level(*tracer): OP_EULER 256 + (256 + 1408/L)/qsize; OP_DIVERGENCE_WK
// 384 + 640/L; OP_LAPLACE_* 256 + (640 | 1152)/L.
//
// CAAR_MODE_STRICT: reference operation order with __dmul_rn/__dadd_rn (bit-identical to the CPU restatement, which is
// bit-identical to the reference's own HOMMEXX code for the weak-form operators): plain point-per-thread kernels below;
// the tracer step's strict variant stays in caar_euler.cu.
#include "caar_fused_kernel.cuh"

namespace caar {
namespace {

#ifndef LEVELOP_NS
#define LEVELOP_NS 4
#endif
#ifndef LEVELOP_NO
#define LEVELOP_NO 2
#endif
#ifndef LEVELOP_WPC
#define LEVELOP_WPC 4
#endif
#ifndef LEVELOP_MINB
#define LEVELOP_MINB 4
#endif
constexpr int NS = LEVELOP_NS;    // input tiles in flight per warp
constexpr int NO = LEVELOP_NO;    // output tiles in flight per warp
constexpr int WPC = LEVELOP_WPC;  // warps per CTA (independent pipelines: no CTA-wide barrier after the prologue)
constexpr int GL = 8;   // levels per tile = levels per warp (8 levels x 4 GLL rows = 32 lanes)

struct LevelOpArgs {
  const double* Dinv;
  const double* metdet;
  const double* rmetdet;
  const double* spheremp;
  const double* tensorvisc;
  int nlev, nets, ngroups, Q, qn0, qsize_d;
  int out_stride, out_off;  // OP_EULER: unit (e, iq) stores slice (e * qsize_d + iq) * out_stride + out_off of M.out
  long long units;  // elements * ngroups * Q
  double dt, rrearth;
  double dvv[16];
};
struct alignas(64) LevelOpMaps {
  CUtensorMap in, out, item;
};

// c[m] = Dvv[m][r] / c[m] = Dvv[r][m] without dynamic indexing of the kernel parameters
__device__ __forceinline__ void dvv_col(const double* __restrict__ dvv, int r, double (&c)[4]) {
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    double x = dvv[m * 4 + 0];
    if (r == 1) x = dvv[m * 4 + 1];
    if (r == 2) x = dvv[m * 4 + 2];
    if (r == 3) x = dvv[m * 4 + 3];
    c[m] = x;
  }
}
__device__ __forceinline__ void dvv_row(const double* __restrict__ dvv, int r, double (&c)[4]) {
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    double x = dvv[0 * 4 + m];
    if (r == 1) x = dvv[1 * 4 + m];
    if (r == 2) x = dvv[2 * 4 + m];
    if (r == 3) x = dvv[3 * 4 + m];
    c[m] = x;
  }
}

enum { OP_EULER = 0, OP_DIVWK = 1, OP_LAP_SIMPLE = 2, OP_LAP_TENSOR = 3 };

// Every WARP is an independent pipeline over a contiguous range of units (element, group of 8 levels, tracer), tracer
// fastest: its lane 0 issues the TMA loads NS tiles ahead and the TMA stores, the warp waits on its own mbarriers and
// synchronises with __syncwarp only.
//
// OP_EULER in place (a stage of caar_advect_tracers with qn0 == np1: M.out is the Qdp map, out_stride 2, out_off np1,
// so every unit loads and stores the same tile). Safe because each unit owns exactly one tile, which no other unit of
// any warp loads or stores; a unit's input tile is in shared memory (its mbarrier has completed and every lane has
// read it) before its store is issued; and the ring only prefetches tiles of this warp's later units, never one an
// earlier unit of any warp stores. The next stage reads the stored tiles back with TMA: the bulk stores are complete
// when the grid is, and the exit below only waits for their shared-memory reads, as the in-place laplacian does.
template <int OP>
__global__ void __launch_bounds__(32 * WPC, LEVELOP_MINB) levelop_kernel(const __grid_constant__ LevelOpArgs A,
                                                              const __grid_constant__ LevelOpMaps M) {
  constexpr unsigned IN_B = (OP == OP_DIVWK) ? 2048u : 1024u;  // bytes of a streamed input tile (8 levels)
  constexpr unsigned OUT_B = 1024u, ITEM_B = (OP == OP_EULER) ? 2048u : 0u;
  constexpr unsigned WARP_B = NS * IN_B + NO * OUT_B + 2 * ITEM_B;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int t = threadIdx.x, w = t >> 5, lane = t & 31, r = lane & 3, lvl = lane >> 2;
  unsigned char* in_tiles = base + w * WARP_B;
  unsigned char* out_tiles = in_tiles + NS * IN_B;
  unsigned char* item_tiles = out_tiles + NO * OUT_B;
  uint64_t* full = reinterpret_cast<uint64_t*>(base + WPC * WARP_B) + w * (NS + 2);  // [NS] input stages, [2] item tiles
  uint64_t* item_full = full + NS;

  const int Q = A.Q, NG = A.ngroups;
  const long long wid = (long long)blockIdx.x * WPC + w, nwarps = (long long)gridDim.x * WPC;
  const long long u0 = A.units * wid / nwarps, u1 = A.units * (wid + 1) / nwarps;
  const int n = (int)(u1 - u0);
  if (n <= 0) return;  // whole warp
  // OP_EULER: this warp's cache of the element's geometry, [row][met*Dinv (16) | -dt*rmetdet*rrearth (4)]
  double* geo = reinterpret_cast<double*>(base + WPC * WARP_B + WPC * (NS + 2) * sizeof(uint64_t)) + w * 80;

  // swizzled offsets of this lane's data inside a scalar tile (row = level) and a (u,v) tile (row = 2*level + r/2)
  const uint32_t sw1 = (uint32_t)lvl * 128u + ((uint32_t)((2 * r) ^ (lvl & 7)) << 4);
  const uint32_t sw2 = (uint32_t)(lane >> 1) * 128u + ((uint32_t)((4 * (r & 1)) ^ ((lane >> 1) & 7)) << 4);

  // (element, group, tracer) of a unit, advanced without divisions: tracer fastest, then group, then element
  struct Pos {
    int e, g, iq;
  };
  auto advance = [&](Pos& p) {
    if (++p.iq == Q) {
      p.iq = 0;
      if (++p.g == NG) p.g = 0, ++p.e;
    }
  };
  Pos cur, pre, pitem;  // the unit being computed, the next unit to prefetch, the next (element, group) whose vstar to fetch
  {
    const long long item0 = u0 / Q;
    cur.iq = (int)(u0 - item0 * Q);
    cur.e = A.nets + (int)(item0 / NG);
    cur.g = (int)(item0 % NG);
    pre = cur;
    pitem = cur;
    pitem.iq = 0;
  }
  int items_left = (int)((u0 + n - 1) / Q - u0 / Q) + 1;  // vstar tiles this warp will need

  auto issue_in = [&](int i) {  // unit `pre` -> stage i % NS (lane 0 only); advances `pre`
    const int s = i % NS, lev0 = pre.g * GL;
    mbar_expect_tx(&full[s], IN_B);
    if (OP == OP_EULER) tma_load(in_tiles + s * IN_B, &M.in, lev0, (pre.e * A.qsize_d + pre.iq) * 2 + A.qn0, &full[s]);
    else if (OP == OP_DIVWK) tma_load(in_tiles + s * IN_B, &M.in, lev0 * 2, pre.e, &full[s]);
    else tma_load(in_tiles + s * IN_B, &M.in, lev0, pre.e, &full[s]);
    advance(pre);
  };
  auto issue_item = [&](int k) {  // vstar of `pitem` -> item buffer k % 2 (lane 0 only); advances `pitem`
    mbar_expect_tx(&item_full[k & 1], ITEM_B);
    tma_load(item_tiles + (k & 1) * ITEM_B, &M.item, pitem.g * GL * 2, pitem.e, &item_full[k & 1]);
    if (++pitem.g == NG) pitem.g = 0, ++pitem.e;
    --items_left;
  };

  if (lane == 0) {
    for (int s = 0; s < NS + 2; ++s) mbar_init(&full[s], 1);
    fence_proxy_async();
    for (int i = 0; i < NS && i < n; ++i) issue_in(i);
    if (OP == OP_EULER) {
      issue_item(0);
      if (items_left > 0) issue_item(1);
    }
  }
  __syncwarp();

  double cx[4], cr[4];  // cx[x] = Dvv[r^x][r] (strong form, sum over the first index); cr[x] = Dvv[r][r^x] (weak form)
  {
    double col[4], row[4];
    dvv_col(A.dvv, r, col);
    dvv_row(A.dvv, r, row);
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      double a = col[0 ^ x], b = row[0 ^ x];  // static index per (r, x): select over r
      if (r == 1) a = col[1 ^ x], b = row[1 ^ x];
      if (r == 2) a = col[2 ^ x], b = row[2 ^ x];
      if (r == 3) a = col[3 ^ x], b = row[3 ^ x];
      cx[x] = a;
      cr[x] = b;
    }
  }

  bool new_item = true, new_elem = true;
  int item_k = -1;
  // weak-form operators: this row's point-local 2x2 matrices in registers (once per element)
  double nm[4][4];
  // OP_EULER: per-item coefficients Ac[x][j] = rm[j] Dvv[r^x][r] w1(r^x, j) for row r^x, this row's w2, and rm
  double Ac[4][4], w2[4], rm[4];

  for (int i = 0; i < n; ++i) {
    const int e = cur.e, lev0 = cur.g * GL, iq = cur.iq;
    if (new_item) {  // uniform over the warp
      ++item_k;
      if (new_elem) {  // once per element, reused over its level groups and tracers
        const size_t ge = (size_t)e;
        if (OP == OP_EULER) {
          __syncwarp();  // the previous element's cache is no longer being read
          if (lvl == 0) {  // the four lanes r = 0..3 fill the warp's geometry cache
            double m4[4], r4[4];
            const double2 a = __ldg(reinterpret_cast<const double2*>(A.metdet + ge * 16 + r * 4));
            const double2 b = __ldg(reinterpret_cast<const double2*>(A.metdet + ge * 16 + r * 4 + 2));
            m4[0] = a.x; m4[1] = a.y; m4[2] = b.x; m4[3] = b.y;
            const double2 c = __ldg(reinterpret_cast<const double2*>(A.rmetdet + ge * 16 + r * 4));
            const double2 d = __ldg(reinterpret_cast<const double2*>(A.rmetdet + ge * 16 + r * 4 + 2));
            const double sc = -A.dt * A.rrearth;
            r4[0] = c.x * sc; r4[1] = c.y * sc; r4[2] = d.x * sc; r4[3] = d.y * sc;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const double2 p0 = __ldg(reinterpret_cast<const double2*>(A.Dinv + ge * 64 + (r * 4 + j) * 4));
              const double2 p1 = __ldg(reinterpret_cast<const double2*>(A.Dinv + ge * 64 + (r * 4 + j) * 4 + 2));
              *reinterpret_cast<double2*>(geo + r * 20 + j * 4) = make_double2(m4[j] * p0.x, m4[j] * p0.y);
              *reinterpret_cast<double2*>(geo + r * 20 + j * 4 + 2) = make_double2(m4[j] * p1.x, m4[j] * p1.y);
            }
            *reinterpret_cast<double2*>(geo + r * 20 + 16) = make_double2(r4[0], r4[1]);
            *reinterpret_cast<double2*>(geo + r * 20 + 18) = make_double2(r4[2], r4[3]);
          }
          __syncwarp();
          const double2 a = *reinterpret_cast<const double2*>(geo + r * 20 + 16);
          const double2 b = *reinterpret_cast<const double2*>(geo + r * 20 + 18);
          rm[0] = a.x; rm[1] = a.y; rm[2] = b.x; rm[3] = b.y;
        } else {
          const double2 ma = __ldg(reinterpret_cast<const double2*>(A.spheremp + ge * 16 + r * 4));
          const double2 mb = __ldg(reinterpret_cast<const double2*>(A.spheremp + ge * 16 + r * 4 + 2));
          const double mpr[4] = {ma.x * A.rrearth, ma.y * A.rrearth, mb.x * A.rrearth, mb.y * A.rrearth};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const double2 a = __ldg(reinterpret_cast<const double2*>(A.Dinv + ge * 64 + (r * 4 + j) * 4));
            const double2 b = __ldg(reinterpret_cast<const double2*>(A.Dinv + ge * 64 + (r * 4 + j) * 4 + 2));
            if (OP == OP_DIVWK) {  // s = (spheremp rrearth Dinv) . v
              nm[j][0] = mpr[j] * a.x; nm[j][1] = mpr[j] * a.y; nm[j][2] = mpr[j] * b.x; nm[j][3] = mpr[j] * b.y;
            } else {
              // the whole point-local part of the laplacian as ONE 2x2 matrix per point, applied to the raw derivatives
              // (a, b) of the scalar: grad = rrearth Dinv^T (a,b); [tensor: grad <- tensorVisc grad;] s = spheremp rrearth
              // Dinv grad  =>  s = N (a,b), N = spheremp rrearth^2 Dinv [tensorVisc] Dinv^T
              double t00 = a.x, t01 = b.x, t10 = a.y, t11 = b.y;  // Dinv^T: grad0 = di0 a + di2 b, grad1 = di1 a + di3 b
              if (OP == OP_LAP_TENSOR) {
                const double2 c = __ldg(reinterpret_cast<const double2*>(A.tensorvisc + ge * 64 + (r * 4 + j) * 4));
                const double2 d = __ldg(reinterpret_cast<const double2*>(A.tensorvisc + ge * 64 + (r * 4 + j) * 4 + 2));
                const double u00 = fma(c.x, t00, c.y * t10), u01 = fma(c.x, t01, c.y * t11);
                const double u10 = fma(d.x, t00, d.y * t10), u11 = fma(d.x, t01, d.y * t11);
                t00 = u00; t01 = u01; t10 = u10; t11 = u11;
              }
              const double sc = mpr[j] * A.rrearth;
              nm[j][0] = sc * fma(a.x, t00, a.y * t10);
              nm[j][1] = sc * fma(a.x, t01, a.y * t11);
              nm[j][2] = sc * fma(b.x, t00, b.y * t10);
              nm[j][3] = sc * fma(b.x, t01, b.y * t11);
            }
          }
        }
      }
      if (OP == OP_EULER) {
        mbar_wait(&item_full[item_k & 1], (item_k >> 1) & 1);
        Row us, vs;
        ld_tile2(reinterpret_cast<const double*>(item_tiles + (item_k & 1) * ITEM_B), sw2, us, vs);
        __syncwarp();  // every lane has read the vstar tile: its buffer may be refilled (two items ahead)
        if (lane == 0 && items_left > 0) issue_item(item_k + 2);
        double w1[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {  // (w1, w2) = metdet Dinv vstar
          const double2 p0 = *reinterpret_cast<const double2*>(geo + r * 20 + j * 4);
          const double2 p1 = *reinterpret_cast<const double2*>(geo + r * 20 + j * 4 + 2);
          w1[j] = fma(p0.x, us.x[j], p0.y * vs.x[j]);
          w2[j] = fma(p1.x, us.x[j], p1.y * vs.x[j]);
        }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const double wx = x == 0 ? w1[j] : __shfl_xor_sync(FULL, w1[j], x);  // w1(r^x, j)
            Ac[x][j] = rm[j] * (cx[x] * wx);
          }
      }
    }
    // position of the next unit, and whether it starts a new item / element
    advance(cur);
    new_item = cur.iq == 0;
    new_elem = new_item && cur.g == 0;

    const int s = i % NS;
    mbar_wait(&full[s], (i / NS) & 1);
    const unsigned char* tile = in_tiles + s * IN_B;
    Row out;
    if (OP == OP_EULER) {
      Row q[4];  // the level's 16 tracer values: row m = chunks 2m, 2m+1 of the 128-byte tile row
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        const int m = r ^ x;
        const uint32_t o = (uint32_t)lvl * 128u + ((uint32_t)((2 * m) ^ (lvl & 7)) << 4);
        q[x] = ld_tile(reinterpret_cast<const double*>(tile), o);
      }
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(NO - 1) : "memory");
      __syncwarp();  // stage s is consumed by every lane; the output tile i % NO is free
      if (lane == 0 && i + NS < n) issue_in(i + NS);
      double g1[4];  // this row's flux along jgp
#pragma unroll
      for (int m = 0; m < 4; ++m) g1[m] = w2[m] * q[0].x[m];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        double dvdy = A.dvv[0 * 4 + j] * g1[0];
#pragma unroll
        for (int m = 1; m < 4; ++m) dvdy = fma(A.dvv[m * 4 + j], g1[m], dvdy);
        double acc = fma(rm[j], dvdy, q[0].x[j]);
#pragma unroll
        for (int x = 0; x < 4; ++x) acc = fma(Ac[x][j], q[x].x[j], acc);
        out.x[j] = acc;
      }
    } else {
      Row g0, g1;  // the vector the point-local matrix is applied to: v, or the raw derivatives of the scalar
      if (OP == OP_DIVWK) {
        ld_tile2(reinterpret_cast<const double*>(tile), sw2, g0, g1);
      } else {
        const Row sc = ld_tile(reinterpret_cast<const double*>(tile), sw1);
        g0 = deriv_i(sc, cx);     // sum_m Dvv[m][r] s(m,j)   (PO/sphere_operators.cpp:21-35)
        g1 = deriv_j(sc, A.dvv);  // sum_m Dvv[m][j] s(r,m)
      }
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(NO - 1) : "memory");
      __syncwarp();
      if (lane == 0 && i + NS < n) issue_in(i + NS);
      // divergence_sphere_wk of s = N . g:  div(r,n) = -(sum_j Dvv[r][j] s0(j,n) + sum_j Dvv[n][j] s1(r,j))
      Row s0, s1;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s0.x[j] = fma(nm[j][0], g0.x[j], nm[j][1] * g1.x[j]);
        s1.x[j] = fma(nm[j][2], g0.x[j], nm[j][3] * g1.x[j]);
      }
#pragma unroll
      for (int nn = 0; nn < 4; ++nn) {
        double acc = cr[0] * s0.x[nn];
#pragma unroll
        for (int x = 1; x < 4; ++x) acc = fma(cr[x], __shfl_xor_sync(FULL, s0.x[nn], x), acc);
#pragma unroll
        for (int j = 0; j < 4; ++j) acc = fma(A.dvv[nn * 4 + j], s1.x[j], acc);
        out.x[nn] = -acc;
      }
    }
    unsigned char* otile = out_tiles + (i % NO) * OUT_B;
    st_tile(reinterpret_cast<double*>(otile), sw1, out);
    fence_proxy_async();
    __syncwarp();  // the output tile is complete and visible to the TMA engine
    if (lane == 0) {
      tma_store(&M.out, lev0, OP == OP_EULER ? (e * A.qsize_d + iq) * A.out_stride + A.out_off : e, otile);
      bulk_commit();
    }
  }
  if (lane == 0) bulk_wait_read_all();  // shared memory must outlive the last bulk stores
}

// ---- laplace_simple / laplace_tensor, second generation: ONE THREAD PER LEVEL ------------------------------------
// The row decomposition above spends most of its issue slots and LSU wavefronts on moving the 16 values of a level
// between its four threads (48 SHFL.32 + 4 LDS/STS.128 per thread and tile, against 80 DFMA). Here a thread owns all 16
// points of one level: its 128-byte row of the swizzled tile is 8 conflict-free LDS.128, both derivatives and the weak
// divergence are thread-local (320 DFMA, no shuffle), and the point-local 2x2 matrices N come from a per-warp
// shared-memory cache read with broadcast LDS.128. The element x level rows of [nets,nete) are ONE flat list (the
// scalar arrays are [E][L][16] without padding), cut into tiles of 32 rows = 4 KB = one warp step, so every lane is busy
// whatever nlev is; a tile may span several elements (at most 3 for nlev >= 16), each lane picks the cache slot of its own
// element. The geometry of new elements is loaded into registers two tiles ahead and turned into N one tile ahead, after
// the math (loaded on demand, a quarter of all warp stall samples sat on those loads; one tile ahead, still 7 %: under
// load a line takes longer than a tile's math). Same per-warp TMA pipeline as above (FN input tiles ahead, FO output
// tiles draining); the tiles themselves are drawn in chunks from a global counter (see the kernel).
#ifndef LAPFLAT_NS
#define LAPFLAT_NS 3
#endif
#ifndef LAPFLAT_NO
#define LAPFLAT_NO 2
#endif
#ifndef LAPFLAT_WPC
#define LAPFLAT_WPC 4
#endif
#ifndef LAPFLAT_MINB
#define LAPFLAT_MINB 2
#endif
static_assert(LAPFLAT_NS >= 3, "the geometry stages look two tiles ahead in the ring of tile numbers");
constexpr int FN = LAPFLAT_NS, FO = LAPFLAT_NO, FW = LAPFLAT_WPC;
constexpr int FT = 32;            // rows (element x level) per tile
constexpr unsigned FT_B = 4096u;  // bytes of a tile
constexpr int FSLOT = 8;          // cached elements per warp (slot = element & 7): <= 3 of this tile + <= 3 of the next
constexpr unsigned FWARP_B = (FN + FO) * FT_B + FSLOT * 512u;

struct LapFlatArgs {
  const double* Dinv;
  const double* spheremp;
  const double* tensorvisc;
  int nlev, nets;
  long long rows;   // (nete - nets) * nlev
  long long tiles;  // ceil(rows / 32)
  unsigned* sched;  // [0] next chunk, [1] warps done: both zero before and after a launch
  int chunk;        // tiles per chunk
  double rrearth;
  double dvv[16];
};
struct alignas(64) LapFlatMaps {
  CUtensorMap in, out;  // [1][rows][16 doubles] starting at element nets, box 32 rows
};

template <bool TENSOR>
__global__ void __launch_bounds__(32 * FW, LAPFLAT_MINB) laplace_flat_kernel(const __grid_constant__ LapFlatArgs A,
                                                                             const __grid_constant__ LapFlatMaps M) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* in_tiles = base + w * FWARP_B;
  unsigned char* out_tiles = in_tiles + FN * FT_B;
  double* ncache = reinterpret_cast<double*>(out_tiles + FO * FT_B);  // [FSLOT][16 points][4]
  uint64_t* full = reinterpret_cast<uint64_t*>(base + FW * FWARP_B) + w * FN;

  int* tq = reinterpret_cast<int*>(base + FW * FWARP_B + FW * FN * sizeof(uint64_t)) + w * FN;  // tile of each stage

  // Work distribution: the tiles are handed out in chunks of A.chunk consecutive tiles from a global counter (a static
  // cut into one range per warp left the early finishers idle: 0.84 of the measured peak against 0.95-0.98 with many
  // short CTAs, which in turn pay their pipeline fill each time). Lane 0 draws the NEXT chunk when the current one starts,
  // so the atomic's latency is never waited for; the stream of tiles feeds the TMA ring FN tiles ahead of the math.
  const int L = A.nlev, ntiles = (int)A.tiles, C = A.chunk, nchunks = (ntiles + C - 1) / C;
  const int nwarps = (int)gridDim.x * FW;
  unsigned pend = 0;
  if (lane == 0) pend = atomicAdd(A.sched, 1u);
  int gen = 0, gen_end = 0;
  bool exhausted = false, first = true;
  auto next_tile = [&]() -> int {  // uniform over the warp
    if (gen == gen_end) {
      if (exhausted) return -1;
      int c = (int)blockIdx.x * FW + w;  // the first chunk of a warp is its own number: no round trip before the first load
      if (!first) {
        c = nwarps + (int)__shfl_sync(FULL, pend, 0);
        if (lane == 0 && c < nchunks) pend = atomicAdd(A.sched, 1u);
      }
      first = false;
      if (c >= nchunks) {
        exhausted = true;
        return -1;
      }
      gen = c * C;
      gen_end = gen + C < ntiles ? gen + C : ntiles;
    }
    return gen++;
  };

  if (lane == 0) {
    for (int s = 0; s < FN; ++s) mbar_init(&full[s], 1);
    fence_proxy_async();
  }
  for (int s = 0; s < FN; ++s) {
    const int t = next_tile();
    if (lane == 0) {
      tq[s] = t;
      if (t >= 0) {
        mbar_expect_tx(&full[s], FT_B);
        tma_load(in_tiles + s * FT_B, &M.in, t * FT, 0, &full[s]);
      }
    }
  }
  __syncwarp();

  const double inv_l = 1.0 / (double)L;
  auto pos_of = [&](int tile, int& e, int& k) {  // (element, level) of a tile's first row; exact: (row + 1/2)/L is at
    const int row = tile * FT;                   // least 1/(2L) away from an integer
    e = __double2int_rd(((double)row + 0.5) * inv_l);
    k = row - e * L;
  };
  const int e_max = (int)((A.rows - 1) / L);  // last element of the range (relative to nets)
  int filled = -1;                            // elements <= filled are (or were) in the cache
  const uint32_t swz = (uint32_t)lane * 128u;
  const uint32_t x7 = (uint32_t)(lane & 7);

  // the element's geometry as loaded (lanes 0-15 / 16-31: point lane & 15 of one element each) and its N into the cache
  struct Geo {
    double2 a, b, c, d;
    double mp;
  };
  const int pt = lane & 15, half = lane >> 4;
  auto load_geo = [&](int e) {
    Geo g;
    const size_t ge = (size_t)(A.nets + e);
    g.a = __ldg(reinterpret_cast<const double2*>(A.Dinv + ge * 64 + pt * 4));
    g.b = __ldg(reinterpret_cast<const double2*>(A.Dinv + ge * 64 + pt * 4 + 2));
    g.mp = __ldg(A.spheremp + ge * 16 + pt);
    if (TENSOR) {
      g.c = __ldg(reinterpret_cast<const double2*>(A.tensorvisc + ge * 64 + pt * 4));
      g.d = __ldg(reinterpret_cast<const double2*>(A.tensorvisc + ge * 64 + pt * 4 + 2));
    }
    return g;
  };
  auto store_n = [&](int e, const Geo& g) {  // N = spheremp rrearth^2 Dinv [tensorVisc] Dinv^T (see levelop_kernel)
    double t00 = g.a.x, t01 = g.b.x, t10 = g.a.y, t11 = g.b.y;
    if (TENSOR) {
      const double u00 = fma(g.c.x, t00, g.c.y * t10), u01 = fma(g.c.x, t01, g.c.y * t11);
      const double u10 = fma(g.d.x, t00, g.d.y * t10), u11 = fma(g.d.x, t01, g.d.y * t11);
      t00 = u00; t01 = u01; t10 = u10; t11 = u11;
    }
    const double sc = g.mp * A.rrearth * A.rrearth;
    double* dst = ncache + (e & (FSLOT - 1)) * 64 + pt * 4;
    *reinterpret_cast<double2*>(dst) = make_double2(sc * fma(g.a.x, t00, g.a.y * t10), sc * fma(g.a.x, t01, g.a.y * t11));
    *reinterpret_cast<double2*>(dst + 2) = make_double2(sc * fma(g.b.x, t00, g.b.y * t10), sc * fma(g.b.x, t01, g.b.y * t11));
  };
  auto last_of_tile = [&](int e0, int k0) {  // last element a 32-row tile starting at (e0, k0) touches
    int k = k0 + FT - 1;
    while (k >= L) k -= L, ++e0;
    return e0 < e_max ? e0 : e_max;
  };

  // Two stages of geometry in registers, one element per half warp each: `gb` = the first two new elements of the next
  // tile (N stored after this tile's math), `ga` = those of the tile after it (loaded at the top of this iteration).
  // `queued` = last element loaded into a stage. What the stages do not cover (the warp's first tile; a third new element
  // after a jump when nlev < 32) is loaded on demand.
  Geo ga, gb;
  int ga_e = 0, gb_e = 0, gb_hi = -1, ga_hi = -1;
  bool ga_ok = false, gb_ok = false;
  int queued = -1;
  auto stage = [&](int t, Geo& g, int& g_e, int& g_hi, bool& g_ok) {  // new elements of tile t (t < 0: none)
    g_ok = false;
    g_hi = -1;
    if (t < 0) return;
    int e, k;
    pos_of(t, e, k);
    const int last = last_of_tile(e, k);
    const int lo = queued > e - 1 ? queued : e - 1;
    g_e = lo + 1 + half;
    g_ok = g_e <= last;
    if (g_ok) g = load_geo(g_e);
    g_hi = lo + 2 < last ? lo + 2 : last;
    if (queued < g_hi) queued = g_hi;
  };

  for (int i = 0;; ++i) {
    const int s = i % FN;
    const int tile_id = tq[s];
    if (tile_id < 0) break;  // uniform
    const int t1 = tq[(i + 1) % FN], t2 = tq[(i + 2) % FN];
    int e_first, k_first;
    pos_of(tile_id, e_first, k_first);
    // this lane's element (relative) and the last element the tile touches
    int e_t = e_first, kk = k_first + lane;
    while (kk >= L) kk -= L, ++e_t;
    if (e_t > e_max) e_t = e_max;  // rows beyond the range: zero-filled input, clipped output
    const int e_last = last_of_tile(e_first, k_first);
    if (filled < e_first - 1) filled = e_first - 1;
    while (filled < e_last) {  // not staged: on demand. Uniform over the warp.
      const int e = filled + 1 + half;
      if (e <= e_last) store_n(e, load_geo(e));
      filled = filled + 2 < e_last ? filled + 2 : e_last;
      __syncwarp();
    }
    if (queued < filled) queued = filled;
    if (i == 0) stage(t1, gb, gb_e, gb_hi, gb_ok);  // nothing was loaded for the second tile yet
    stage(t2, ga, ga_e, ga_hi, ga_ok);

    mbar_wait(&full[s], (i / FN) & 1);
    const unsigned char* tile = in_tiles + s * FT_B + swz;
    double sv[16];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const double2 v = *reinterpret_cast<const double2*>(tile + (((uint32_t)c ^ x7) << 4));
      sv[2 * c] = v.x;
      sv[2 * c + 1] = v.y;
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(FO - 1) : "memory");
    __syncwarp();  // stage s is consumed by every lane; the output tile i % FO is free
    {
      const int t = next_tile();
      if (lane == 0) {
        tq[s] = t;
        if (t >= 0) {
          mbar_expect_tx(&full[s], FT_B);
          tma_load(in_tiles + s * FT_B, &M.in, t * FT, 0, &full[s]);
        }
      }
    }
    unsigned char* otile = out_tiles + (i % FO) * FT_B;
#if defined(LAPFLAT_DIAG_COPY)  // development: the pipeline without the math
#pragma unroll
    for (int c = 0; c < 8; ++c)
      *reinterpret_cast<double2*>(otile + swz + (((uint32_t)c ^ x7) << 4)) = make_double2(sv[2 * c], sv[2 * c + 1] + (double)e_t);
#else
    // raw derivatives: g0(i,j) = sum_m Dvv[m][i] s(m,j), g1(i,j) = sum_m Dvv[m][j] s(i,m); then s = N g in place
    double g0[16], g1[16];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        double x = A.dvv[0 * 4 + a] * sv[0 * 4 + b], y = A.dvv[0 * 4 + b] * sv[a * 4 + 0];
#pragma unroll
        for (int m = 1; m < 4; ++m) {
          x = fma(A.dvv[m * 4 + a], sv[m * 4 + b], x);
          y = fma(A.dvv[m * 4 + b], sv[a * 4 + m], y);
        }
        g0[a * 4 + b] = x;
        g1[a * 4 + b] = y;
      }
    const double* nc = ncache + (e_t & (FSLOT - 1)) * 64;
#pragma unroll
    for (int p = 0; p < 16; ++p) {
      const double2 n01 = *reinterpret_cast<const double2*>(nc + p * 4);
      const double2 n23 = *reinterpret_cast<const double2*>(nc + p * 4 + 2);
      const double x = g0[p], y = g1[p];
      g0[p] = fma(n01.x, x, n01.y * y);
      g1[p] = fma(n23.x, x, n23.y * y);
    }
    // weak divergence: out(i,j) = -(sum_m Dvv[i][m] s0(m,j) + sum_m Dvv[j][m] s1(i,m))
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      double o[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int a = c >> 1, b = 2 * (c & 1) + h;
        double acc = A.dvv[a * 4 + 0] * g0[0 * 4 + b];
#pragma unroll
        for (int m = 1; m < 4; ++m) acc = fma(A.dvv[a * 4 + m], g0[m * 4 + b], acc);
#pragma unroll
        for (int m = 0; m < 4; ++m) acc = fma(A.dvv[b * 4 + m], g1[a * 4 + m], acc);
        o[h] = -acc;
      }
      *reinterpret_cast<double2*>(otile + swz + (((uint32_t)c ^ x7) << 4)) = make_double2(o[0], o[1]);
    }
#endif
    __syncwarp();  // after a jump the staged elements may take the cache slots this tile was reading
    if (gb_ok) store_n(gb_e, gb);
    if (filled < gb_hi) filled = gb_hi;
    gb = ga; gb_e = ga_e; gb_hi = ga_hi; gb_ok = ga_ok;
    fence_proxy_async();
    __syncwarp();  // the output tile is complete and visible to the TMA engine; so is the cache to the next tile
    if (lane == 0) {
      tma_store(&M.out, tile_id * FT, 0, otile);
      bulk_commit();
    }
  }
  if (lane == 0) {
    bulk_wait_read_all();  // shared memory must outlive the last bulk stores
    // the last warp of the grid to get here leaves the scheduler's counters at zero for the next launch
    __threadfence();
    const unsigned done = atomicAdd(A.sched + 1, 1u);
    if (done == gridDim.x * FW - 1) {
      A.sched[0] = 0;
      A.sched[1] = 0;
    }
  }
}

// ---- CAAR_MODE_STRICT: the reference's operation order, one thread per point, 16 levels per CTA ------------------
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }

struct StrictWkArgs {
  const double* Dinv;
  const double* spheremp;
  const double* tensorvisc;
  const double* vin;   // [E][L][16][2]
  const double* sin;   // [E][L][16]
  double* out;         // [E][L][16]
  int nlev, nets, nelem_run, op;
  double rrearth;
  double dvv[16];
};

__global__ void __launch_bounds__(256) sphere_wk_strict_kernel(const StrictWkArgs A) {
  __shared__ double g[16][16][2];  // per level of this CTA: the vector field the weak divergence is taken of
  __shared__ double sc[16][16];
  const int t = threadIdx.x, kl = t >> 4, q = t & 15, i = q >> 2, j = q & 3;
  const long long rows = (long long)A.nelem_run * A.nlev;
  const long long gk0 = (long long)blockIdx.x * 16 + kl;
  const bool live = gk0 < rows;
  const long long gk = live ? gk0 : rows - 1;
  const size_t e = (size_t)A.nets + (size_t)(gk / A.nlev);
  const size_t n = (e * A.nlev + (size_t)(gk % A.nlev)) * 16;
  const double* dinv = A.Dinv + e * 64;
  if (A.op == 0) {
    g[kl][q][0] = A.vin[(n + q) * 2];
    g[kl][q][1] = A.vin[(n + q) * 2 + 1];
  } else {
    sc[kl][q] = A.sin[n + q];
  }
  __syncthreads();
  if (A.op != 0) {  // gradient_sphere at point (i,j) in the reference's order (PO/sphere_operators.cpp:21-47)
    double sx = 0.0, sy = 0.0;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      sx = add(sx, mul(A.dvv[m * 4 + i], sc[kl][m * 4 + j]));
      sy = add(sy, mul(A.dvv[m * 4 + j], sc[kl][i * 4 + m]));
    }
    const double a = mul(sx, A.rrearth), b = mul(sy, A.rrearth);
    const double* di = dinv + q * 4;
    double g0 = add(mul(di[0], a), mul(di[2], b));
    double g1 = add(mul(di[1], a), mul(di[3], b));
    if (A.op == 2) {  // tensorVisc . grad (LV/SphereOperators.hpp:574-585)
      const double* tv = A.tensorvisc + e * 64 + q * 4;
      const double x0 = g0, x1 = g1;
      g0 = add(mul(tv[0], x0), mul(tv[1], x1));
      g1 = add(mul(tv[2], x0), mul(tv[3], x1));
    }
    g[kl][q][0] = g0;
    g[kl][q][1] = g1;
  }
  __syncthreads();
  // divergence_sphere_wk at point (m,n) = (i,j) (LV/SphereOperators.hpp:493-535)
  const double* mp = A.spheremp + e * 16;
  double dd = 0.0;
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    const int pa = jj * 4 + j, pb = i * 4 + jj;  // points (jj, n) and (m, jj)
    const double ta = add(mul(dinv[pa * 4 + 0], g[kl][pa][0]), mul(dinv[pa * 4 + 1], g[kl][pa][1]));
    const double tb = add(mul(dinv[pb * 4 + 2], g[kl][pb][0]), mul(dinv[pb * 4 + 3], g[kl][pb][1]));
    const double term = mul(add(mul(mul(mp[pa], ta), A.dvv[i * 4 + jj]), mul(mul(mp[pb], tb), A.dvv[j * 4 + jj])), A.rrearth);
    dd = __dsub_rn(dd, term);
  }
  if (live) A.out[n + q] = dd;
}

int encode3(CUtensorMap* m, const void* base, cuuint64_t slices, cuuint64_t rows, cuuint32_t box_rows) {
  typedef CUresult (*encode_t)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static encode_t encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) return 1;
    encode = reinterpret_cast<encode_t>(fn);
  }
  const cuuint64_t gdim[3] = {16, rows, slices};
  const cuuint64_t gstride[2] = {128, rows * 128};
  const cuuint32_t box[3] = {16, box_rows, 1};
  const cuuint32_t estride[3] = {1, 1, 1};
  return encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<void*>(base), gdim, gstride, box, estride,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS ? 0 : 1;
}

template <int OP>
cudaError_t launch_op(const LevelOpArgs& a, const LevelOpMaps& m, cudaStream_t s) {
  const unsigned in_b = (OP == OP_DIVWK) ? 2048u : 1024u, item_b = (OP == OP_EULER) ? 2048u : 0u;
  const size_t smem = (size_t)WPC * (NS * in_b + NO * 1024u + 2 * item_b) + WPC * (NS + 2) * sizeof(uint64_t) +
                      WPC * 80 * sizeof(double) + 1024;
  // function attributes and occupancy are per (instance, device): set / queried once
  static int cached_per_sm[64] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  int per_sm = (dev >= 0 && dev < 64) ? cached_per_sm[dev] : 0;
  if (per_sm == 0) {
    e = cudaFuncSetAttribute(levelop_kernel<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(levelop_kernel<OP>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, levelop_kernel<OP>, 32 * WPC, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    if (dev >= 0 && dev < 64) cached_per_sm[dev] = per_sm;
  }
  // grid = waves x the resident CTAs. A static cut into one range per resident warp (1 wave) leaves the early finishers
  // idle, many short CTAs pay their pipeline fill more often; the best number of waves grows with the size (tracer step,
  // qsize 4: 1-2 at 5400 elements, 6-8 at 21600, 16 at 86400; divergence_sphere_wk: 1 / 8 / 16 — profiles/README.md):
  // about 48 (tracer step) / 12 (weak-form operators) units per warp and CTA, at most 16 waves
  static const int waves_env = [] { const char* v = getenv("CAAR_LEVELOP_WAVES"); return v ? atoi(v) : 0; }();
  const long long per_wave = (long long)sm_count() * per_sm * WPC * (OP == OP_EULER ? 48 : 12);
  long long wv = (a.units + per_wave / 2) / per_wave;
  wv = (wv < 1 || OP == OP_LAP_SIMPLE || OP == OP_LAP_TENSOR) ? 1 : wv > 16 ? 16 : wv;  // row-decomposed laplacians (nlev < 16): 1
  const int waves = waves_env > 0 ? waves_env : (int)wv;
  long long blocks = (long long)sm_count() * per_sm * waves;
  const long long need = (a.units + WPC - 1) / WPC;
  if (blocks > need) blocks = need;
  levelop_kernel<OP><<<(unsigned)blocks, 32 * WPC, smem, s>>>(a, m);
  return cudaGetLastError();
}

template <bool TENSOR>
cudaError_t launch_lapflat(LapFlatArgs a, const LapFlatMaps& m, cudaStream_t s) {
  const size_t smem = (size_t)FW * FWARP_B + FW * FN * (sizeof(uint64_t) + sizeof(int)) + 1024;
  static int cached_per_sm[64] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  int per_sm = cached_per_sm[dev];
  if (per_sm == 0) {
    e = cudaFuncSetAttribute(laplace_flat_kernel<TENSOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(laplace_flat_kernel<TENSOR>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, laplace_flat_kernel<TENSOR>, 32 * FW, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    cached_per_sm[dev] = per_sm;
  }
  // one wave of resident CTAs; chunks of 4 consecutive tiles (49152 x 128: 0.81 / 0.98 / 1.01 / 0.99 / 0.95 / 0.90 of the
  // measured peak with 1 / 2 / 4 / 8 / 16 / 32; one tile per chunk exposes the draw), 2 when a warp sees few tiles
  static const int chunk_env = [] { const char* v = getenv("CAAR_LAPLACE_CHUNK"); return v ? atoi(v) : 0; }();
  const long long resident_warps = (long long)sm_count() * per_sm * FW;
  a.chunk = chunk_env > 0 ? chunk_env : (a.tiles < resident_warps * 16 ? 2 : 4);
  long long blocks = (long long)sm_count() * per_sm;
  const long long need = (a.tiles + FW - 1) / FW;
  if (blocks > need) blocks = need;
  laplace_flat_kernel<TENSOR><<<(unsigned)blocks, 32 * FW, smem, s>>>(a, m);
  return cudaGetLastError();
}

}  // namespace

// Level-local operator on elements [nets,nete). op: 0 tracer step (in = Qdp mirror, item = vstar, out = qtens or
// Qdp), 1 divergence_sphere_wk (in = vector [E][L][16][2]), 2 laplace_simple, 3 laplace_tensor (in = scalar
// [E][L][16]); out [E][L][16] (tracer step: [slice][L][16], tracer iq of element e at slice (e * qsize_d + iq) *
// out_stride + out_off; other ops ignore the two). in == out is allowed for 2 and 3 (the reference's *_replace) and
// for 0 with (2, qn0) (a stage of caar_advect_tracers).
cudaError_t launch_levelop(int op, const KernelArgs& k, const double* in, const double* item, double* out,
                           const double* tensorvisc, int nets, int nete, int qn0, int qsize, double dt, int out_stride,
                           int out_off, bool strict, cudaStream_t s) {
  if (nete <= nets || (op == 0 && qsize <= 0)) return cudaSuccess;
  if (strict) {
    if (op == 0) return cudaErrorInvalidValue;  // the strict tracer step lives in caar_euler.cu
    StrictWkArgs a;
    a.Dinv = k.Dinv; a.spheremp = k.spheremp; a.tensorvisc = tensorvisc; a.vin = in; a.sin = in; a.out = out;
    a.nlev = k.nlev; a.nets = nets; a.nelem_run = nete - nets; a.op = op - 1; a.rrearth = k.rrearth;
    for (int i = 0; i < 16; ++i) a.dvv[i] = k.dvv[i];
    const long long rows = (long long)(nete - nets) * k.nlev;
    sphere_wk_strict_kernel<<<(unsigned)((rows + 15) / 16), 256, 0, s>>>(a);
    return cudaGetLastError();
  }
  static const bool lap_v1 = [] { const char* v = getenv("CAAR_LAPLACE_V1"); return v && atoi(v) != 0; }();
  const long long flat_rows = (long long)(nete - nets) * k.nlev;
  if (op >= 2 && !lap_v1 && k.nlev >= 16 && flat_rows + FT < (1ll << 31)) {  // thread-per-level laplacians
    LapFlatArgs a;
    a.Dinv = k.Dinv; a.spheremp = k.spheremp; a.tensorvisc = tensorvisc;
    a.nlev = k.nlev; a.nets = nets; a.rows = flat_rows; a.tiles = (flat_rows + FT - 1) / FT; a.rrearth = k.rrearth;
    // the calling handle's scheduler pair: launches of other handles, on other streams, never touch it
    a.sched = k.lapflat_sched;
    if (!a.sched) return cudaErrorInvalidValue;
    for (int i = 0; i < 16; ++i) a.dvv[i] = k.dvv[i];
    LapFlatMaps m;
    const size_t off = (size_t)nets * k.nlev * 16;
    if (encode3(&m.in, in + off, 1, (cuuint64_t)flat_rows, FT) | encode3(&m.out, out + off, 1, (cuuint64_t)flat_rows, FT))
      return cudaErrorInvalidValue;
    return op == 2 ? launch_lapflat<false>(a, m, s) : launch_lapflat<true>(a, m, s);
  }
  LevelOpArgs a;
  a.Dinv = k.Dinv; a.metdet = k.metdet; a.rmetdet = k.rmetdet; a.spheremp = k.spheremp; a.tensorvisc = tensorvisc;
  a.nlev = k.nlev; a.nets = nets; a.qn0 = qn0; a.qsize_d = k.qsize_d; a.dt = dt; a.rrearth = k.rrearth;
  a.out_stride = out_stride; a.out_off = out_off;
  for (int i = 0; i < 16; ++i) a.dvv[i] = k.dvv[i];
  a.ngroups = (k.nlev + GL - 1) / GL;  // groups of 8 levels; the last one may stick out of the column (zero-filled / clipped)
  a.Q = op == 0 ? qsize : 1;
  a.units = (long long)(nete - nets) * a.ngroups * a.Q;
  LevelOpMaps m;
  const cuuint64_t E = (cuuint64_t)k.nelem, L = (cuuint64_t)k.nlev;
  int bad = 0;
  if (op == 0) {
    bad |= encode3(&m.in, in, E * (cuuint64_t)k.qsize_d * 2, L, GL);
    bad |= encode3(&m.item, item, E, 2 * L, 2 * GL);
    bad |= encode3(&m.out, out, E * (cuuint64_t)k.qsize_d * (cuuint64_t)out_stride, L, GL);
  } else {
    bad |= encode3(&m.in, in, E, op == 1 ? 2 * L : L, op == 1 ? 2 * GL : GL);
    bad |= encode3(&m.out, out, E, L, GL);
    m.item = m.in;
  }
  if (bad) return cudaErrorInvalidValue;
  switch (op) {
    case 0: return launch_op<OP_EULER>(a, m, s);
    case 1: return launch_op<OP_DIVWK>(a, m, s);
    case 2: return launch_op<OP_LAP_SIMPLE>(a, m, s);
    case 3: return launch_op<OP_LAP_TENSOR>(a, m, s);
  }
  return cudaErrorInvalidValue;
}

}  // namespace caar
