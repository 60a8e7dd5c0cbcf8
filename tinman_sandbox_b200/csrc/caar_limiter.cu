// caar_limiter.cu — HOMME's quasi-monotone tracer limiter (euler_step with limiter_option == 8) on the resident Qdp:
//   * caar_tracer_bounds: the element-local bounds (qmin, qmax) of Qdp/dp3d per element, tracer and level;
//   * caar_limit_tracers: limiter_optim_iter_full on each (element, tracer, level) with weights spheremp * dp3d.
// The algorithm is specified in include/caar_b200.h; both kernels restate it operation for operation (every operation
// rounded separately, sums sequential in Fortran point order), so their results are bit-reproducible and equal the FP64
// restatement of tests/limiter_oracle.py.
//
// Shape: one thread per problem (e, iq, k), the 16 x and c of its level in registers. The rows of a warp are 32
// consecutive problems of the flat list [nets, nete) x [0, qsize) x [0, L) — consecutive levels of one tracer are
// consecutive 128 B rows of Qdp and dp3d — so the warp stages its 32 rows of each through shared memory with loads in
// which every half-warp reads one whole row (coalesced), and each thread then reads its own row from there. Rows are
// padded to 17 doubles, so that 16 threads reading the same column of 16 rows hit 16 different bank pairs. The limited
// Qdp goes back the same way. Warps walk the tiles of 32 problems with a grid stride; the grid is one wave of resident
// CTAs, or fewer when there are fewer tiles.
#include "caar_device.cuh"

namespace caar {

namespace {

constexpr int LIM_WARPS = 8;    // warps per CTA
constexpr int LIM_ROW = 17;     // padded row of one problem in shared memory, doubles
constexpr int LIM_MAXITER = 15;  // np*np - 1
constexpr double LIM_TOL = 5e-14;
constexpr size_t LIM_SMEM = (size_t)LIM_WARPS * 2 * 32 * LIM_ROW * sizeof(double);

struct LimiterArgs {
  double* Qdp;               // [E][qsize_d][2][L][16]
  const double* dp3d;        // [E][ntl][L][16]
  const double* spheremp;    // [E][16]
  double2* bounds;           // [E][qsize_d][L] of (min, max)
  unsigned long long nprob;  // (nete - nets) * qsize * L
  int L, qsize, qsize_d, ntl, nets, qtl, dp_tl;
};

// C offset 4*igp + jgp of the m-th point in Fortran sequence-association order (i = igp fastest)
__device__ __forceinline__ int fortran_point(int m) { return 4 * (m & 3) + (m >> 2); }

// LIMIT = false: the bounds (caar_tracer_bounds); LIMIT = true: the limiter (caar_limit_tracers)
template <bool LIMIT>
__global__ void __launch_bounds__(LIM_WARPS * 32, 2) limiter_kernel(const LimiterArgs A) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* qs = smem + warp * (2 * 32 * LIM_ROW);  // the warp's 32 rows of Qdp(qtl)
  double* ds = qs + 32 * LIM_ROW;                 // and of dp3d(dp_tl)
  const unsigned long long ntiles = (A.nprob + 31) / 32;
  for (unsigned long long t = (unsigned long long)blockIdx.x * LIM_WARPS + warp; t < ntiles;
       t += (unsigned long long)gridDim.x * LIM_WARPS) {
    const unsigned long long p = t * 32 + lane;
    const bool live = p < A.nprob;
    // row indices in units of 16 doubles: Qdp holds fewer than 2^32 rows of 128 B on any device
    unsigned qrow = 0, drow = 0, brow = 0, e = 0;
    if (live) {
      const unsigned long long r = p / A.L;
      const unsigned k = (unsigned)(p - r * A.L);
      const unsigned iq = (unsigned)(r % A.qsize);
      e = A.nets + (unsigned)(r / A.qsize);
      brow = (e * A.qsize_d + iq) * A.L + k;
      qrow = ((e * A.qsize_d + iq) * 2 + A.qtl) * A.L + k;
      drow = (e * A.ntl + A.dp_tl) * A.L + k;
    }
    double2 b = make_double2(0.0, 0.0);
    if (LIMIT && live) b = A.bounds[brow];
    const int col = lane & 15;
#pragma unroll
    for (int j = 0; j < 16; ++j) {  // rows 2j and 2j+1, one per half-warp
      const int r = 2 * j + (lane >> 4);
      const unsigned qr = __shfl_sync(0xffffffffu, qrow, r), dr = __shfl_sync(0xffffffffu, drow, r);
      if (t * 32 + r < A.nprob) {
        qs[r * LIM_ROW + col] = A.Qdp[(size_t)qr * 16 + col];
        ds[r * LIM_ROW + col] = __ldg(A.dp3d + (size_t)dr * 16 + col);
      }
    }
    __syncwarp();
    if (live) {
      const double* qv = qs + lane * LIM_ROW;
      const double* dv = ds + lane * LIM_ROW;
      double x[16];
#pragma unroll
      for (int m = 0; m < 16; ++m) x[m] = __ddiv_rn(qv[fortran_point(m)], dv[fortran_point(m)]);
      if (!LIMIT) {
        double qmin = x[0], qmax = x[0];
#pragma unroll
        for (int m = 1; m < 16; ++m) {
          if (x[m] < qmin) qmin = x[m];
          if (x[m] > qmax) qmax = x[m];
        }
        if (qmin < 0.0) qmin = 0.0;
        A.bounds[brow] = make_double2(qmin, qmax);
      } else {
        const double* w = A.spheremp + (size_t)e * 16;
        double c[16], sumc = 0.0;
#pragma unroll
        for (int m = 0; m < 16; ++m) {
          c[m] = __dmul_rn(__ldg(w + fortran_point(m)), dv[fortran_point(m)]);
          sumc = __dadd_rn(sumc, c[m]);
        }
        if (!(sumc <= 0.0)) {  // sumc <= 0: the problem (Qdp and its bounds) stays as it is
          double minp = b.x, maxp = b.y, mass = 0.0;
#pragma unroll
          for (int m = 0; m < 16; ++m) mass = __dadd_rn(mass, __dmul_rn(c[m], x[m]));
          // relax the bounds so that a solution exists
          if (mass < __dmul_rn(minp, sumc)) minp = __ddiv_rn(mass, sumc);
          if (mass > __dmul_rn(maxp, sumc)) maxp = __ddiv_rn(mass, sumc);
          const double tol = __dmul_rn(LIM_TOL, fabs(mass));
#pragma unroll 1
          for (int it = 0; it < LIM_MAXITER; ++it) {
            double addmass = 0.0;
#pragma unroll
            for (int m = 0; m < 16; ++m) {
              if (x[m] > maxp) {
                addmass = __dadd_rn(addmass, __dmul_rn(__dsub_rn(x[m], maxp), c[m]));
                x[m] = maxp;
              }
              if (x[m] < minp) {
                addmass = __dsub_rn(addmass, __dmul_rn(__dsub_rn(minp, x[m]), c[m]));
                x[m] = minp;
              }
            }
            if (fabs(addmass) <= tol) break;
            // spread the clipped mass over the points that can still take it; ws == 0 can only follow rounding
            // (the relaxed bounds admit a solution), and the literal Fortran would divide by it
            const bool up = addmass > 0.0;
            double ws = 0.0;
#pragma unroll
            for (int m = 0; m < 16; ++m)
              if (up ? x[m] < maxp : x[m] > minp) ws = __dadd_rn(ws, c[m]);
            if (ws == 0.0) break;
            const double inc = __ddiv_rn(addmass, ws);
#pragma unroll
            for (int m = 0; m < 16; ++m)
              if (up ? x[m] < maxp : x[m] > minp) x[m] = __dadd_rn(x[m], inc);
          }
          double* qw = qs + lane * LIM_ROW;
#pragma unroll
          for (int m = 0; m < 16; ++m) qw[fortran_point(m)] = __dmul_rn(x[m], dv[fortran_point(m)]);
          A.bounds[brow] = make_double2(minp, maxp);
        }
      }
    }
    if (LIMIT) {
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int r = 2 * j + (lane >> 4);
        const unsigned qr = __shfl_sync(0xffffffffu, qrow, r);
        if (t * 32 + r < A.nprob) A.Qdp[(size_t)qr * 16 + col] = qs[r * LIM_ROW + col];
      }
    }
    __syncwarp();  // the next tile overwrites the rows
  }
}

template <bool LIMIT>
cudaError_t launch(const KernelArgs& a, int nets, int nete, int qtl, int qsize, int dp_tl, double* bounds,
                   cudaStream_t s) {
  if (nete <= nets || qsize <= 0) return cudaSuccess;
  static LaunchCache cache;
  int per_sm = 1;
  cudaError_t e = setup_launch(limiter_kernel<LIMIT>, LIM_WARPS * 32, LIM_SMEM, cache, &per_sm);
  if (e != cudaSuccess) return e;
  LimiterArgs A;
  A.Qdp = const_cast<double*>(a.Qdp);  // the handle's own mirror; const in KernelArgs for the kernels that read it
  A.dp3d = a.dp3d;
  A.spheremp = a.spheremp;
  A.bounds = reinterpret_cast<double2*>(bounds);
  A.nprob = (unsigned long long)(nete - nets) * qsize * a.nlev;
  A.L = a.nlev;
  A.qsize = qsize;
  A.qsize_d = a.qsize_d;
  A.ntl = a.ntl;
  A.nets = nets;
  A.qtl = qtl;
  A.dp_tl = dp_tl;
  const unsigned long long tiles = (A.nprob + 31) / 32;
  unsigned long long blocks = (tiles + LIM_WARPS - 1) / LIM_WARPS;
  const unsigned long long wave = (unsigned long long)per_sm * sm_count();
  if (blocks > wave) blocks = wave;
  limiter_kernel<LIMIT><<<(unsigned)blocks, LIM_WARPS * 32, LIM_SMEM, s>>>(A);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_tracer_bounds(const KernelArgs& a, int nets, int nete, int qtl, int qsize, int dp_tl, double* bounds,
                                 cudaStream_t s) {
  return launch<false>(a, nets, nete, qtl, qsize, dp_tl, bounds, s);
}

cudaError_t launch_limit_tracers(const KernelArgs& a, int nets, int nete, int qtl, int qsize, int dp_tl, double* bounds,
                                 cudaStream_t s) {
  return launch<true>(a, nets, nete, qtl, qsize, dp_tl, bounds, s);
}

}  // namespace caar
