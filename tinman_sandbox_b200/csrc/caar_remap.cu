// caar_remap.cu — HOMME's vertical remap for rsplit > 0 (vertical_remap with remap_Q_ppm, vert_remap_q_alg = 1) on
// the resident state: T and v of time level tl (remapped as T*dp_star and v*dp_star) and Qdp(qtl) of tracers
// iq < qsize, from the thicknesses dp_star = dp3d(tl) to those of the hybrid reference levels, then dp3d(tl) = dp. The
// algorithm is specified in include/caar_b200.h; the kernels restate it operation for operation (every operation
// rounded separately through the _rn intrinsics, sums sequential in k), so the results are bit-reproducible and equal
// the FP64 restatement of tests/remap_oracle.py.
//
// Shape: one thread per (column, batch of fields). A batch is the state (T, v0, v1) or REMAP_QB tracers. The 16 columns
// of an element are one 128 B row per level, so a warp (32 consecutive columns = two elements) reads two whole rows per
// load. The warp items are (group of 32 columns, batch) with the batch fastest, so the batches of one group run on
// neighbouring warps and share their dp3d reads in L1/L2. Warps walk the items with a grid stride over one wave.
//
// Per thread: a first pass sums dp_star into ps. The second pass walks the new levels k = 1..L once and pushes the old
// levels through a window in registers: after old level m is pushed, the window holds dx and a at m-3..m, pio and masso
// at m-2..m+1, and ai at m-3, m-2, so the PPM coefficients of cell j = m-2 are ready. kid(k) is non-decreasing, so one
// forward cursor serves every new level, and every old level is read once. The ghost cells are mirrored from the window:
// old levels L+1 and L+2 are copies of L and L-1 already in registers, never re-read (those rows may already hold new
// values). f(k) is written in place after level k+1 was read (kid(k) >= k-1 and the window runs two levels ahead), so
// no level is overwritten before it is read.
//
// dp3d(tl) is every batch's source, so the remap kernel does not write it: the state batch stores ps per column into a
// handle scratch [E][16], and a second launch, ordered after the first on the stream, writes dp3d(tl) = dp from ps.
#include "caar_device.cuh"

namespace caar {

namespace {

constexpr int REMAP_QB = 4;        // tracers per thread
constexpr int REMAP_WARPS = 4;     // warps per CTA
constexpr int REMAP_DP_THREADS = 256;

struct RemapArgs {
  double* dp3d;          // [E][ntl][L][16]
  double* v;             // [E][ntl][L][16][2]
  double* T;             // [E][ntl][L][16]
  double* Qdp;           // [E][qsize_d][2][L][16]
  const double* hyai;    // [L+1]
  const double* hybi;    // [L+1]
  double* ps;            // [E][16]: written by the state batch, read by the dp3d launch
  double ps0;
  unsigned long long nitems;  // warp items: groups of 32 columns x nbatch
  int L, ntl, qsize_d, nets, ncols, tl, qtl, qsize, nbatch;
};

__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dv(double a, double b) { return __ddiv_rn(a, b); }

// the state batch: f = (T, v0, v1) * dp_star in, (T, v0, v1) = f / dp out; p points at level 0 of the column
struct StateIO {
  static constexpr int NF = 3;
  double* T;
  double2* v;
  __device__ void load(int k, double dx, double* f) const {
    const double2 w = v[(size_t)k * 16];
    f[0] = mul(T[(size_t)k * 16], dx);
    f[1] = mul(w.x, dx);
    f[2] = mul(w.y, dx);
  }
  __device__ void store(int k, double dp, const double* f) const {
    T[(size_t)k * 16] = dv(f[0], dp);
    v[(size_t)k * 16] = make_double2(dv(f[1], dp), dv(f[2], dp));
  }
};

// a tracer batch: nf <= REMAP_QB tracers of Qdp(qtl), `stride` doubles apart; the mass itself is remapped
struct TracerIO {
  static constexpr int NF = REMAP_QB;
  double* q;
  size_t stride;
  int nf;
  __device__ void load(int k, double, double* f) const {
#pragma unroll
    for (int i = 0; i < NF; ++i) f[i] = i < nf ? q[i * stride + (size_t)k * 16] : 0.0;
  }
  __device__ void store(int k, double, const double* f) const {
#pragma unroll
    for (int i = 0; i < NF; ++i)
      if (i < nf) q[i * stride + (size_t)k * 16] = f[i];
  }
};

// one column of one batch; dpc points at dp3d(tl) level 0 of the column
template <class IO>
__device__ __forceinline__ void remap_column(const RemapArgs& A, const double* dpc, const IO& io, double* ps_out) {
  constexpr int NF = IO::NF;
  const int L = A.L;
  double S = 0.0;
  for (int k = 0; k < L; ++k) S = add(S, dpc[(size_t)k * 16]);
  const double ps = add(mul(A.hyai[0], A.ps0), S);
  if (ps_out) *ps_out = ps;

  // the window (Fortran level indices; m is the last old level pushed, -1 and 0 and L+1, L+2 are ghosts)
  double d3 = 0.0, d2 = 0.0, d1 = 0.0, d0 = 0.0;          // dx(m-3..m)
  double P0 = 0.0, P1 = 0.0, P2 = 0.0, P3 = 0.0;          // pio(m-2..m+1)
  double a2[NF], a1[NF], a0[NF], dmp[NF], i3[NF], i2[NF], M0[NF], M1[NF], M2[NF], M3[NF];
#pragma unroll
  for (int i = 0; i < NF; ++i) a2[i] = a1[i] = a0[i] = dmp[i] = i3[i] = i2[i] = M0[i] = M1[i] = M2[i] = M3[i] = 0.0;
  int m = -2;
  // push old level m+1 with thickness dxn, mixing ratios an and (for a real level) values fn
  auto push = [&](double dxn, const double* an, const double* fn, bool real) {
    ++m;
    d3 = d2; d2 = d1; d1 = d0; d0 = dxn;
    P0 = P1; P1 = P2; P2 = P3;
    P3 = real ? add(P2, dxn) : (m > 0 ? add(P2, 1.0) : 0.0);
    // r1..r3 at j = m-1
    const double r1 = dv(d1, add(add(d2, d1), d0));
    const double r2 = dv(add(mul(2.0, d2), d1), add(d0, d1));
    const double r3 = dv(add(d1, mul(2.0, d0)), add(d2, d1));
    // r4..r10 at j = m-2
    const double r4 = dv(d2, add(d2, d1));
    const double r5 = dv(1.0, add(add(add(d3, d2), d1), d0));
    const double r6 = dv(mul(mul(2.0, d1), d2), add(d2, d1));
    const double r7 = dv(add(d3, d2), add(mul(2.0, d2), d1));
    const double r8 = dv(add(d0, d1), add(mul(2.0, d1), d2));
    const double r9 = dv(mul(d2, add(d3, d2)), add(mul(2.0, d2), d1));
    const double r10 = dv(mul(d1, add(d1, d0)), add(d2, mul(2.0, d1)));
    const double g = mul(r6, sub(r7, r8));
#pragma unroll
    for (int i = 0; i < NF; ++i) {
      a2[i] = a1[i]; a1[i] = a0[i]; a0[i] = an[i];
      M0[i] = M1[i]; M1[i] = M2[i]; M2[i] = M3[i];
      M3[i] = real ? add(M2[i], fn[i]) : M2[i];
      // dma(m-1) from a(m-2..m)
      const double up = sub(a0[i], a1[i]), dn = sub(a1[i], a2[i]);
      const double da = mul(r1, add(mul(r2, up), mul(r3, dn)));
      double mn = fabs(da);
      const double b = mul(2.0, fabs(dn)), c = mul(2.0, fabs(up));
      if (b < mn) mn = b;
      if (c < mn) mn = c;
      double dma = mul(mn, copysign(1.0, da));
      if (mul(up, dn) <= 0.0) dma = 0.0;
      // ai(m-2) from a(m-2), a(m-1), dma(m-2), dma(m-1)
      const double ai = add(add(a2[i], mul(r4, dn)), mul(r5, add(sub(mul(g, dn), mul(r9, dma)), mul(r10, dmp[i]))));
      dmp[i] = dma;
      i3[i] = i2[i];
      i2[i] = ai;
    }
  };
  // push old level m+1 (push has this one call site): a real level 1..L, and the ghosts -1, 0 (levels 2, 1, read before
  // any store), from memory; the ghosts L+1, L+2 (levels L, L-1) from the window, never re-read
  auto advance = [&]() {
    const int nm = m + 1;
    double dxn, f[NF], an[NF];
    if (nm <= L) {
      const int lev = nm >= 1 ? nm : 1 - nm;
      dxn = dpc[(size_t)(lev - 1) * 16];
      io.load(lev - 1, dxn, f);
#pragma unroll
      for (int i = 0; i < NF; ++i) an[i] = dv(f[i], dxn);
    } else {
      dxn = nm == L + 1 ? d0 : d2;
#pragma unroll
      for (int i = 0; i < NF; ++i) an[i] = f[i] = nm == L + 1 ? a0[i] : a2[i];
    }
    push(dxn, an, f, nm >= 1 && nm <= L);
  };
  while (m < 2) advance();

  double pin = 0.0, massn1[NF];
#pragma unroll
  for (int i = 0; i < NF; ++i) massn1[i] = 0.0;
  int kid = 0;
  for (int k = 1; k <= L; ++k) {
    const double dp = add(mul(sub(A.hyai[k], A.hyai[k - 1]), A.ps0), mul(sub(A.hybi[k], A.hybi[k - 1]), ps));
    pin = k == L ? S : add(pin, dp);  // pin(k+1); pin(L+1) = pio(L+1)
    // kid(k) = min(c, L) with c = max(k-1, kid(k-1)) advanced while pio(c+1) <= pin(k+1): HOMME's search from kk = k
    int c = max(k - 1, kid);
    while (c <= L) {
      while (m < c && m < L + 2) advance();
      const int o = c + 1 - (m - 2);  // pio(c+1) in the window: 1, 2 or 3
      const double pc = o == 1 ? P1 : (o == 2 ? P2 : P3);
      if (!(pc <= pin)) break;
      ++c;
    }
    kid = max(min(c, L), 1);
    while (m - 2 < kid && m < L + 2) advance();
    // the window's cell j = m-2 is kid(k). A division by 2 or 4 is exact as a product by 0.5 or 0.25 (the same real
    // quotient, rounded once), so those are products; the divisions by 3 and 6 stay IEEE divisions.
    const double x2 = dv(sub(pin, mul(add(P0, P1), 0.5)), d2);
    const double x1 = -0.5;
    const double t1 = sub(x2, x1);
    const double t2 = sub(mul(x2, x2), mul(x1, x1));
    const double t3 = sub(mul(mul(x2, x2), x2), mul(mul(x1, x1), x1));
    double fk[NF];
#pragma unroll
    for (int i = 0; i < NF; ++i) {
      double al = i3[i], ar = i2[i];
      const double aj = a2[i];
      if (mul(sub(ar, aj), sub(aj, al)) <= 0.0) al = ar = aj;
      double w = sub(ar, al);
      double q6 = dv(mul(w, w), 6.0);
      if (mul(w, sub(aj, mul(add(al, ar), 0.5))) > q6) {
        al = sub(mul(3.0, aj), mul(2.0, ar));
        w = sub(ar, al);
        q6 = dv(mul(w, w), 6.0);
      }
      if (mul(w, sub(aj, mul(add(al, ar), 0.5))) < -q6) ar = sub(mul(3.0, aj), mul(2.0, al));
      const double c0 = sub(mul(1.5, aj), mul(add(al, ar), 0.25));
      const double c1 = sub(ar, al);
      const double c2 = add(mul(-6.0, aj), mul(3.0, add(al, ar)));
      const double integral = add(add(mul(c0, t1), mul(mul(c1, t2), 0.5)), dv(mul(c2, t3), 3.0));
      const double massn2 = add(M0[i], mul(integral, d2));
      fk[i] = sub(massn2, massn1[i]);
      massn1[i] = massn2;
    }
    io.store(k - 1, dp, fk);
  }
}

__global__ void __launch_bounds__(REMAP_WARPS * 32) remap_kernel(const RemapArgs A) {
  const int lane = threadIdx.x & 31;
  const unsigned long long nw = (unsigned long long)gridDim.x * REMAP_WARPS;
  for (unsigned long long w = (unsigned long long)blockIdx.x * REMAP_WARPS + (threadIdx.x >> 5); w < A.nitems; w += nw) {
    const unsigned long long grp = w / A.nbatch;
    const int b = (int)(w - grp * A.nbatch);
    const unsigned long long col = grp * 32 + lane;
    if (col >= (unsigned long long)A.ncols) continue;
    const size_t e = (size_t)A.nets + col / 16;
    const int p = (int)(col % 16);
    const double* dpc = A.dp3d + ((e * A.ntl + A.tl) * A.L) * 16 + p;
    if (b == 0) {
      StateIO io;
      io.T = A.T + ((e * A.ntl + A.tl) * A.L) * 16 + p;
      io.v = reinterpret_cast<double2*>(A.v) + ((e * A.ntl + A.tl) * A.L) * 16 + p;
      remap_column(A, dpc, io, A.ps + e * 16 + p);
    } else {
      const int iq0 = (b - 1) * REMAP_QB;
      TracerIO io;
      io.stride = (size_t)2 * A.L * 16;
      io.q = A.Qdp + (((e * A.qsize_d + iq0) * 2 + A.qtl) * A.L) * 16 + p;
      io.nf = min(REMAP_QB, A.qsize - iq0);
      remap_column(A, dpc, io, nullptr);
    }
  }
}

// dp3d(tl) = (hyai[k+1]-hyai[k])*ps0 + (hybi[k+1]-hybi[k])*ps, one thread per value of [nets, nete) x L x 16
__global__ void __launch_bounds__(REMAP_DP_THREADS) remap_dp_kernel(const RemapArgs A) {
  const unsigned long long n = (unsigned long long)A.ncols * A.L;
  for (unsigned long long i = (unsigned long long)blockIdx.x * REMAP_DP_THREADS + threadIdx.x; i < n;
       i += (unsigned long long)gridDim.x * REMAP_DP_THREADS) {
    const unsigned long long r = i / 16;
    const int p = (int)(i % 16);
    const size_t e = (size_t)A.nets + r / A.L;
    const int k = (int)(r % A.L);
    const double ps = A.ps[e * 16 + p];
    A.dp3d[((e * A.ntl + A.tl) * A.L + k) * 16 + p] =
        add(mul(sub(A.hyai[k + 1], A.hyai[k]), A.ps0), mul(sub(A.hybi[k + 1], A.hybi[k]), ps));
  }
}

}  // namespace

cudaError_t launch_vertical_remap(const KernelArgs& a, const double* hyai, double* ps, int nets, int nete, int tl,
                                  int qtl, int qsize, cudaStream_t s) {
  if (nete <= nets) return cudaSuccess;
  static LaunchCache cache, cache_dp;
  int per_sm = 1, per_sm_dp = 1;
  cudaError_t e = setup_launch(remap_kernel, REMAP_WARPS * 32, 0, cache, &per_sm);
  if (e == cudaSuccess) e = setup_launch(remap_dp_kernel, REMAP_DP_THREADS, 0, cache_dp, &per_sm_dp);
  if (e != cudaSuccess) return e;
  RemapArgs A;
  A.dp3d = a.dp3d;
  A.v = a.v;
  A.T = a.T;
  A.Qdp = const_cast<double*>(a.Qdp);  // the handle's own mirror; const in KernelArgs for the kernels that read it
  A.hyai = hyai;
  A.hybi = a.hybi;
  A.ps = ps;
  A.ps0 = a.ps0;
  A.L = a.nlev;
  A.ntl = a.ntl;
  A.qsize_d = a.qsize_d;
  A.nets = nets;
  A.ncols = (nete - nets) * 16;
  A.tl = tl;
  A.qtl = qtl;
  A.qsize = qsize;
  A.nbatch = 1 + (qsize + REMAP_QB - 1) / REMAP_QB;
  A.nitems = (unsigned long long)((A.ncols + 31) / 32) * A.nbatch;
  const unsigned long long wave = (unsigned long long)per_sm * sm_count();
  unsigned long long blocks = (A.nitems + REMAP_WARPS - 1) / REMAP_WARPS;
  if (blocks > wave) blocks = wave;
  remap_kernel<<<(unsigned)blocks, REMAP_WARPS * 32, 0, s>>>(A);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const unsigned long long n = (unsigned long long)A.ncols * A.L;
  const unsigned long long wave_dp = (unsigned long long)per_sm_dp * sm_count();
  blocks = (n + REMAP_DP_THREADS - 1) / REMAP_DP_THREADS;
  if (blocks > wave_dp) blocks = wave_dp;
  remap_dp_kernel<<<(unsigned)blocks, REMAP_DP_THREADS, 0, s>>>(A);
  return cudaGetLastError();
}

}  // namespace caar
