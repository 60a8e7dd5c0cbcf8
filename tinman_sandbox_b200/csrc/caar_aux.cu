// caar_aux.cu — the two small kernels beside the hot path:
//   * norms: sum of squares of v, T, dp3d at one time level per element, then over elements
//     (what print_results_2norm reduces, PO/compute_and_apply_rhs.cpp:372-399);
//   * saxpby: x = a*x + b*y, the reference's bandwidth yardstick (saxpby_test/cxx/common.cpp:3-15);
//   * the RK5 step's combination of two time levels (caar_run_rk5) and the tracer SSP step's time average of Qdp
//     (caar_advect_tracers), on one grid-stride skeleton.
#include "caar_device.cuh"

namespace caar {

// number of SMs of the current device (cached per device ordinal): grid caps are multiples of it
int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!cached[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

namespace {

__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double s = 0;
  if (w == 0) {
    s = (lane < (int)(blockDim.x >> 5)) ? red[lane] : 0.0;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  }
  return s;  // valid in warp 0
}

// one CTA per element: partial[e] = { sum v^2, sum T^2, sum dp^2 } at time level tl
__global__ void __launch_bounds__(256) norms_partial_kernel(const KernelArgs A, int tl, int nets, double* partial) {
  __shared__ double red[8];
  const size_t e = (size_t)(nets + blockIdx.x);
  const int lf = A.nlev * PTS;
  const double2* v = reinterpret_cast<const double2*>(A.v + (e * A.ntl + tl) * (size_t)lf * 2);
  const double* T = A.T + (e * A.ntl + tl) * (size_t)lf;
  const double* dp = A.dp3d + (e * A.ntl + tl) * (size_t)lf;
  double sv = 0, sT = 0, sd = 0;
  for (int n = threadIdx.x; n < lf; n += blockDim.x) {
    const double2 a = v[n];
    sv = fma(a.x, a.x, fma(a.y, a.y, sv));
    const double b = T[n], c = dp[n];
    sT = fma(b, b, sT);
    sd = fma(c, c, sd);
  }
  sv = block_sum(sv, red);
  sT = block_sum(sT, red);
  sd = block_sum(sd, red);
  if (threadIdx.x == 0) {
    partial[e * 3 + 0] = sv;
    partial[e * 3 + 1] = sT;
    partial[e * 3 + 2] = sd;
  }
}

// one CTA: fixed-order reduction of the per-element partials over [nets, nete)
__global__ void __launch_bounds__(1024) norms_final_kernel(const double* partial, int nets, int nete, double* out3) {
  __shared__ double red[32];
  double s[3] = {0, 0, 0};
  for (int e = nets + threadIdx.x; e < nete; e += blockDim.x) {
    s[0] += partial[(size_t)e * 3 + 0];
    s[1] += partial[(size_t)e * 3 + 1];
    s[2] += partial[(size_t)e * 3 + 2];
  }
  for (int c = 0; c < 3; ++c) {
    const double r = block_sum(s[c], red);
    if (threadIdx.x == 0) out3[c] = r;
  }
}

__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v, unsigned long long* red) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  unsigned long long s = 0;
  if (w == 0) {
    s = (lane < (int)(blockDim.x >> 5)) ? red[lane] : 0ull;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  }
  return s;  // valid in warp 0
}

// Checksums of the seven arrays compute_and_apply_rhs writes, one CTA per element:
// partial[e][f] = { sum, sum of squares } for f = dp3d(tl), v(tl), T(tl), eta_dot_dpdn, omega_p, phi, vn0,
// partial[e][7] = { KE, IE }: sum of spheremp*0.5*(u^2+v^2)*dp3d and spheremp*cp*T*dp3d at time level tl (the
// integrands of the reference's energy diagnostics, F/routine_extracted.F90:396-410), bits[e][f] = sum of the IEEE
// bit patterns mod 2^64 (exact and order-independent: equal data <=> equal sums, up to 2^-64 collisions).
__global__ void __launch_bounds__(256) checksums_partial_kernel(const KernelArgs A, int tl, int nets, double cp,
                                                                 double* partial /*[nelem][8][2]*/,
                                                                 unsigned long long* bits /*[nelem][7]*/) {
  __shared__ double red[8];
  __shared__ unsigned long long redu[8];
  const size_t e = (size_t)(nets + blockIdx.x);
  const int lf = A.nlev * PTS;
  const double* f[7] = {A.dp3d + (e * A.ntl + tl) * (size_t)lf, A.v + (e * A.ntl + tl) * (size_t)lf * 2,
                        A.T + (e * A.ntl + tl) * (size_t)lf,    A.eta_dot_dpdn + e * (size_t)(lf + PTS),
                        A.omega_p + e * (size_t)lf,             A.phi + e * (size_t)lf,
                        A.vn0 + e * (size_t)lf * 2};
  const int n[7] = {lf, 2 * lf, lf, lf + PTS, lf, lf, 2 * lf};
#pragma unroll 1
  for (int a = 0; a < 7; ++a) {
    double s = 0, q = 0;
    unsigned long long b = 0;
    for (int i = threadIdx.x; i < n[a]; i += blockDim.x) {
      const double x = f[a][i];
      s += x;
      q = fma(x, x, q);
      b += (unsigned long long)__double_as_longlong(x);
    }
    s = block_sum(s, red);
    q = block_sum(q, red);
    b = block_sum_u64(b, redu);
    if (threadIdx.x == 0) {
      partial[(e * 8 + a) * 2 + 0] = s;
      partial[(e * 8 + a) * 2 + 1] = q;
      bits[e * 7 + a] = b;
    }
  }
  double ke = 0, ie = 0;
  const double2* v = reinterpret_cast<const double2*>(f[1]);
  for (int i = threadIdx.x; i < lf; i += blockDim.x) {
    const double w = A.spheremp[e * PTS + (i & 15)] * f[0][i];
    const double2 u = v[i];
    ke = fma(w * 0.5, fma(u.x, u.x, u.y * u.y), ke);
    ie = fma(w * cp, f[2][i], ie);
  }
  ke = block_sum(ke, red);
  ie = block_sum(ie, red);
  if (threadIdx.x == 0) {
    partial[(e * 8 + 7) * 2 + 0] = ke;
    partial[(e * 8 + 7) * 2 + 1] = ie;
  }
}

// one CTA: fixed-order reduction over [nets, nete) of the 16 doubles and 7 bit sums per element
__global__ void __launch_bounds__(1024) checksums_final_kernel(const double* partial, const unsigned long long* bits,
                                                                int nets, int nete, double* out16,
                                                                unsigned long long* out7) {
  __shared__ double red[32];
  __shared__ unsigned long long redu[32];
#pragma unroll 1
  for (int c = 0; c < 16; ++c) {
    double s = 0;
    for (int e = nets + threadIdx.x; e < nete; e += blockDim.x) s += partial[(size_t)e * 16 + c];
    const double r = block_sum(s, red);
    if (threadIdx.x == 0) out16[c] = r;
  }
#pragma unroll 1
  for (int c = 0; c < 7; ++c) {
    unsigned long long s = 0;
    for (int e = nets + threadIdx.x; e < nete; e += blockDim.x) s += bits[(size_t)e * 7 + c];
    const unsigned long long r = block_sum_u64(s, redu);
    if (threadIdx.x == 0) out7[c] = r;
  }
}

// grid-stride, 2 doubles per thread per trip (LDG.128/STG.128), x read-modify-write, y read-only
__global__ void __launch_bounds__(512) saxpby_kernel(double a, double b, double* __restrict__ x,
                                                      const double* __restrict__ y, size_t n2, size_t n) {
  double2* x2 = reinterpret_cast<double2*>(x);
  const double2* y2 = reinterpret_cast<const double2*>(y);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n2; i += 4 * stride) {
    double2 xv[4], yv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { xv[u] = x2[i + u * stride]; yv[u] = __ldg(y2 + i + u * stride); }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      xv[u].x = a * xv[u].x + b * yv[u].x;
      xv[u].y = a * xv[u].y + b * yv[u].y;
      x2[i + u * stride] = xv[u];
    }
  }
  for (; i < n2; i += stride) {
    double2 xv = x2[i];
    const double2 yv = __ldg(y2 + i);
    xv.x = a * xv.x + b * yv.x;
    xv.y = a * xv.y + b * yv.y;
    x2[i] = xv;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && (n & 1)) x[n - 1] = a * x[n - 1] + b * y[n - 1];
}

// pointers that are 8- but not 16-byte aligned (a sub-array offset): plain 64-bit accesses
__global__ void __launch_bounds__(512) saxpby_scalar_kernel(double a, double b, double* __restrict__ x,
                                                             const double* __restrict__ y, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) x[i] = a * x[i] + b * __ldg(y + i);
}

// RK5 step (caar_run_rk5), between stages 4 and 5: X(nm1) = (5*X(nm1) - X(n0))/4 for X = v, T, dp3d on elements
// [nets, nete). Per element the combined rows are [0,16L) of v, [16L,24L) of T and [24L,32L) of dp3d in double2
// units; each time-level slice is a contiguous block of 8L (T, dp3d) or 16L (v) double2 starting on a 128 B boundary.
// Rounded mul, sub, mul, never contracted: scaling by 0.25 is exact, so this is Fortran's (5*a - b)/4 bit for bit
// in both modes. nm1 != n0 (caar_run_rk5 checks it), so the n0 block is read-only here.
struct Rk5Combine {
  double *v, *T, *dp;
  unsigned per, lf2;  // double2 rows per element (32L) and per time-level slice of T / dp3d (8L)
  int ntl, nets, nm1, n0;
  static constexpr int ROWS = 4;  // rows of 16 B per thread and trip in flight

  // row i of the combination at time level nm1; *dn0 = distance in double2 to the same row at n0
  __device__ __forceinline__ double2* row(size_t i, ptrdiff_t* dn0) const {
    const size_t e = (size_t)nets + i / per;
    unsigned r = (unsigned)(i % per);
    double* f = v;
    unsigned slice = 2 * lf2;
    if (r >= slice) {
      r -= slice;
      slice = lf2;
      f = r < slice ? T : dp;
      if (r >= slice) r -= slice;
    }
    *dn0 = (ptrdiff_t)(n0 - nm1) * slice;
    return reinterpret_cast<double2*>(f) + (e * ntl + nm1) * slice + r;
  }
  // a = the row at nm1, b = the same row at n0
  static __device__ __forceinline__ double mix(double a, double b) { return __dmul_rn(__dsub_rn(__dmul_rn(5.0, a), b), 0.25); }
};

// Tracer SSP step (caar_advect_tracers), after its third stage: Qdp(np1) = (Qdp(n0) + 2*Qdp(np1))/3 for tracers
// iq < qsize of elements [nets, nete). Per element the rows are qsize blocks of 8L double2, one per tracer, each the
// tracer's np1 slice of Qdp [E][qsize_d][2][L][16] (128 B aligned). Rounded as Fortran's (a + 2*b)/3: 2*b is exact, then
// one rounded add and one rounded division, never contracted and never a multiplication by 1/3, in both modes.
// np1 != n0, so the n0 slices are read-only here.
struct QdpAverage {
  double* Qdp;
  unsigned per, lf2;  // double2 rows per element (qsize * 8L) and per tracer slice (8L)
  int qsize_d, nets, np1, n0;
  // rows per thread and trip: with 4, the registers live across the division's slow-path call exceed the 64 of two
  // resident CTAs of 512 and spill
  static constexpr int ROWS = 2;

  // row i of the average at np1; *dn0 = distance in double2 to the same row at n0
  __device__ __forceinline__ double2* row(size_t i, ptrdiff_t* dn0) const {
    const size_t e = (size_t)nets + i / per;
    const unsigned r = (unsigned)(i % per), iq = r / lf2;
    *dn0 = (ptrdiff_t)(n0 - np1) * lf2;
    return reinterpret_cast<double2*>(Qdp) + ((e * qsize_d + iq) * 2 + np1) * lf2 + (r - iq * lf2);
  }
  // a = the row at np1 (stage 3's result), b = the same row at n0
  static __device__ __forceinline__ double mix(double a, double b) { return __ddiv_rn(__dadd_rn(b, __dmul_rn(2.0, a)), 3.0); }
};

template <class C>
__device__ __forceinline__ double2 mix2(double2 a, double2 b) { return make_double2(C::mix(a.x, b.x), C::mix(a.y, b.y)); }

// x = C::mix(x, y) over the rows C::row maps out, y the row *dn0 away (read-only in the launch); grid-stride,
// C::ROWS rows of 16 B per thread per trip in flight
template <class C>
__global__ void __launch_bounds__(512, 2) combine_kernel(const C c, size_t n) {
  constexpr int R = C::ROWS;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + (R - 1) * stride < n; i += R * stride) {
    double2* p[R];
    double2 a[R], b[R];
#pragma unroll
    for (int u = 0; u < R; ++u) {
      ptrdiff_t d;
      p[u] = c.row(i + u * stride, &d);
      a[u] = *p[u];
      b[u] = __ldg(p[u] + d);
    }
#pragma unroll
    for (int u = 0; u < R; ++u) *p[u] = mix2<C>(a[u], b[u]);
  }
  for (; i < n; i += stride) {
    ptrdiff_t d;
    double2* p = c.row(i, &d);
    *p = mix2<C>(*p, __ldg(p + d));
  }
}

// blocks of the combination kernels: 4 rows per thread, at most two resident CTAs of 512 per SM
unsigned combine_blocks(size_t n) {
  size_t blocks = (n + 512 * 4 - 1) / (512 * 4);
  if (blocks > (size_t)sm_count() * 2) blocks = (size_t)sm_count() * 2;
  return (unsigned)blocks;
}

// ---- host-layout conversion for the Fortran (F90 flat pointer) boundary --------------------------------------
// The reference's C++ arrays are row-major [igp][jgp]([comp]) with C [igp][jgp] == Fortran (i,j) index for index
// (PO/test_macros.hpp), i.e. the Fortran arrays of F/element_state_mod.F90:17-23 / F/element_mod.F90:69-121, whose
// memory order is first-index-fastest, hold every 4x4 block transposed, the (u,v) component as a slower
// dimension (v(np,np,2,nlev,tl)) and the 2x2 tensor indices slowest (D(np,np,2,2)) — the order HOMMEXX reads its
// F90 pointers in (LV/Elements.cpp:48-99,164-292). Per block of B doubles (16 scalar, 32 vector, 64 tensor):
//   scalar  cxx[i*4+j]               <-> f90[j*4+i]
//   vector  cxx[(i*4+j)*2+c]         <-> f90[c*16+j*4+i]
//   tensor  cxx[((i*4+j)*2+a)*2+b]   <-> f90[(b*2+a)*16+j*4+i]
// Tracers: cxx blocks [iq][qni][lev] <-> f90 blocks [qni][iq][lev] (Qdp(np,np,nlev,qsize_d,2)).
__device__ __forceinline__ int f90_index(int kind, int q) {
  if (kind == 0) return (q & 3) * 4 + (q >> 2);
  if (kind == 1) return (q & 1) * 16 + ((q >> 1) & 3) * 4 + (q >> 3);
  return ((q & 1) * 2 + ((q >> 1) & 1)) * 16 + ((q >> 2) & 3) * 4 + (q >> 4);
}

// cxx and f90 point at block 0 of the same chunk; blk0 = index of that block in the whole field (tracer remap)
__global__ void __launch_bounds__(256) relayout_kernel(double* __restrict__ cxx, double* __restrict__ f90, size_t nblocks,
                                                        int kind, int to_cxx, int q_dim, int nlev, size_t blk0) {
  const int B = 16 << kind;
  const size_t n = nblocks * B;
  for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < n; g += (size_t)gridDim.x * blockDim.x) {
    const size_t blk = g >> (4 + kind);
    const int q = (int)(g & (B - 1));
    size_t fblk = blk;
    if (q_dim > 1) {  // tracer block order: cxx [e][iq][qni][lev] -> f90 [e][qni][iq][lev]
      const size_t gb = blk0 + blk;
      const size_t lev = gb % nlev, qni = (gb / nlev) % 2, iq = (gb / nlev / 2) % q_dim, e = gb / nlev / 2 / q_dim;
      fblk = ((e * 2 + qni) * q_dim + iq) * nlev + lev - blk0;  // relative to the same chunk origin (chunks are whole elements)
    }
    double* c = cxx + g;
    double* f = f90 + fblk * B + f90_index(kind, q);
    if (to_cxx) *c = *f; else *f = *c;
  }
}

__global__ void __launch_bounds__(256) reciprocal_kernel(double* __restrict__ out, const double* __restrict__ in, size_t n) {
  for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < n; g += (size_t)gridDim.x * blockDim.x)
    out[g] = __ddiv_rn(1.0, in[g]);
}

}  // namespace

cudaError_t launch_relayout(double* cxx, double* f90, size_t nblocks, int kind, bool to_cxx, int q_dim, int nlev,
                            size_t blk0, cudaStream_t s) {
  if (nblocks == 0) return cudaSuccess;
  const size_t n = nblocks * (16u << kind);
  size_t blocks = (n + 255) / 256;
  if (blocks > (size_t)sm_count() * 32) blocks = (size_t)sm_count() * 32;
  relayout_kernel<<<(unsigned)blocks, 256, 0, s>>>(cxx, f90, nblocks, kind, to_cxx ? 1 : 0, q_dim, nlev, blk0);
  return cudaGetLastError();
}

cudaError_t launch_reciprocal(double* out, const double* in, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  size_t blocks = (n + 255) / 256;
  if (blocks > (size_t)sm_count() * 32) blocks = (size_t)sm_count() * 32;
  reciprocal_kernel<<<(unsigned)blocks, 256, 0, s>>>(out, in, n);
  return cudaGetLastError();
}

cudaError_t launch_norms(const KernelArgs& a, int tl, int nets, int nete, double* partial, double* out3,
                         cudaStream_t s) {
  if (nete > nets) norms_partial_kernel<<<nete - nets, 256, 0, s>>>(a, tl, nets, partial);
  norms_final_kernel<<<1, 1024, 0, s>>>(partial, nets, nete, out3);
  return cudaGetLastError();
}

cudaError_t launch_saxpby(double a, double b, double* x, const double* y, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const size_t n2 = n / 2;
  size_t blocks = (n2 + 512 * 4 - 1) / (512 * 4);
  if (blocks < 1) blocks = 1;
  const size_t cap = (size_t)sm_count() * 4 * 8;  // a few waves of 4 resident CTAs per SM
  if (blocks > cap) blocks = cap;
  if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) != 0)  // not double2-aligned
    saxpby_scalar_kernel<<<(unsigned)blocks, 512, 0, s>>>(a, b, x, y, n);
  else
    saxpby_kernel<<<(unsigned)blocks, 512, 0, s>>>(a, b, x, y, n2, n);
  return cudaGetLastError();
}

cudaError_t launch_rk5_combine(const KernelArgs& a, int nets, int nete, int nm1, int n0, cudaStream_t s) {
  if (nete <= nets) return cudaSuccess;
  const size_t n = (size_t)(nete - nets) * a.nlev * 32;  // double2 rows
  combine_kernel<<<combine_blocks(n), 512, 0, s>>>(Rk5Combine{a.v, a.T, a.dp3d, 32u * a.nlev, 8u * a.nlev, a.ntl, nets, nm1, n0}, n);
  return cudaGetLastError();
}

cudaError_t launch_qdp_avg(const KernelArgs& a, int nets, int nete, int qsize, int n0, int np1, cudaStream_t s) {
  if (nete <= nets || qsize <= 0) return cudaSuccess;
  const size_t n = (size_t)(nete - nets) * qsize * a.nlev * 8;  // double2 rows
  // the kernel writes Qdp; the mirror is const only for the operators that read it
  const QdpAverage c{const_cast<double*>(a.Qdp), (unsigned)qsize * 8u * a.nlev, 8u * a.nlev, a.qsize_d, nets, np1, n0};
  combine_kernel<<<combine_blocks(n), 512, 0, s>>>(c, n);
  return cudaGetLastError();
}

cudaError_t launch_checksums(const KernelArgs& a, int tl, int nets, int nete, double cp, double* partial,
                             unsigned long long* bits, double* out16, unsigned long long* out7, cudaStream_t s) {
  if (nete > nets) checksums_partial_kernel<<<nete - nets, 256, 0, s>>>(a, tl, nets, cp, partial, bits);
  checksums_final_kernel<<<1, 1024, 0, s>>>(partial, bits, nets, nete, out16, out7);
  return cudaGetLastError();
}

}  // namespace caar
