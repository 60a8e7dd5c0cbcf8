// caar_euler.cu — CAAR_MODE_STRICT of the tracer step that follows compute_and_apply_rhs (SURVEY §8f rank 4):
//
//     qtens[ie][iq][k] = Qdp[ie][iq][qn0][k] - dt * divergence_sphere(vstar[ie][k] * Qdp[ie][iq][qn0][k])
//
// for every tracer iq < qsize and level k — level_vectorized_ppscan/EulerStepFunctor.hpp:33-66
// (v_buf = vstar*qdp, q_buf = qdp, divergence_sphere_update(alpha = -dt, beta = 1),
// level_vectorized_ppscan/SphereOperators.hpp:362-403), with the reference's tested operator
// divergence_sphere (PO/sphere_operators.cpp:50-89) and the pointers_only array conventions:
// vstar [E][L][4][4][2] (like derived_vn0), qtens [E][qsize_d][L][4][4].
//
// The operations follow the reference's order without FMA contraction. Fast mode runs on levelop_kernel<OP_EULER>
// (caar_levelops.cu).
//
// Bound: HBM. Per element·level·tracer the kernel reads Qdp (128 B) and writes qtens (128 B); vstar (256 B per
// element·level) and the geometry are read once per element and reused for all tracers:
// B_alg = 256 + (256 + 1408/L)/qsize bytes per element·level·tracer.
//
// Work decomposition: levels are independent here (no vertical integral), so the unit of work is one level of one
// element = 4 threads (thread = GLL row, 4 points each, as in the fused CAAR kernel: derivative along jgp
// thread-local, along igp through shuffles from the other lanes of the level). Persistent CTAs of 256 threads walk the
// flat (element, level) index space in groups of 64 rows with a grid-stride loop, one tracer per trip.
//
// The output of tracer iq of element e is the level slice (e * qsize_d + iq) * out_stride + out_off of `out`
// ([slice][L][16]): (qtens, 1, 0) for caar_euler_step, (Qdp, 2, np1) for a stage of caar_advect_tracers, which may
// read and write the same Qdp level (qn0 == np1). That in-place form is safe as the kernel stands: a thread loads only
// its own GLL row of each tracer (ld4 of qbase below), takes its neighbours' values through shuffles of registers the
// neighbours already loaded, and stores that same row afterwards; no thread reads a row another thread stores (the
// clamped tail rows only feed dead lanes). Qdp is read with plain loads, never __ldg / ld.global.nc, because the
// launch may write it.
#include <cstdlib>

#include "caar_device.cuh"

namespace caar {
namespace {

constexpr unsigned FULL = 0xffffffffu;

struct EulerArgs {
  const double* Dinv;
  const double* metdet;
  const double* rmetdet;
  const double* Qdp;    // [E][qsize_d][2][L][16]
  const double* vstar;  // [E][L][16][2]
  double* out;          // tracer 0 of element 0 of the output: qtens, or Qdp + np1 * lf
  size_t out_stride;    // doubles from one tracer to the next in `out`: lf (qtens) or 2 lf (Qdp)
  int nlev, qsize_d, nets, nelem_run, qn0, qsize;
  double dt, rrearth;
  double dvv[16];
};

__device__ __forceinline__ void ld4(const double* p, double (&x)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2);
  x[0] = a.x; x[1] = a.y; x[2] = b.x; x[3] = b.y;
}
__device__ __forceinline__ void st4(double* p, const double (&x)[4]) {
  *reinterpret_cast<double2*>(p) = make_double2(x[0], x[1]);
  *reinterpret_cast<double2*>(p + 2) = make_double2(x[2], x[3]);
}

// one tracer of one level-row: q -> qtens, in the reference's operation order without contraction
// (PO/sphere_operators.cpp:62-88)
__device__ __forceinline__ void tracer_row(const EulerArgs& A, const double (&q)[4], const double (&u)[4],
                                           const double (&v)[4], const double (&di)[4][4], const double (&met)[4],
                                           const double (&rmet)[4], int lane, int r, double (&out)[4]) {
  double g0[4], g1[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double v0 = __dmul_rn(u[j], q[j]), v1 = __dmul_rn(v[j], q[j]);
    g0[j] = __dmul_rn(met[j], __dadd_rn(__dmul_rn(di[j][0], v0), __dmul_rn(di[j][1], v1)));
    g1[j] = __dmul_rn(met[j], __dadd_rn(__dmul_rn(di[j][2], v0), __dmul_rn(di[j][3], v1)));
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    double dudx = 0.0, dvdy = 0.0;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const double gm = __shfl_sync(FULL, g0[j], (lane & ~3) | m);
      dudx = __dadd_rn(dudx, __dmul_rn(A.dvv[m * 4 + r], gm));
      dvdy = __dadd_rn(dvdy, __dmul_rn(A.dvv[m * 4 + j], g1[m]));
    }
    const double div = __dmul_rn(__dmul_rn(__dadd_rn(dudx, dvdy), rmet[j]), A.rrearth);
    out[j] = __dadd_rn(__dmul_rn(q[j], 1.0), __dmul_rn(-A.dt, div));
  }
}

__global__ void __launch_bounds__(256, 2) euler_step_kernel(const __grid_constant__ EulerArgs A) {
  const int t = threadIdx.x, lane = t & 31, r = t & 3;
  const int L = A.nlev;
  const size_t lf = (size_t)L * PTS;
  // persistent CTAs: grid-stride loop over groups of 64 (element, level) rows. The tail group computes on clamped
  // indices (the shuffles need every lane) and skips the stores.
  const long long n_rows = (long long)A.nelem_run * L;
  const long long n_groups = (n_rows + 63) / 64;
  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    long long gk = grp * 64 + (t >> 2);
    const bool live = gk < n_rows;
    if (!live) gk = n_rows - 1;
    const size_t e = (size_t)A.nets + (size_t)(gk / L);
    const int k = (int)(gk % L);
    const size_t off = (size_t)k * PTS + r * 4;
    // this row's inputs: vstar (u,v), Dinv [jgp][2][2], metdet, rmetdet
    double u[4], v[4], di[4][4], met[4], rmet[4];
    {
      const double* p = A.vstar + (e * lf + off) * 2;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double2 a = __ldg(reinterpret_cast<const double2*>(p + 2 * j));
        u[j] = a.x;
        v[j] = a.y;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) ld4(A.Dinv + e * 64 + (r * 4 + j) * 4, di[j]);
    ld4(A.metdet + e * 16 + r * 4, met);
    ld4(A.rmetdet + e * 16 + r * 4, rmet);
    const double* qbase = A.Qdp + (e * A.qsize_d * 2 + A.qn0) * lf + off;  // + iq * 2 * lf
    double* obase = A.out + e * A.qsize_d * A.out_stride + off;            // + iq * out_stride
    // one tracer per trip: the reference-order evaluation keeps many values live, and two per trip spilled at the
    // 128 registers of two resident CTAs per SM
    for (int iq = 0; iq < A.qsize; ++iq) {
      double qa[4], oa[4];
      ld4(qbase + (size_t)iq * 2 * lf, qa);
      tracer_row(A, qa, u, v, di, met, rmet, lane, r, oa);
      if (live) st4(obase + (size_t)iq * A.out_stride, oa);
    }
  }
}

}  // namespace

cudaError_t launch_euler_step(const KernelArgs& a, const double* vstar, double* out, int out_stride, int out_off,
                              int nets, int nete, int qn0, int qsize, double dt, cudaStream_t s) {
  if (nete <= nets || qsize <= 0) return cudaSuccess;
  const size_t lf = (size_t)a.nlev * PTS;
  EulerArgs e;
  e.Dinv = a.Dinv; e.metdet = a.metdet; e.rmetdet = a.rmetdet; e.Qdp = a.Qdp; e.vstar = vstar;
  e.out = out + (size_t)out_off * lf; e.out_stride = (size_t)out_stride * lf;
  e.nlev = a.nlev; e.qsize_d = a.qsize_d; e.nets = nets; e.nelem_run = nete - nets; e.qn0 = qn0; e.qsize = qsize;
  e.dt = dt; e.rrearth = a.rrearth;
  for (int i = 0; i < 16; ++i) e.dvv[i] = a.dvv[i];
  const long long rows = (long long)(nete - nets) * a.nlev;
  const long long groups = (rows + 63) / 64;
  const long long cap = (long long)sm_count() * 3 * 2;  // persistent CTAs: 2 waves of 3 per SM
  const unsigned blocks = (unsigned)(groups > cap ? cap : groups);
  euler_step_kernel<<<blocks, 256, 0, s>>>(e);
  return cudaGetLastError();
}

}  // namespace caar
