// caar_device.cuh — types shared by the CAAR kernels and the C-ABI layer (device layout == host layout).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

#include "caar_b200.h"

namespace caar {

constexpr int NP = 4;
constexpr int PTS = 16;

// Everything a kernel needs, passed by value (lives in the constant bank of the launch).
struct KernelArgs {
  // device pointers, layout of struct Arrays (PO/data_structures.cpp:14-31)
  const double* D;
  const double* Dinv;
  const double* fcor;
  const double* spheremp;
  const double* metdet;
  const double* rmetdet;
  double* dp3d;
  double* v;
  double* T;
  const double* phis;
  const double* Qdp;
  double* eta_dot_dpdn;
  double* omega_p;
  double* phi;
  const double* pecnd;
  double* vn0;
  // dims
  int nelem, nlev, qsize_d, ntl;
  // Control (element range is LOCAL to this handle)
  int nets, nete, n0, np1, nm1, qn0;
  double dt2;
  // Constants
  double rrearth, eta_ave_w, Rwv, Rgas, kappa;
  // HVCoord: only hyai[0]*ps0 enters the path (PO/compute_and_apply_rhs.cpp:82)
  double hyai0, ps0;
  // Derivative, row-major Dvv[i][j]
  double dvv[16];
  // host pointer to the handle's TMA descriptors (TmaMaps), or null; only the launcher reads it
  const void* tma;
  // vertical coordinate: rsplit > 0 vertically Lagrangian (the reference's C++ path), rsplit == 0 Eulerian
  // (F/routine_extracted.F90:227-262) with hybi[nlev+1] in device memory
  int rsplit;
  const double* hybi;
  // L2 prefetch distance in elements (0 = off): CTA e prefetches the early inputs of element e + pf_dist
  int pf_dist;
  // the handle's tile scheduler pair of the thread-per-level laplacians (device [2], zero between launches)
  unsigned* lapflat_sched;
};

// TMA tensor maps over the level-field arrays viewed as 3-D [slice][rows of 128 B][16 doubles] (slice = element x
// time level / tracer, rows = levels), box = one CTA's slab of one slice, SWIZZLE_128B (conflict-free shared-memory
// tiles). Built once per handle.
struct alignas(64) TmaMaps {
  CUtensorMap dp3d, T, v, vn0, pecnd, omega_p, phi, Qdp;
};
// returns 0 on success; on failure writes a message
int build_tma_maps(TmaMaps* out, const KernelArgs& a, char* err, size_t errlen);

// launchers (defined in the .cu files); return cudaError_t of the launch
cudaError_t launch_strict(const KernelArgs& a, cudaStream_t s);
cudaError_t launch_fused(const KernelArgs& a, cudaStream_t s);
bool fused_supports(int nlev);
bool fused_supports_eulerian(int nlev);  // rsplit == 0 on the fused path
int fused_instance_levels(int nlev);     // compiled level count that serves nlev (>= nlev), 0 = none
int fused_instance_cluster(int nlev);    // CTAs per element of that instance
cudaError_t launch_fused_more(const KernelArgs& a, cudaStream_t s);  // level counts other than 72 / 128
size_t strict_smem_bytes(int nlev);

cudaError_t launch_norms(const KernelArgs& a, int tl, int nets, int nete, double* partial /*[nelem][3]*/,
                         double* out3, cudaStream_t s);
// host-layout conversion (Fortran boundary): kind 0 = 4x4 scalar blocks, 1 = (u,v) level blocks, 2 = 2x2 tensors
cudaError_t launch_relayout(double* cxx, double* f90, size_t nblocks, int kind, bool to_cxx, int q_dim, int nlev,
                            size_t blk0, cudaStream_t s);
cudaError_t launch_reciprocal(double* out, const double* in, size_t n, cudaStream_t s);
// tracer step after CAAR (caar_euler.cu): Qdp(qn0) - dt*divergence_sphere(vstar*Qdp(qn0)) into the level slice
// (e * qsize_d + iq) * out_stride + out_off of out [slice][L][16]: (qtens, 1, 0), or (Qdp, 2, np1) in place
cudaError_t launch_euler_step(const KernelArgs& a, const double* vstar, double* out, int out_stride, int out_off,
                              int nets, int nete, int qn0, int qsize, double dt, bool strict, cudaStream_t s);
// level-local operators on the TMA-pipelined skeleton (caar_levelops.cu): op 0 tracer step (output slices as in
// launch_euler_step), 1 divergence_sphere_wk, 2 laplace_simple, 3 laplace_tensor
cudaError_t launch_levelop(int op, const KernelArgs& k, const double* in, const double* item, double* out,
                           const double* tensorvisc, int nets, int nete, int qn0, int qsize, double dt, int out_stride,
                           int out_off, bool strict, cudaStream_t s);
cudaError_t launch_saxpby(double a, double b, double* x, const double* y, size_t n, cudaStream_t s);
// RK5 step (caar_aux.cu): v, T, dp3d at nm1 = (5*X(nm1) - X(n0))/4 on [nets,nete), one launch; nm1 != n0
cudaError_t launch_rk5_combine(const KernelArgs& a, int nets, int nete, int nm1, int n0, cudaStream_t s);
// tracer SSP step (caar_aux.cu): Qdp(np1) = (Qdp(n0) + 2*Qdp(np1))/3 for tracers < qsize on [nets,nete), one launch
cudaError_t launch_qdp_avg(const KernelArgs& a, int nets, int nete, int qsize, int n0, int np1, cudaStream_t s);
// checksums of the seven mutated arrays + energy norms (caar_aux.cu); partial [nelem][8][2], bits [nelem][7]
cudaError_t launch_checksums(const KernelArgs& a, int tl, int nets, int nete, double cp, double* partial,
                             unsigned long long* bits, double* out16, unsigned long long* out7, cudaStream_t s);
int sm_count();  // SMs of the current device

}  // namespace caar
