// caar_device.cuh — types shared by the CAAR kernels and the C-ABI layer (device layout == host layout).
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>
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
// The one tensor-map format of the fused kernel and the level operators: *m over the doubles at `base` as
// [slices][rows of 128 B][16 doubles], box = box_rows rows of one slice, SWIZZLE_128B, 256 B L2 promotion. A box that
// sticks out of its slice is zero-filled on load and clipped on store. Returns 0 on success; on failure writes a
// message naming the map `name` into err (errlen may be 0).
int encode_tma_map(CUtensorMap* m, const void* base, cuuint64_t slices, cuuint64_t rows, cuuint32_t box_rows,
                   const char* name, char* err, size_t errlen);

// Launch set-up of one kernel on the current device: its dynamic shared-memory limit becomes `smem`, it asks for the
// largest shared-memory carveout (so that several CTAs can be resident per SM), and *per_sm (>= 1) is how many CTAs of
// `threads` threads and `smem` bytes an SM holds. Function attributes are per (kernel, device), so this is done once per
// device and `smem`, remembered in `cache`: one static per kernel, owned by its launcher (a static inside this template
// would be shared by all kernels of one signature). Device ordinals >= 64 are set up again on every call.
struct LaunchCache {
  size_t smem[64];
  int per_sm[64];
};
template <typename Kernel>
cudaError_t setup_launch(Kernel* kernel, int threads, size_t smem, LaunchCache& cache, int* per_sm) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const bool cached = dev >= 0 && dev < 64;
  if (cached && cache.per_sm[dev] > 0 && cache.smem[dev] == smem) {
    *per_sm = cache.per_sm[dev];
    return cudaSuccess;
  }
  int n = 0;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem);
  if (e != cudaSuccess) return e;
  *per_sm = n < 1 ? 1 : n;
  if (cached) {
    cache.smem[dev] = smem;
    cache.per_sm[dev] = *per_sm;
  }
  return cudaSuccess;
}

// launchers (defined in the .cu files); return cudaError_t of the launch
cudaError_t launch_strict(const KernelArgs& a, cudaStream_t s);
cudaError_t launch_fused(const KernelArgs& a, cudaStream_t s);
bool fused_supports(int nlev);           // both vertical coordinates
int fused_instance_levels(int nlev);     // compiled level count that serves nlev (>= nlev), 0 = none
int fused_instance_cluster(int nlev);    // CTAs per element of that instance
cudaError_t launch_fused_more(const KernelArgs& a, cudaStream_t s);  // level counts other than 72 / 128
size_t strict_smem_bytes(int nlev);
bool strict_supports(int nlev);  // the strict kernel's shared memory fits

cudaError_t launch_norms(const KernelArgs& a, int tl, int nets, int nete, double* partial /*[nelem][3]*/,
                         double* out3, cudaStream_t s);
// host-layout conversion (Fortran boundary): kind 0 = 4x4 scalar blocks, 1 = (u,v) level blocks, 2 = 2x2 tensors
cudaError_t launch_relayout(double* cxx, double* f90, size_t nblocks, int kind, bool to_cxx, int q_dim, int nlev,
                            size_t blk0, cudaStream_t s);
cudaError_t launch_reciprocal(double* out, const double* in, size_t n, cudaStream_t s);
// strict tracer step after CAAR (caar_euler.cu): Qdp(qn0) - dt*divergence_sphere(vstar*Qdp(qn0)) into the level slice
// (e * qsize_d + iq) * out_stride + out_off of out [slice][L][16]: (qtens, 1, 0), or (Qdp, 2, np1) in place
cudaError_t launch_euler_step(const KernelArgs& a, const double* vstar, double* out, int out_stride, int out_off,
                              int nets, int nete, int qn0, int qsize, double dt, cudaStream_t s);
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
// tracer limiter (caar_limiter.cu), one launch each, on problems (e, iq, k) of [nets,nete) x [0,qsize) x [0,L):
// bounds[e][iq][k] = (max(min Qdp(qtl)/dp3d(dp_tl), 0), max Qdp(qtl)/dp3d(dp_tl)), and limiter_optim_iter_full on
// Qdp(qtl) with weights spheremp * dp3d(dp_tl) within bounds[e][iq][k] (relaxed bounds written back);
// bounds [E][qsize_d][L][2]
cudaError_t launch_tracer_bounds(const KernelArgs& a, int nets, int nete, int qtl, int qsize, int dp_tl, double* bounds,
                                 cudaStream_t s);
cudaError_t launch_limit_tracers(const KernelArgs& a, int nets, int nete, int qtl, int qsize, int dp_tl, double* bounds,
                                 cudaStream_t s);
// vertical remap (caar_remap.cu) of T, v at time level tl and Qdp(qtl) of tracers < qsize on [nets,nete) from dp3d(tl)
// to the reference levels of hyai [nlev+1] (device) and a.hybi, then dp3d(tl) = dp; ps [nelem][16] is scratch. Two
// launches, none for an empty range.
cudaError_t launch_vertical_remap(const KernelArgs& a, const double* hyai, double* ps, int nets, int nete, int tl,
                                  int qtl, int qsize, cudaStream_t s);
// DSS and neighbour bounds (caar_dss.cu) over the connectivity of caar_set_connectivity. The groups of copies of one
// global id, in the order of their owners (first copies in (e, p) order): group g is copy[start[g] .. start[g+1]), each
// copy e*16 + p in (e, p) order. nb[nb_start[e] .. nb_start[e+1]) are the other elements that share a point with e,
// ascending.
struct DssHostTables {
  std::vector<int> start, copy, nb_start, nb;
};
struct DssTables {  // the same on the device
  int ngroups;
  int *start, *copy, *nb_start, *nb;
};
// gid [nelem][16] in the C order; returns the number of groups
int build_dss_tables(const long long* gid, int nelem, DssHostTables* t);
// in place on the selected slices (CAAR_F_DP3D / V / T at time level tl, Qdp(qtl) of tracers < qsize); one launch,
// none when nothing is selected
cudaError_t launch_dss(const KernelArgs& a, const DssTables& t, unsigned mask, int tl, int qtl, int qsize,
                       int weighting, cudaStream_t s);
// out = neighbor_minmax(in) for tracers < qsize, out = in for the others; bounds [nelem][qsize_d][L][2]; one launch,
// none for qsize == 0
cudaError_t launch_neighbor_minmax(const DssTables& t, int nelem, int qsize_d, int L, int qsize, const double* in,
                                   double* out, cudaStream_t s);
// The exchange of shared points between partitioned handles (caar_set_partition). A record is what one part sends
// another for one of its copies (DSS) or one of its elements (neighbour bounds); segment q of a buffer holds the
// records for or from part q, in the order of the global sort by (gid, global e, p) (DSS) or of ascending global
// element (bounds), so that sender and receiver derive the same order from the same map.
//   DSS:    every local group, its copies in global (e, p) order; a local copy is e*16 + p, a remote one -1 - R with R
//           its record in the receive buffer. Segment q is [nv][n_q] (value v of record r at v*n_q + r, v = 0 the
//           copy's spheremp, then the selected slices level by level), starting at double rec_start_q * nv.
//   bounds: nb[nb_start[e] .. nb_start[e+1]) is N(e) in ascending global order, a local element e or nelem + R for row
//           R of the receive buffer; row R is the [qsize][L][2] bounds of one element at double R * qsize * L * 2.
//   The local groups split in two CSRs of the same form, each in owner order: interior (istart / icopy: every copy
//   local) and boundary (bstart / bcopy: at least one remote copy, encoded as in copy). Every copy dss_pack reads is a
//   boundary copy, so the interior launch may run while the segments are in flight.
struct HaloHostTables {
  std::vector<int> start, copy, nb_start, nb;
  std::vector<int> istart, icopy, bstart, bcopy;
  std::vector<int> send_copy, send_el;  // the local copy of every DSS send record, the local element of every row
  // record offsets of the segments, [nparts + 1] each: DSS send, DSS receive, bounds send, bounds receive
  std::vector<int> rec[4];
};
struct HaloTables {  // on the device, but for the record offsets
  int nparts, ngroups, nsend, nrecv, nsend_el, nrecv_el, ninterior, nboundary;
  int *start, *copy, *nb_start, *nb, *send_copy, *send_el, *istart, *icopy, *bstart, *bcopy;
  int2 *send_seg, *recv_seg;  // per DSS record: {first record of its segment, records in that segment}
  int* rec;                   // host [4][nparts + 1]: HaloHostTables::rec
  double *send, *recv;        // the exchange buffers
};
// gid [nelem_global][16] in the C order; part_start as caar_set_partition checks it
void build_halo_tables(const long long* gid, int nelem_global, const int* part_start, int nparts, int part,
                       HaloHostTables* t);
// doubles of one DSS record for a selection (spheremp + every selected value of a copy); 0 when nothing is selected
size_t dss_record_doubles(unsigned mask, int qsize, int L);
// one launch each; the pack none when nothing is selected or there is no record to send
cudaError_t launch_dss_pack(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                            cudaStream_t s);
cudaError_t launch_dss_unpack(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                              int weighting, cudaStream_t s);
// unpack split in two: the interior groups (dss_kernel on istart / icopy), none when there is none, and the boundary
// groups (dss_boundary_kernel on bstart / bcopy, reading the receive buffer), none when there is none
cudaError_t launch_dss_interior(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                                int weighting, cudaStream_t s);
cudaError_t launch_dss_boundary(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                                int weighting, cudaStream_t s);
cudaError_t launch_neighbor_minmax_pack(const HaloTables& t, int qsize_d, int L, int qsize, const double* bounds,
                                        cudaStream_t s);
cudaError_t launch_neighbor_minmax_unpack(const HaloTables& t, int nelem, int qsize_d, int L, int qsize,
                                          const double* in, double* out, cudaStream_t s);
// checksums of the seven mutated arrays + energy norms (caar_aux.cu); partial [nelem][8][2], bits [nelem][7]
cudaError_t launch_checksums(const KernelArgs& a, int tl, int nets, int nete, double cp, double* partial,
                             unsigned long long* bits, double* out16, unsigned long long* out7, cudaStream_t s);
int sm_count();  // SMs of the current device

}  // namespace caar
