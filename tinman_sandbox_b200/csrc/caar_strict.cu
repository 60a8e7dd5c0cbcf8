// caar_strict.cu — CAAR_MODE_STRICT: compute_and_apply_rhs in the reference's own operation order.
//
// Purpose: a GPU result that is BIT-IDENTICAL to the reference's `g++ -O3` x86-64 build, so that the
// parity of the algorithm is proven independently of FMA contraction and parallel-sum reordering.
// Every floating-point operation is an explicit round-to-nearest intrinsic (__dmul_rn/__dadd_rn/
// __ddiv_rn: never contracted into FMAs), the 4-term Dvv contractions are summed in index order
// starting from 0.0, and the three vertical integrals run sequentially per column.
//
// One CTA per element; level-local phases use one thread per (level, igp, jgp) point in a strided
// loop; the vertical integrals use 16 threads (one per column). Temporaries live in shared memory
// (11 level-fields = 11*nlev*128 B), mirroring the reference's per-call temporaries
// (PO/compute_and_apply_rhs.cpp:18-35). This is the correctness anchor, not the fast path.
//
// Reference line numbers in comments: PO = compute_and_apply_rhs_test/cxx/pointers_only.
#include "caar_device.cuh"

namespace caar {
namespace {

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dvd(double a, double b) { return __ddiv_rn(a, b); }

// gradient_sphere at point (a,b) of a 4x4 scalar tile s (PO/sphere_operators.cpp:21-47).
// v1[a][b] = (sum_i Dvv[i][a]*s[i][b])*rrearth ; v2[a][b] = (sum_i Dvv[i][b]*s[a][i])*rrearth
__device__ __forceinline__ void grad_point(const double* s, const double* dvv, const double* dinv_pt,
                                           double rrearth, int a, int b, double& g0, double& g1) {
  double sx = 0.0, sy = 0.0;
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    sx = add(sx, mul(dvv[i * NP + a], s[i * NP + b]));
    sy = add(sy, mul(dvv[i * NP + b], s[a * NP + i]));
  }
  const double v1 = mul(sx, rrearth), v2 = mul(sy, rrearth);
  g0 = add(mul(dinv_pt[0], v1), mul(dinv_pt[2], v2));
  g1 = add(mul(dinv_pt[1], v1), mul(dinv_pt[3], v2));
}

__global__ void __launch_bounds__(512) caar_strict_kernel(const KernelArgs A) {
  extern __shared__ double sm[];
  const int L = A.nlev;
  const int lf = L * PTS;
  double* p = sm;                 // [L][16]
  double* gp = p + lf;            // [L][16][2]
  double* vgp = gp + 2 * lf;      // [L][16]      vgrad_p, later ttens
  double* vdp = vgp + lf;         // [L][16][2]   later vtens1 | vtens2
  double* divdp = vdp + 2 * lf;   // [L][16]
  double* vort = divdp + lf;      // [L][16]
  double* Tv = vort + lf;         // [L][16]
  double* om = Tv + lf;           // [L][16]
  double* ph = om + lf;           // [L][16]      phii during the scan, then Ephi
  double* eta = ph + lf;          // [L+1][16]    eta_dot_dpdn at the interfaces (Eulerian branch only)
  const bool eul = (A.rsplit == 0);
  __shared__ double geo_D[64], geo_Dinv[64], geo_met[16], geo_rmet[16], s_dvv[16];

  const int ie = A.nets + blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x;
  const size_t e = (size_t)ie;

  const double* dp_n0 = A.dp3d + (e * A.ntl + A.n0) * lf;
  const double* v_n0 = A.v + (e * A.ntl + A.n0) * lf * 2;
  const double* T_n0 = A.T + (e * A.ntl + A.n0) * lf;
  double* vn0 = A.vn0 + e * lf * 2;
  double* phi = A.phi + e * lf;
  double* omega_p = A.omega_p + e * lf;
  double* eta_dot = A.eta_dot_dpdn + e * (size_t)(L + 1) * PTS;
  const double* pecnd = A.pecnd + e * lf;
  const double* fcor = A.fcor + e * PTS;
  const double* spheremp = A.spheremp + e * PTS;
  const double* phis = A.phis + e * PTS;

  if (tid < 64) {
    geo_D[tid] = A.D[e * 64 + tid];
    geo_Dinv[tid] = A.Dinv[e * 64 + tid];
  }
  if (tid < 16) {
    geo_met[tid] = A.metdet[e * 16 + tid];
    geo_rmet[tid] = A.rmetdet[e * 16 + tid];
    s_dvv[tid] = A.dvv[tid];
  }

  // A: pressure at mid levels, top-down (PO:76-97)
  if (tid < PTS) {
    double pk = add(mul(A.hyai0, A.ps0), mul(0.5, dp_n0[tid]));
    p[tid] = pk;
    for (int k = 1; k < L; ++k) {
      pk = add(add(pk, mul(0.5, dp_n0[(k - 1) * PTS + tid])), mul(0.5, dp_n0[k * PTS + tid]));
      p[k * PTS + tid] = pk;
    }
  }
  __syncthreads();

  // B1: grad_p, vgrad_p, vdp, derived_vn0 (PO:103-120); C: T_v (PO:126-156)
  for (int n = tid; n < lf; n += nt) {
    const int k = n >> 4, q = n & 15, a = q >> 2, b = q & 3;
    double g0, g1;
    grad_point(p + k * PTS, s_dvv, geo_Dinv + q * 4, A.rrearth, a, b, g0, g1);
    gp[n * 2] = g0;
    gp[n * 2 + 1] = g1;
    const double v1 = v_n0[n * 2], v2 = v_n0[n * 2 + 1], dpn = dp_n0[n];
    vgp[n] = add(mul(v1, g0), mul(v2, g1));
    const double u = mul(v1, dpn), w = mul(v2, dpn);
    vdp[n * 2] = u;
    vdp[n * 2 + 1] = w;
    vn0[n * 2] = add(vn0[n * 2], mul(A.eta_ave_w, u));
    vn0[n * 2 + 1] = add(vn0[n * 2 + 1], mul(A.eta_ave_w, w));
    if (A.qn0 == -1) {
      Tv[n] = T_n0[n];
    } else {
      const double* Qdp = A.Qdp + ((e * A.qsize_d + 0) * 2 + A.qn0) * lf;
      const double Qt = dvd(Qdp[n], dpn);
      Tv[n] = mul(T_n0[n], add(1.0, mul(sub(dvd(A.Rwv, A.Rgas), 1.0), Qt)));
    }
  }
  __syncthreads();

  // B2: divergence_sphere(vdp) (PO/sphere_operators.cpp:62-88), vorticity_sphere(v_n0) (:102-128)
  for (int n = tid; n < lf; n += nt) {
    const int k = n >> 4, q = n & 15, a = q >> 2, b = q & 3;
    const double* vd = vdp + k * PTS * 2;
    const double* vv = v_n0 + k * PTS * 2;
    double dudx = 0.0, dvdy = 0.0, dvdx = 0.0, dudy = 0.0;
#pragma unroll
    for (int m = 0; m < NP; ++m) {
      const int qc = m * NP + b;  // point [m][b]
      const int qr = a * NP + m;  // point [a][m]
      // gv[m][b][0], gv[a][m][1]
      const double gvc = mul(geo_met[qc], add(mul(geo_Dinv[qc * 4 + 0], vd[qc * 2]), mul(geo_Dinv[qc * 4 + 1], vd[qc * 2 + 1])));
      const double gvr = mul(geo_met[qr], add(mul(geo_Dinv[qr * 4 + 2], vd[qr * 2]), mul(geo_Dinv[qr * 4 + 3], vd[qr * 2 + 1])));
      dudx = add(dudx, mul(s_dvv[m * NP + a], gvc));
      dvdy = add(dvdy, mul(s_dvv[m * NP + b], gvr));
      // vcov[m][b][1], vcov[a][m][0]
      const double vc1 = add(mul(geo_D[qc * 4 + 1], vv[qc * 2]), mul(geo_D[qc * 4 + 3], vv[qc * 2 + 1]));
      const double vc0 = add(mul(geo_D[qr * 4 + 0], vv[qr * 2]), mul(geo_D[qr * 4 + 2], vv[qr * 2 + 1]));
      dvdx = add(dvdx, mul(s_dvv[m * NP + a], vc1));
      dudy = add(dudy, mul(s_dvv[m * NP + b], vc0));
    }
    divdp[n] = mul(mul(add(dudx, dvdy), geo_rmet[q]), A.rrearth);
    vort[n] = mul(mul(sub(dvdx, dudy), geo_rmet[q]), A.rrearth);
  }
  __syncthreads();

  // D: preq_hydrostatic, bottom-up (PO:287-311) on warp 0; E: preq_omega_ps, top-down (PO:319-351) on warp 1
  if (tid < PTS) {
    const int q = tid;
    int k = L - 1;
    double hkk = dvd(mul(0.5, dp_n0[k * PTS + q]), p[k * PTS + q]);
    double hkl = mul(2.0, hkk);
    double phii = mul(mul(A.Rgas, Tv[k * PTS + q]), hkl);
    double out = add(phis[q], mul(mul(A.Rgas, Tv[k * PTS + q]), hkk));
    phi[k * PTS + q] = out;
    ph[k * PTS + q] = out;
    for (k = L - 2; k > 0; --k) {
      hkk = dvd(mul(0.5, dp_n0[k * PTS + q]), p[k * PTS + q]);
      hkl = mul(2.0, hkk);
      out = add(add(phis[q], phii), mul(mul(A.Rgas, Tv[k * PTS + q]), hkk));
      phii = add(phii, mul(mul(A.Rgas, Tv[k * PTS + q]), hkl));
      phi[k * PTS + q] = out;
      ph[k * PTS + q] = out;
    }
    hkk = dvd(mul(0.5, dp_n0[q]), p[q]);
    out = add(add(phis[q], phii), mul(mul(A.Rgas, Tv[q]), hkk));
    phi[q] = out;
    ph[q] = out;
  } else if (tid >= 32 && tid < 32 + PTS) {
    const int q = tid - 32;
    double ckk = dvd(0.5, p[q]);
    double term = divdp[q];
    om[q] = sub(dvd(vgp[q], p[q]), mul(ckk, term));
    double suml = term;
    for (int k = 1; k < L - 1; ++k) {
      ckk = dvd(0.5, p[k * PTS + q]);
      const double ckl = mul(2.0, ckk);
      term = divdp[k * PTS + q];
      om[k * PTS + q] = sub(sub(dvd(vgp[k * PTS + q], p[k * PTS + q]), mul(ckl, suml)), mul(ckk, term));
      suml = add(suml, term);
    }
    const int k = L - 1;
    ckk = dvd(0.5, p[k * PTS + q]);
    const double ckl = mul(2.0, ckk);
    term = divdp[k * PTS + q];
    om[k * PTS + q] = sub(sub(dvd(vgp[k * PTS + q], p[k * PTS + q]), mul(ckl, suml)), mul(ckk, term));
  } else if (eul && tid >= 64 && tid < 64 + PTS) {
    // Eulerian branch: eta_dot_dpdn at the interfaces from the running sum of divdp and hybi
    // (F/routine_extracted.F90:233-254), on warp 2
    const int q = tid - 64;
    double sdot = 0.0;
    for (int k = 0; k < L; ++k) {
      sdot = add(sdot, divdp[k * PTS + q]);
      eta[(k + 1) * PTS + q] = sdot;
    }
    for (int k = 0; k < L - 1; ++k) eta[(k + 1) * PTS + q] = sub(mul(A.hybi[k + 1], sdot), eta[(k + 1) * PTS + q]);
    eta[q] = 0.0;
    eta[L * PTS + q] = 0.0;
  }
  __syncthreads();

  // F: accumulate derived fields (PO:164-183; Eulerian: F/routine_extracted.F90:270-277); Ephi (PO:196)
  for (int n = tid; n < lf + PTS; n += nt) {
    eta_dot[n] = add(eta_dot[n], mul(A.eta_ave_w, eul ? eta[n] : 0.0));
    if (n < lf) {
      omega_p[n] = add(omega_p[n], mul(A.eta_ave_w, om[n]));
      const double v1 = v_n0[n * 2], v2 = v_n0[n * 2 + 1];
      ph[n] = add(add(mul(0.5, add(mul(v1, v1), mul(v2, v2))), ph[n]), pecnd[n]);
    }
  }
  __syncthreads();

  // G: tendencies (PO:200-231). vtens1|vtens2 overwrite vdp, ttens overwrites vgrad_p.
  for (int n = tid; n < lf; n += nt) {
    const int k = n >> 4, q = n & 15, a = q >> 2, b = q & 3;
    double t0, t1, e0, e1;
    grad_point(T_n0 + k * PTS, s_dvv, geo_Dinv + q * 4, A.rrearth, a, b, t0, t1);
    const double v1 = v_n0[n * 2], v2 = v_n0[n * 2 + 1];
    const double vgrad_T = add(mul(v1, t0), mul(v2, t1));
    grad_point(ph + k * PTS, s_dvv, geo_Dinv + q * 4, A.rrearth, a, b, e0, e1);
    const double gpterm = dvd(Tv[n], p[n]);
    const double glnps1 = mul(mul(A.Rgas, gpterm), gp[n * 2]);
    const double glnps2 = mul(mul(A.Rgas, gpterm), gp[n * 2 + 1]);
    const double fv = add(fcor[q], vort[n]);
    double vt1, vt2, tt;
    if (eul) {
      // preq_vertadv (LV/CaarFunctor.hpp:504-547) and the Fortran tendencies (F/routine_extracted.F90:325-334)
      const double rdp = dvd(1.0, dp_n0[n]);
      const double facp = mul(mul(0.5, rdp), eta[n + PTS]), facm = mul(mul(0.5, rdp), eta[n]);
      double T_vadv, vv0, vv1;
      if (k == 0) {
        T_vadv = mul(facp, sub(T_n0[n + PTS], T_n0[n]));
        vv0 = mul(facp, sub(v_n0[(n + PTS) * 2], v1));
        vv1 = mul(facp, sub(v_n0[(n + PTS) * 2 + 1], v2));
      } else if (k < L - 1) {
        T_vadv = add(mul(facp, sub(T_n0[n + PTS], T_n0[n])), mul(facm, sub(T_n0[n], T_n0[n - PTS])));
        vv0 = add(mul(facp, sub(v_n0[(n + PTS) * 2], v1)), mul(facm, sub(v1, v_n0[(n - PTS) * 2])));
        vv1 = add(mul(facp, sub(v_n0[(n + PTS) * 2 + 1], v2)), mul(facm, sub(v2, v_n0[(n - PTS) * 2 + 1])));
      } else {
        T_vadv = mul(facm, sub(T_n0[n], T_n0[n - PTS]));
        vv0 = mul(facm, sub(v1, v_n0[(n - PTS) * 2]));
        vv1 = mul(facm, sub(v2, v_n0[(n - PTS) * 2 + 1]));
      }
      vt1 = sub(sub(add(-vv0, mul(v2, fv)), e0), glnps1);
      vt2 = sub(sub(sub(-vv1, mul(v1, fv)), e1), glnps2);
      tt = add(sub(-T_vadv, vgrad_T), mul(mul(A.kappa, Tv[n]), om[n]));
    } else {
      // -v_vadv + ... with v_vadv == +0.0: (-0.0) + x == x and (-0.0) - x == -x for every x
      vt1 = sub(sub(mul(v2, fv), e0), glnps1);
      vt2 = sub(sub(-mul(v1, fv), e1), glnps2);
      // T_vadv - vgrad_T with T_vadv == +0.0
      tt = add(sub(0.0, vgrad_T), mul(mul(A.kappa, Tv[n]), om[n]));
    }
    vdp[n] = vt1;
    vdp[lf + n] = vt2;
    vgp[n] = tt;
  }
  __syncthreads();

  // H: apply (PO:245-257)
  {
    double* v_np1 = A.v + (e * A.ntl + A.np1) * lf * 2;
    double* T_np1 = A.T + (e * A.ntl + A.np1) * lf;
    double* dp_np1 = A.dp3d + (e * A.ntl + A.np1) * lf;
    const double* v_nm1 = A.v + (e * A.ntl + A.nm1) * lf * 2;
    const double* T_nm1 = A.T + (e * A.ntl + A.nm1) * lf;
    const double* dp_nm1 = A.dp3d + (e * A.ntl + A.nm1) * lf;
    for (int n = tid; n < lf; n += nt) {
      const int q = n & 15;
      const double mp = spheremp[q];
      const double a0 = mul(mp, add(v_nm1[n * 2], mul(A.dt2, vdp[n])));
      const double a1 = mul(mp, add(v_nm1[n * 2 + 1], mul(A.dt2, vdp[lf + n])));
      const double a2 = mul(mp, add(T_nm1[n], mul(A.dt2, vgp[n])));
      const double dflux = eul ? sub(add(divdp[n], eta[n + PTS]), eta[n]) : divdp[n];  // F/routine_extracted.F90:515-517
      const double a3 = mul(mp, sub(dp_nm1[n], mul(A.dt2, dflux)));
      v_np1[n * 2] = a0;
      v_np1[n * 2 + 1] = a1;
      T_np1[n] = a2;
      dp_np1[n] = a3;
    }
  }
}

}  // namespace

size_t strict_smem_bytes(int nlev) { return ((size_t)12 * nlev + 1) * PTS * sizeof(double); }
bool strict_supports(int nlev) { return strict_smem_bytes(nlev) <= 200 * 1024; }

cudaError_t launch_strict(const KernelArgs& a, cudaStream_t s) {
  const size_t smem = strict_smem_bytes(a.nlev);
  static LaunchCache cache;
  int per_sm = 0;
  if (cudaError_t e = setup_launch(caar_strict_kernel, 512, smem, cache, &per_sm)) return e;
  const int n = a.nete - a.nets;
  if (n <= 0) return cudaSuccess;
  caar_strict_kernel<<<n, 512, smem, s>>>(a);
  return cudaGetLastError();
}

}  // namespace caar
