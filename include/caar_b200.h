/* caar_b200.h — C-ABI of the B200-native compute_and_apply_rhs ("CAAR") library.
 *
 * This is the drop-in boundary for the one hot path this repository implements:
 * HOMME's compute_and_apply_rhs as extracted in E3SM-Project/tinman_sandbox.
 * Every entry point takes only plain pointers, ints and doubles (no C++ types,
 * no torch types), so it can be bound from C++, Fortran (bind(C)), ctypes, cgo…
 *
 * Reference interfaces replaced (paths relative to the reference checkout,
 * compute_and_apply_rhs_test/cxx/pointers_only/ = "PO/"):
 *
 *   caar_arrays      <- struct Arrays              PO/data_structures.hpp:18-44
 *   caar_constants   <- struct Constants           PO/data_structures.hpp:46-56
 *   caar_control     <- struct Control             PO/data_structures.hpp:58-69
 *   dvv[16]          <- struct Derivative          PO/data_structures.hpp:71-76
 *   ps0, hyai        <- struct HVCoord             PO/data_structures.hpp:10-16
 *   caar_run()       <- Homme::compute_and_apply_rhs(TestData&)
 *                                                  PO/compute_and_apply_rhs.hpp:9
 *                       (body PO/compute_and_apply_rhs.cpp:15-278, callees
 *                        preq_hydrostatic :280-312, preq_omega_ps :314-352,
 *                        gradient/divergence/vorticity_sphere
 *                        PO/sphere_operators.cpp:9-129)
 *   caar_norms()     <- print_results_2norm        PO/compute_and_apply_rhs.cpp:372-399
 *   caar_saxpby_*()  <- saxpby                     saxpby_test/cxx/common.cpp:3-15
 *
 * Host array layout is the reference's, bit for bit: row-major
 * [ie][timelevel][lev][igp][jgp]([comp]) and [ie][igp][jgp][2][2]
 * (PO/test_macros.hpp:7-54, extents PO/data_structures.cpp:14-31).
 *
 * Error convention (the reference has none beyond std::exit/abort): every call
 * returns CAAR_OK (0) or a CAAR_ERR_* code; caar_last_error() returns a
 * thread-local, human readable message for the last failing call.
 * There is NO CPU fallback: without a CUDA device every compute call fails
 * with CAAR_ERR_CUDA.
 */
#ifndef CAAR_B200_H
#define CAAR_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAAR_NP 4 /* GLL points per element edge; compile-time in the reference (config.h.in:1) */

enum {
  CAAR_OK = 0,
  CAAR_ERR_INVALID = 1,     /* bad argument (null pointer, bad dims, bad time level …) */
  CAAR_ERR_CUDA = 2,        /* CUDA runtime/driver error, or no device */
  CAAR_ERR_NOMEM = 3,       /* device or pinned-host allocation failed */
  CAAR_ERR_UNSUPPORTED = 4, /* dims the compiled kernels do not cover */
  CAAR_ERR_STATE = 5        /* call sequence error (e.g. run before set_params) */
};

/* Kernel selection for caar_run. */
enum {
  CAAR_MODE_FAST = 0,   /* fused kernel, register-resident element, parallel warp-shuffle scans,
                           FMA contraction, shared reciprocals: within 1e-12 of the reference */
  CAAR_MODE_STRICT = 1  /* reference operation order, no FMA contraction, IEEE divisions,
                           sequential vertical sums: bit-identical to the reference CPU build */
};

/* Field bits for caar_upload / caar_download (order = struct Arrays). */
enum {
  CAAR_F_D = 1u << 0,
  CAAR_F_DINV = 1u << 1,
  CAAR_F_FCOR = 1u << 2,
  CAAR_F_SPHEREMP = 1u << 3,
  CAAR_F_METDET = 1u << 4,
  CAAR_F_RMETDET = 1u << 5,
  CAAR_F_DP3D = 1u << 6,
  CAAR_F_V = 1u << 7,
  CAAR_F_T = 1u << 8,
  CAAR_F_PHIS = 1u << 9,
  CAAR_F_QDP = 1u << 10,
  CAAR_F_ETA_DOT_DPDN = 1u << 11,
  CAAR_F_OMEGA_P = 1u << 12,
  CAAR_F_PHI = 1u << 13,
  CAAR_F_PECND = 1u << 14,
  CAAR_F_VN0 = 1u << 15,
  CAAR_F_ALL = 0xFFFFu,
  /* the arrays compute_and_apply_rhs writes (PO/compute_and_apply_rhs.cpp:117-118,172-173,251-254,
     and phi via preq_hydrostatic :161) */
  CAAR_F_MUTATED = CAAR_F_DP3D | CAAR_F_V | CAAR_F_T | CAAR_F_ETA_DOT_DPDN | CAAR_F_OMEGA_P |
                   CAAR_F_PHI | CAAR_F_VN0
};
#define CAAR_NUM_FIELDS 16

/* Compile-time dimensions of the reference (config.h.in:1-7), made run-time here. */
typedef struct caar_dims {
  int nelem;   /* number of elements held by this handle (a rank's slice)      */
  int nlev;    /* PLEV: fused kernel instances for 72 and 128 (tuned), every other multiple of 8 up to 64, 80, 96, 112,
                  120; any other value in [2,128] runs on the next larger instance with masked padding levels;
                  above 128 CAAR_MODE_FAST falls back to the reference-order kernel (caar_describe tells) */
  int np;      /* must be 4 */
  int qsize_d; /* QSIZE_D (1 in the reference) */
  int ntl;     /* NUM_TIME_LEVELS (3) */
} caar_dims;

/* struct Arrays, PO/data_structures.hpp:18-44 — same members, same order. */
typedef struct caar_arrays {
  double* elem_D;        /* [E][4][4][2][2] */
  double* elem_Dinv;     /* [E][4][4][2][2] */
  double* elem_fcor;     /* [E][4][4] */
  double* elem_spheremp; /* [E][4][4] */
  double* elem_metdet;   /* [E][4][4] */
  double* elem_rmetdet;  /* [E][4][4] */
  double* elem_state_dp3d; /* [E][ntl][L][4][4] */
  double* elem_state_v;    /* [E][ntl][L][4][4][2] */
  double* elem_state_T;    /* [E][ntl][L][4][4] */
  double* elem_state_phis; /* [E][4][4] */
  double* elem_state_Qdp;  /* [E][qsize_d][2][L][4][4] */
  double* elem_derived_eta_dot_dpdn; /* [E][L+1][4][4] */
  double* elem_derived_omega_p;      /* [E][L][4][4] */
  double* elem_derived_phi;          /* [E][L][4][4] */
  double* elem_derived_pecnd;        /* [E][L][4][4] */
  double* elem_derived_vn0;          /* [E][L][4][4][2] */
} caar_arrays;

/* struct Constants, PO/data_structures.hpp:46-56. */
typedef struct caar_constants {
  double rrearth;
  double eta_ave_w;
  double cp;
  double Rwater_vapor;
  double Rgas;
  double kappa;
} caar_constants;

/* struct Control, PO/data_structures.hpp:58-69. nets/nete are LOCAL to the handle's slice. */
typedef struct caar_control {
  int nets;
  int nete;
  int n0;
  int np1;
  int nm1;
  int qn0; /* -1 = dry (T_v = T), else tracer time level index into Qdp[ie][0][qn0] */
  double dt2;
} caar_control;

typedef struct caar_handle_s* caar_handle;

/* ---- library ---- */
const char* caar_last_error(void);
const char* caar_version(void);
/* number of doubles in field `field_index` (0..15, order of caar_arrays) for given dims; 0 on bad input */
size_t caar_field_count(const caar_dims* dims, int field_index);
/* number of visible CUDA devices, or a negative CAAR_ERR_* */
int caar_device_count(void);

/* ---- handle lifecycle: one handle per GPU (or per element slice) ---- */
/* Allocates the device mirrors of all 16 arrays on `device` and creates a stream. */
int caar_create(caar_handle* out, const caar_dims* dims, int device);
int caar_destroy(caar_handle h);

/* Constants + Derivative + HVCoord of TestData (PO/data_structures.cpp:117-163). hyai has nlev+1 entries. caar_run*
   read only hyai[0]; the whole hyai is kept on the device for caar_vertical_remap. Synchronous. */
int caar_set_params(caar_handle h, const caar_constants* c, const double dvv[16], double ps0,
                    const double* hyai);

/* Vertical coordinate of the following caar_run* calls (SURVEY §8f rank 3). rsplit > 0 (default 1): vertically
   Lagrangian — eta_dot_dpdn = T_vadv = v_vadv = 0, the only branch the reference's C++ code runs
   (PO/compute_and_apply_rhs.cpp:164-171,222-231). rsplit == 0: Eulerian — eta_dot_dpdn at the interfaces from the
   running sum of div(v dp) and hybi, vertical advection of T and v (preq_vertadv), the dp3d update with the
   vertical flux difference, and derived_eta_dot_dpdn accumulates the real flux:
   F/routine_extracted.F90:227-262,270-277,325-334,515-517; LV/CaarFunctor.hpp:504-547. hybi has nlev+1 entries
   (F hvcoord%hybi). A given hybi is kept on the device whatever rsplit is (a NULL hybi with rsplit > 0 keeps the one
   given before): caar_vertical_remap reads it, while caar_run* read hybi only when rsplit == 0, so with rsplit > 0 their
   results do not depend on it. The reference holds no runnable implementation of the Eulerian branch:
   parity is against the tests' own CPU restatement of these formulas only ("parity unpinned", DESIGN.md §3). */
int caar_set_vertical_coordinate(caar_handle h, int rsplit, const double* hybi);

/* Use the caller's CUDA stream (a cudaStream_t passed as void*) for all later work; NULL restores the
   handle's own stream. Lets a torch program time the kernels with its own events. Ordering contract: everything
   already queued through this handle on the previous stream is ordered BEFORE work submitted after the switch (an
   event recorded on the old stream is waited on by the new one); the call itself does not block the host. */
int caar_set_stream(caar_handle h, void* cuda_stream);

/* Host <-> device copies of the selected fields (CAAR_F_* mask). Host pointers are caller-owned and
   are never freed by the library. Pinned host memory makes these asynchronous DMA copies; both calls
   return after the copies completed. */
int caar_upload(caar_handle h, const caar_arrays* host, unsigned field_mask);
int caar_download(caar_handle h, const caar_arrays* host, unsigned field_mask);

/* The same for the element range [e0, e1) only: `host` points at arrays holding exactly those e1-e0 elements of each
   selected field (a rank's window, a test's sample), in the layout above. */
int caar_upload_range(caar_handle h, const caar_arrays* host, unsigned field_mask, int e0, int e1);
int caar_download_range(caar_handle h, const caar_arrays* host, unsigned field_mask, int e0, int e1);

/* ---- second host layout: Fortran flat pointers (SURVEY §8b "alt boundary") ----
   CAAR_LAYOUT_CXX is the layout above. CAAR_LAYOUT_F90 is the memory order of the Fortran arrays themselves
   (F/element_state_mod.F90:17-23, F/element_mod.F90:69-121), element index slowest, exactly what HOMMEXX's
   Elements::init_2d / pull_from_f90_pointers / push_to_f90_pointers read and write
   (LV/Elements.hpp:92-117, LV/Elements.cpp:48-99,154-435):
     fcor, spheremp, metdet, rmetdet, phis  (np,np,nelemd)            = [ie][j][i]
     D, Dinv                                (np,np,2,2,nelemd)        = [ie][b][a][j][i]
     dp3d, T                                (np,np,nlev,tl,nelemd)    = [ie][tl][lev][j][i]
     v                                      (np,np,2,nlev,tl,nelemd)  = [ie][tl][lev][c][j][i]
     Qdp                                    (np,np,nlev,qsize_d,2,nelemd) = [ie][qni][iq][lev][j][i]
     eta_dot_dpdn (nlev+1), omega_p, phi, pecnd (np,np,nlev,nelemd)   = [ie][lev][j][i]
     vn0                                    (np,np,2,nlev,nelemd)     = [ie][lev][c][j][i]
   (the reference's C++ [igp][jgp] equals Fortran (i,j) index for index, so every 4x4 block is transposed in
   memory). The device layout does not change: the copies pass through a device staging buffer and a relayout
   kernel, the hot kernels are the same. With CAAR_LAYOUT_F90 a NULL elem_rmetdet is accepted on upload
   (HOMMEXX passes none): rmetdet = 1/metdet is then computed on the device. */
enum { CAAR_LAYOUT_CXX = 0, CAAR_LAYOUT_F90 = 1 };
int caar_upload_layout(caar_handle h, const caar_arrays* host, unsigned field_mask, int layout);
int caar_download_layout(caar_handle h, const caar_arrays* host, unsigned field_mask, int layout);
/* caar_set_params with Dvv in Fortran memory order (deriv%Dvv(np,np), LV/Derivative.cpp:11-23) */
int caar_set_params_f90(caar_handle h, const caar_constants* c, const double dvv_f90[16], double ps0,
                        const double* hyai);

/* Page-lock / unlock a caller-owned host range in place (cudaHostRegister), so that later
   caar_upload/caar_download of it are DMA copies at PCIe speed. Optional. */
int caar_host_register(void* ptr, size_t bytes);
int caar_host_unregister(void* ptr);

/* Device pointers of the mirrors (for interop, e.g. wrapping in torch tensors, or peer access). */
int caar_device_arrays(caar_handle h, caar_arrays* dev_out);

/* ---- the hot path ---- */
/* nsteps back-to-back evaluations of compute_and_apply_rhs on the resident data, asynchronously on the
   handle's stream. Identical to calling the reference routine nsteps times with the same Control
   (PO/main.cpp:113-121: no time-level rotation between calls). mode = CAAR_MODE_*. */
int caar_run(caar_handle h, const caar_control* ctl, int nsteps, int mode);
/* Which kernel a caar_run in `mode` launches on this handle, as text in buf ("caar_fused_kernel<32,1,0>: nlev=30
   (padded), ..."); *is_fused (may be NULL) = 1 for a fused instance, 0 for the reference-order kernel — for
   CAAR_MODE_FAST that is the fallback for nlev > 128, also announced once on stderr. */
int caar_describe(caar_handle h, int mode, char* buf, size_t len, int* is_fused);

/* Time stepping on the resident state (SURVEY §8f rank 2): nsteps evaluations with the reference's leapfrog
   rotation of the time levels after each one — TestData::update_time_levels, PO/data_structures.cpp:174-180
   (np1 <- nm1, nm1 <- n0, n0 <- old np1), the call the reference driver keeps next to its timed loop
   (PO/main.cpp:118). Asynchronous like caar_run; *ctl holds the rotated levels on return. Aliased levels
   (nm1 = np1 = n0: forward Euler / RK stages, F/routine_extracted.F90:6-16) are legal in every entry point. */
int caar_run_stepping(caar_handle h, caar_control* ctl, int nsteps, int mode);
void caar_update_time_levels(caar_control* ctl);
/* HOMME's default explicit dynamics step, tstep_type == 5 of prim_advance_exp (preqx prim_advance_mod.F90): nsteps
   steps of five compute_and_apply_rhs calls on the resident state, asynchronously on the handle's stream, with the
   rotation of caar_update_time_levels after each step. With (n0, np1, nm1) the levels on entry and w the eta_ave_w
   of caar_set_params, one step is (ctl levels n0 / np1 / nm1, dt2, eta_ave_w; all scalars in double precision):
     1  n0  / nm1 / n0    dt/5      w/4       u1 = u0 + dt/5 R(u0), stored in nm1
     2  nm1 / np1 / n0    dt/5      0         u2 = u0 + dt/5 R(u1)
     3  np1 / np1 / n0    dt/3      0         u3 = u0 + dt/3 R(u2)
     4  np1 / np1 / n0    (2*dt)/3  0         u4 = u0 + 2dt/3 R(u3)
     c  v, T, dp3d at nm1 = (5*X(nm1) - X(n0))/4 on [nets,nete), rounded as Fortran's expression
     5  np1 / np1 / nm1   (3*dt)/4  (3*w)/4   u5 = (5u1 - u0)/4 + 3dt/4 R(u4)
   After the step n0 holds u0, nm1 the combination and np1 u5; then the levels rotate. The per-stage dt2 and
   eta_ave_w apply to that stage only: the handle's constants and ctl->dt2 are neither read nor written. Stages run
   on the kernel caar_run would use in `mode`; each step issues 6 launches (none for an empty element range, which
   still rotates). The levels must be pairwise distinct (stage 1 would overwrite u0), so ntl >= 3. Returns
   CAAR_ERR_STATE before caar_set_params and CAAR_ERR_INVALID for a null control, nsteps < 0, a bad mode or
   levels that are not pairwise distinct, leaving *ctl unchanged. No DSS runs between stages; caar_run_rk5_dss runs one. */
int caar_run_rk5(caar_handle h, caar_control* ctl, double dt, int nsteps, int mode);
/* One stage of caar_run_rk5's step: row `stage` in [0, 5) of the table above (rows 1..5 are stages 0..4), with
   *ctl holding the levels on entry to the step. Stage 4 first launches the combination c, as caar_run_rk5 does. *tl
   receives the level the stage wrote: nm1 for stage 0, np1 for the others; that is the level a DSS after the stage
   assembles. *ctl is not rotated: the caller calls caar_update_time_levels after stage 4. Exactly:
     stages 0..4, then caar_update_time_levels(ctl)                          is caar_run_rk5(h, ctl, dt, 1, mode)
     the same with caar_dss(h, CAAR_F_V | CAAR_F_T | CAAR_F_DP3D, *tl, 0, 0, CAAR_DSS_ASSEMBLE) after every stage
                                                                             is caar_run_rk5_dss(h, ctl, dt, 1, mode)
   bit for bit: both run these stages' launches in this order. On partitioned handles (caar_set_partition) the DSS
   after every stage is caar_dss_pack, the caller's transport, caar_dss_interior and caar_dss_boundary (below); over a
   block partition the parts then hold, bit for bit, the slices of caar_run_rk5_dss on one handle that holds the whole
   mesh. Asynchronous on the handle's stream; 1 launch (2 for stage 4), none for an empty element range. Returns every
   error of caar_run_rk5 (pairwise-distinct levels included) and CAAR_ERR_INVALID for a stage outside [0, 5) or a null
   tl; a rejected call launches nothing and changes nothing, *tl included. */
int caar_rk5_stage(caar_handle h, const caar_control* ctl, double dt, int stage, int mode, int* tl);
int caar_sync(caar_handle h);
/* number of kernel launches issued through this handle since creation (caar_run, caar_run_rk5: 6 per step,
   caar_run_rk5_dss: 11 per step, caar_rk5_stage: 1 (2 for stage 4), caar_advect_tracers: 4 per step, caar_tracer_bounds and caar_limit_tracers: 1 per call
   (none for an empty range or qsize == 0), caar_dss and caar_neighbor_minmax: 1 per call (none when nothing is
   selected), caar_dss_pack / caar_dss_unpack and caar_neighbor_minmax_pack / caar_neighbor_minmax_unpack: 1 per call
   (none when nothing is selected, and none for a pack of a part that shares no point), caar_dss_interior /
   caar_dss_boundary: at most 1 per call (none when nothing is selected or the part has no interior / boundary group),
   caar_vertical_remap: 2 per call (none for an empty range), caar_euler_step, caar_norms,
   ...) */
long long caar_launch_count(caar_handle h);
/* CUDA-event stopwatch on the stream the kernels are launched on: start records an event, stop records a
   second one, waits for it and returns the device time between the two in milliseconds. */
int caar_timer_start(caar_handle h);
int caar_timer_stop(caar_handle h, float* ms);

/* ---- the step after CAAR: tracer advection RHS (SURVEY §8f rank 4) ----
   qtens[ie][iq][k] = Qdp[ie][iq][qn0][k] - dt * divergence_sphere(vstar[ie][k] * Qdp[ie][iq][qn0][k]) for tracers
   iq < qsize, every level, elements [nets,nete): EulerStepFunctor::operator() (LV/EulerStepFunctor.hpp:33-66) =
   divergence_sphere_update(alpha=-dt, beta=1) (LV/SphereOperators.hpp:362-403) with the reference's
   divergence_sphere (PO/sphere_operators.cpp:50-89). Uses the handle's Dinv/metdet/rmetdet/Qdp mirrors, Dvv and
   rrearth, plus two arrays that struct Arrays does not hold, owned by the handle and moved with
   caar_extra_upload/download in the pointers_only conventions:
     CAAR_X_VSTAR  vstar [E][L][4][4][2]        (derived%vstar(np,np,2,nlev), F/element_mod.F90:70; input)
     CAAR_X_QTENS  qtens [E][qsize_d][L][4][4]  (buffers.qtens, LV/Elements.hpp:71; output)
   Asynchronous on the handle's stream (caar_sync / caar_extra_download wait). mode as in caar_run. */
enum { CAAR_X_VSTAR = 0, CAAR_X_QTENS = 1, CAAR_X_TENSORVISC = 2, CAAR_X_SCALAR_IN = 3, CAAR_X_SCALAR_OUT = 4 };
#define CAAR_NUM_EXTRA 5
size_t caar_extra_count(const caar_dims* dims, int which);
int caar_extra_upload(caar_handle h, int which, const double* host);
int caar_extra_download(caar_handle h, int which, double* host);
int caar_euler_step(caar_handle h, int nets, int nete, int qn0, int qsize, double dt, int mode);
/* HOMME's Eulerian tracer advection step with rkstage = 3 (prim_advection_mod: three euler_step calls and
   qdp_time_avg): nsteps steps of length dt on the resident Qdp, asynchronously on the handle's stream. With n0 = *qn0
   on entry and np1 = 1 - n0, one step is, for tracers iq < qsize of elements [nets,nete):
     1  Qdp(np1) = Qdp(n0)  - dt/2 div(vstar Qdp(n0))
     2  Qdp(np1) = Qdp(np1) - dt/2 div(vstar Qdp(np1))      (in place)
     3  Qdp(np1) = Qdp(np1) - dt/2 div(vstar Qdp(np1))      (in place)
     a  Qdp(np1) = (Qdp(n0) + 2*Qdp(np1))/3, rounded as Fortran's expression (one add, one division; 2*b is exact)
   then *qn0 = np1 (TimeLevel_Qdp swaps n0_qdp and np1_qdp). Each stage is exactly caar_euler_step with dt/2 (exact in
   double) on the kernel caar_euler_step uses in `mode`, storing into Qdp(np1) instead of
   CAAR_X_QTENS, so a stage is bit-identical to caar_euler_step's qtens. The stability polynomial is
   1 + z + z^2/2 + z^3/12: second order. Only Qdp[nets:nete][0:qsize][np1] changes: Qdp(n0), the tracers iq >= qsize,
   the elements outside the range, CAAR_X_VSTAR and CAAR_X_QTENS (which this call does not allocate) keep their values.
   Element-local, like caar_run_rk5: no DSS, no limiter and no tracer hyperviscosity run between stages. HOMME stores
   spheremp*Qtens, runs the DSS and multiplies by rspheremp; without the DSS the two products cancel up to rounding,
   so a stage stores Qtens itself. vstar is CAAR_X_VSTAR, fixed for all three stages; HOMME recomputes it each stage
   from vn0 and a dp that moves with rhs_multiplier, so the two agree only when that term vanishes (coupling vstar to
   vn0 is not part of this call). Each step issues 4 launches (none for an empty range or qsize == 0, which still
   toggle *qn0). Returns CAAR_ERR_STATE before caar_set_params and CAAR_ERR_INVALID for a null handle or qn0,
   *qn0 not 0 or 1, a bad element range, qsize outside [0, qsize_d], nsteps < 0 or a bad mode, leaving *qn0 unchanged. */
int caar_advect_tracers(caar_handle h, int nets, int nete, int* qn0, int qsize, double dt, int nsteps, int mode);

/* ---- the tracer limiter: HOMME's quasi-monotone limiter, euler_step with limiter_option == 8 ----
   The element-local bounds at the start of a tracer step, and limiter_optim_iter_full, which euler_step applies to
   Qtens with the weights spheremp and dp_star. Both work on the handle's Qdp, dp3d and spheremp mirrors and on one more
   handle-owned array (it is not a CAAR_X_* extra array):
     bounds [E][qsize_d][L][2] = (qmin, qmax) per element, tracer and level; zero on first use.
   caar_bounds_upload / caar_bounds_download copy the whole array and return when the copy is complete.

   One problem is one (e, iq, k) with e in [nets, nete), iq < qsize, k < L; p[n] are the 16 values of
   Qdp[e][iq][qtl][k], d[n] those of dp3d[e][dp_tl][k], w[n] those of spheremp[e]. The index n visits the points in
   Fortran sequence-association order, i fastest: Fortran (i,j) is [igp][jgp] here, so n runs over the offsets
   4*igp + jgp in the order 0, 4, 8, 12, 1, 5, ... . Every sum is sequential in that order, and every operation is
   rounded separately (no FMA contraction).

   caar_tracer_bounds: per problem qmin = min_n p[n]/d[n], qmax = max_n p[n]/d[n], then if (qmin < 0) qmin = 0, written
   to bounds[e][iq][k]. This is HOMME's Qtens_biharmonic = Qdp(n0)/dp; qmin = max(minval, 0); qmax = maxval. HOMME
   then widens the bounds over neighbouring elements (neighbor_minmax); that is the caller's job, between the two calls,
   through caar_bounds_download and caar_bounds_upload.

   caar_limit_tracers: per problem, in place on Qdp(qtl) and on the problem's bounds (minp, maxp), with TOL = 5e-14 and
   MAXITER = 15 (np*np - 1):
     c[n] = w[n]*d[n];  x[n] = p[n]/d[n]
     sumc = sum c[n]
     if (sumc <= 0) leave the problem (p and its bounds) untouched
     mass = sum (c[n]*x[n])
     if (mass < minp*sumc) minp = mass/sumc            relax the bounds so that a solution exists
     if (mass > maxp*sumc) maxp = mass/sumc
     repeat MAXITER times:
       addmass = 0
       for n: if (x[n] > maxp) { addmass = addmass + (x[n]-maxp)*c[n]; x[n] = maxp }
              if (x[n] < minp) { addmass = addmass - (minp-x[n])*c[n]; x[n] = minp }
       if (|addmass| <= TOL*|mass|) exit
       if (addmass > 0) { ws = sum over x[n] < maxp of c[n]; if (ws == 0) exit; for x[n] < maxp: x[n] = x[n] + addmass/ws }
       else             { ws = sum over x[n] > minp of c[n]; if (ws == 0) exit; for x[n] > minp: x[n] = x[n] + addmass/ws }
     p[n] = x[n]*d[n];  bounds[e][iq][k] = (minp, maxp)    the relaxed bounds persist (Fortran's intent(inout))
   A problem that leaves the loop after MAXITER keeps the state after its last redistribution, as HOMME does. The one
   departure from the literal Fortran is the ws == 0 exit: there the Fortran divides by zero. After the relaxation
   that point can only be reached through rounding.

   Both calls are asynchronous on the handle's stream, always run in this order (there is no mode: the results are
   bit-reproducible) and read no parameter, so they work before caar_set_params. They leave dp3d, spheremp, the other
   Qdp time level, the tracers iq >= qsize, the elements outside [nets, nete) and the bounds outside the problems
   untouched; caar_tracer_bounds leaves Qdp untouched too. Each call adds one launch, none for an empty range or
   qsize == 0. CAAR_ERR_INVALID for a null handle or host pointer, a bad element range, qtl not 0 or 1, dp_tl outside
   [0, ntl) or qsize outside [0, qsize_d]; a rejected call launches nothing and changes nothing.

   One limited tracer step on the resident state (the bounds of the step's input, the limiter once on its output; this
   is not HOMME's per-stage limiting inside the step, whose dp_star this library does not hold):
     1  caar_tracer_bounds(h, nets, nete, qn0, qsize, dp_tl)
     2  caar_neighbor_minmax(h, qsize)                                 widen the bounds over neighbouring elements
     3  caar_advect_tracers(h, nets, nete, &qn0, qsize, dt, 1, mode)
     4  caar_limit_tracers(h, nets, nete, qn0, qsize, dp_tl)          with the new qn0
     5  caar_dss(h, CAAR_F_QDP, 0, qn0, qsize, CAAR_DSS_PROJECT)      with the new qn0
   Steps 2 and 5 need caar_set_connectivity and act on every element of the handle. HOMME also runs a DSS
   after each of the three stages inside the step; caar_advect_tracers does not, so this step equals HOMME's only up to
   that difference. */
int caar_bounds_upload(caar_handle h, const double* host);
int caar_bounds_download(caar_handle h, double* host);
int caar_tracer_bounds(caar_handle h, int nets, int nete, int qtl, int qsize, int dp_tl);
int caar_limit_tracers(caar_handle h, int nets, int nete, int qtl, int qsize, int dp_tl);

/* ---- the vertical remap: HOMME's vertical_remap for rsplit > 0 ----
   On the vertically Lagrangian coordinate (rsplit > 0) every step moves mass between the layers of dp3d; HOMME brings
   the columns back to the hybrid reference levels every rsplit steps, after prim_step. caar_vertical_remap is that call
   with remap1 = remap_Q_ppm and vert_remap_q_alg = 1 (PPM with mirrored ghost cells), on the columns (e, p) of the
   elements [nets, nete), asynchronously on the handle's stream. Per column:
     dp_star = dp3d(tl);  ps = hyai[0]*ps0 + S, S the sequential sum of dp_star over k
     dp[k] = (hyai[k+1]-hyai[k])*ps0 + (hybi[k+1]-hybi[k])*ps         (hyai of caar_set_params, hybi of
                                                                       caar_set_vertical_coordinate)
     T(tl) is remapped as T*dp_star and divided by dp; so is each component of v(tl); Qdp(qtl) of the tracers
     iq < qsize is remapped as mass; finally dp3d(tl) = dp.
   Nothing else changes: the other time levels, the other Qdp level, the tracers iq >= qsize, the elements outside the
   range and every derived field. There is no mode: every operation is rounded separately (no FMA contraction, IEEE
   divisions, sums sequential in k), so the results are bit-reproducible and equal tests/remap_oracle.py bit for bit.

   The restatement, in HOMME's 1-based indices (C level k-1 is Fortran level k). Ghost cells gs = 2 are mirrored:
   x(1-i) = x(i) and x(nlev+i) = x(nlev+1-i) for i = 1, 2. Integer powers are products: x**2 = x*x, x**3 = (x*x)*x.
   Expressions evaluate left to right as written. Per column:
     pio(1)=0; pin(1)=0; for k=1..nlev: pio(k+1)=pio(k)+dpo(k); pin(k+1)=pin(k)+dpn(k)     (dpo=dp_star, dpn=dp)
     pio(nlev+2)=pio(nlev+1)+1;  pin(nlev+1)=pio(nlev+1);  mirror dpo into -1..nlev+2
     for k=1..nlev: kk=k; while pio(kk) <= pin(k+1) { kk=kk+1; if kk==nlev+2 break }; kk=kk-1; if kk==nlev+1 kk=nlev
                    kid(k)=kk;  z2(k) = (pin(k+1) - (pio(kk)+pio(kk+1))*0.5) / dpo(kk)          (z1 = -0.5)
     grid, with dx = dpo:
       j=0..nlev+1: r1=dx(j)/((dx(j-1)+dx(j))+dx(j+1));  r2=(2*dx(j-1)+dx(j))/(dx(j+1)+dx(j));
                    r3=(dx(j)+2*dx(j+1))/(dx(j-1)+dx(j))
       j=0..nlev:   r4=dx(j)/(dx(j)+dx(j+1));  r5=1/(((dx(j-1)+dx(j))+dx(j+1))+dx(j+2));
                    r6=((2*dx(j+1))*dx(j))/(dx(j)+dx(j+1));  r7=(dx(j-1)+dx(j))/(2*dx(j)+dx(j+1));
                    r8=(dx(j+2)+dx(j+1))/(2*dx(j+1)+dx(j));  r9=(dx(j)*(dx(j-1)+dx(j)))/(2*dx(j)+dx(j+1));
                    r10=(dx(j+1)*(dx(j+1)+dx(j+2)))/(dx(j)+2*dx(j+1))
     per field f (the values to remap: T*dp_star, v_c*dp_star, or Qdp):
       masso(1)=0; k=1..nlev: masso(k+1)=masso(k)+f(k); a(k)=f(k)/dpo(k);   mirror a into -1..nlev+2
       j=0..nlev+1: da = r1*(r2*(a(j+1)-a(j)) + r3*(a(j)-a(j-1)))
                    dma(j) = min(|da|, 2*|a(j)-a(j-1)|, 2*|a(j+1)-a(j)|) * copysign(1, da)
                    if ((a(j+1)-a(j))*(a(j)-a(j-1)) <= 0) dma(j) = 0
       j=0..nlev:   ai(j) = (a(j) + r4*(a(j+1)-a(j))) + r5*(((r6*(r7-r8))*(a(j+1)-a(j)) - r9*dma(j+1)) + r10*dma(j))
       j=1..nlev:   al=ai(j-1); ar=ai(j)
                    if ((ar-a(j))*(a(j)-al) <= 0) { al=a(j); ar=a(j) }
                    if ((ar-al)*(a(j)-(al+ar)/2) >  (ar-al)**2/6) al = 3*a(j) - 2*ar
                    if ((ar-al)*(a(j)-(al+ar)/2) < -(ar-al)**2/6) ar = 3*a(j) - 2*al
                    c0(j) = 1.5*a(j) - (al+ar)/4;  c1(j) = ar-al;  c2(j) = -6*a(j) + 3*(al+ar)
       massn1=0; k=1..nlev: kk=kid(k); x2=z2(k); x1=-0.5
                    massn2 = masso(kk) + ((c0*(x2-x1) + (c1*(x2**2-x1**2))/2) + (c2*(x2**3-x1**3))/3)(kk) * dpo(kk)
                    f(k) = massn2 - massn1;  massn1 = massn2
   The result is T = f/dp, v_c = f/dp and Qdp = f. The search never returns a cell above k-1, so a new interface more
   than one cell above its old position falls into HOMME's extrapolated parabola of cell k-1; the result still
   conserves mass. The contract covers dp_star > 0 and dp > 0 (HOMME aborts on a negative thickness); outside it the
   call only keeps every index in bounds, with kid clamped to [1, nlev].

   Errors: CAAR_ERR_STATE before caar_set_params or when no hybi was ever given; CAAR_ERR_UNSUPPORTED on a handle with
   rsplit == 0; CAAR_ERR_INVALID for a null handle, a bad element range, tl outside [0, ntl), qtl not 0 or 1 or qsize
   outside [0, qsize_d]. A rejected call launches nothing and changes nothing. 2 launches, none for an empty range.

   One remap interval of HOMME's rsplit > 0 time loop, on a handle that holds the whole mesh (E elements):
     rsplit times: caar_run_rk5_dss(h, &ctl, dt, 1, mode), then the limited tracer step above (with the new qn0)
     caar_vertical_remap(h, 0, E, ctl.n0, qn0, qsize)     ctl.n0: after the rotation, the level the last step wrote
   The remap is column-local (no connectivity, no DSS, no exchange), so partitioned handles run it unchanged. */
int caar_vertical_remap(caar_handle h, int nets, int nete, int tl, int qtl, int qsize);

/* ---- the direct stiffness summation (DSS) over shared element-boundary points ----
   HOMME's compute_and_apply_rhs stores spheremp*(state + dt*rhs) and then assembles the values at the GLL points that two
   to four elements share: edgeVpack, bndry_exchangeV, edgeVunpack, then a multiply by rspheremp
   (F/routine_extracted.F90:519+); euler_step does the same to spheremp*Qtens. These calls do that on the device, over
   every element of the handle, from a map of the points' global ids.

   caar_set_connectivity: gid[E][4][4] is the global id of every GLL point, in the [igp][jgp] order of the C++ layout with
   CAAR_LAYOUT_CXX; with CAAR_LAYOUT_F90 it is the memory order of HOMME's elem%gdofP(np,np,nelemd) = [ie][j][i]. Points
   with equal ids are one point; any 64-bit values are accepted, and two points of one element may share an id.
   Synchronous; replaces an earlier map; works before caar_set_params. The tables are built once on the host
   (a sort of the 16 E copies) and kept on the device until caar_destroy. CAAR_ERR_INVALID for a null handle or gid or a
   bad layout, CAAR_ERR_UNSUPPORTED for nelem >= 2^27 (a copy is packed as e*16 + p in 32 bits).

   caar_dss, exactly. The copies of a point are the pairs (e, p) with equal gid, p = 4*igp + jgp, ordered by ascending
   (e, p); the first is the point's owner. With f_c the field value at copy c and s_c = spheremp[e][p] at call time
   (a re-uploaded spheremp is used; nothing is cached):
     m = s_c0 + s_c1 + ...                   sequential in copy order
     r = 1.0 / m                             IEEE division: HOMME's rspheremp, the reciprocal of the assembled mass
     CAAR_DSS_ASSEMBLE: S = f_c0 + f_c1 + ...               for inputs that carry spheremp already (the output of
                                                            compute_and_apply_rhs, weak-form operators)
     CAAR_DSS_PROJECT:  S = s_c0*f_c0 + s_c1*f_c1 + ...     each product rounded; for fields without the factor (Qtens
                                                            as caar_advect_tracers stores it, Qdp)
     every copy = S * r
   Every operation is rounded separately (no FMA contraction; there is no mode), so the result is bit-reproducible; a
   point with one copy gets f*r or (s*f)*r, with no add. Each component of v is a scalar field of its own (HOMME's v is
   in lat-lon components, continuous across panels). m == 0 gives what IEEE gives. The fields are those of field_mask
   within {CAAR_F_DP3D, CAAR_F_V, CAAR_F_T} at time level tl, and Qdp(qtl) of tracers iq < qsize when CAAR_F_QDP is set;
   nothing else changes. tl, qtl and qsize are checked whatever the mask.
   Departure from HOMME: edgeVunpack adds an element's neighbours to that element's own value, so HOMME's copies of one
   point may differ in the last bit; here every copy receives the identical value.
   Partitioned handles: only the copies this handle holds are summed; caar_dss_pack / caar_dss_unpack below assemble
   the copies other handles hold too.

   caar_neighbor_minmax: HOMME's neighbor_minmax on the handle's limiter bounds (caar_tracer_bounds). N(e) is the set of
   elements other than e that share at least one gid with e (on a cubed sphere the edge and vertex neighbours). For every
   e, tracer iq < qsize and level k: qmin starts from e's own value, then for each n in N(e) in ascending order
   if (qmin_n < qmin) qmin = qmin_n; qmax the same with >. Every neighbour's bounds are read before any is changed (a
   second handle-owned array), so the result does not depend on launch order. Tracers iq >= qsize are unchanged.

   Both are asynchronous on the handle's stream and add one launch; caar_dss none when nothing is selected (mask 0, or
   only CAAR_F_QDP with qsize == 0), caar_neighbor_minmax none for qsize == 0. They need no caar_set_params.
   CAAR_ERR_STATE before caar_set_connectivity; CAAR_ERR_INVALID for a null handle, mask bits outside the four fields,
   tl outside [0, ntl), qtl not 0 or 1, qsize outside [0, qsize_d] or a weighting other than the two below. A rejected
   call launches nothing and changes nothing. */
enum { CAAR_DSS_ASSEMBLE = 0, CAAR_DSS_PROJECT = 1 };
int caar_set_connectivity(caar_handle h, const long long* gid, int layout);
int caar_dss(caar_handle h, unsigned field_mask, int tl, int qtl, int qsize, int weighting);
int caar_neighbor_minmax(caar_handle h, int qsize);
/* caar_run_rk5's step with caar_dss(h, CAAR_F_V | CAAR_F_T | CAAR_F_DP3D, np1 of the stage, 0, 0, CAAR_DSS_ASSEMBLE)
   after each of its five stages: HOMME's tstep_type 5 with the DSS of compute_and_apply_rhs. The combination reads the
   assembled u1. Each step issues 11 launches (5 stages, the combination, 5 DSS); the levels rotate as in caar_run_rk5.
   Returns CAAR_ERR_STATE before caar_set_params or caar_set_connectivity, CAAR_ERR_INVALID for an element range other than
   [0, nelem) (the DSS spans the handle), and every error of caar_run_rk5, leaving *ctl unchanged. */
int caar_run_rk5_dss(caar_handle h, caar_control* ctl, double dt, int nsteps, int mode);

/* ---- the DSS and neighbor_minmax across partitioned handles: HOMME's edgeVpack / bndry_exchangeV / edgeVunpack ----
   A mesh of nelem_global elements is cut into nparts contiguous blocks, one per handle (one per GPU or rank). The
   library packs what other parts need into a device send buffer; the caller moves opaque segments with its own
   transport (NCCL, CUDA-aware MPI, device copies between handles of one process); the library unpacks from a device
   receive buffer and finishes the sum. Over any block partition the assembled values of every handle are, bit for bit,
   those caar_dss / caar_neighbor_minmax give on one handle that holds the whole mesh: the copies of a point are ordered
   by (global e, p), and every operation is rounded separately as there.

   caar_set_partition: gid[nelem_global][4][4] is the global-id map of the whole mesh, in CAAR_LAYOUT_CXX or
   CAAR_LAYOUT_F90 order as in caar_set_connectivity. part_start[nparts + 1] ascends strictly from 0 to nelem_global;
   this handle holds global elements [part_start[part], part_start[part + 1]), local element e being global
   part_start[part] + e. Callers whose parts are not contiguous (HOMME's space-filling-curve partitions give each rank a
   set) renumber their elements first, so that each rank's local order defines its block. Synchronous; builds every
   table on the host once (a sort of the 16 nelem_global copies); replaces any earlier connectivity or partition, and a
   later caar_set_connectivity replaces it; works before caar_set_params. From then on caar_dss and
   caar_neighbor_minmax keep their local-only meaning, as if caar_set_connectivity had been given the handle's slice of
   gid; so does caar_run_rk5_dss. On a part, HOMME's step is caar_rk5_stage with caar_dss_pack, the transport,
   caar_dss_interior and caar_dss_boundary after every stage (at caar_rk5_stage).
   Allocates the two exchange buffers, sized for the largest selection (all four fields with qsize_d tracers, and the
   bounds of qsize_d tracers), until caar_destroy or the next map. CAAR_ERR_INVALID for a null handle, gid or
   part_start, nparts < 1, part outside [0, nparts), part_start not ascending from 0 to nelem_global, a block size other
   than the handle's nelem, or a bad layout; CAAR_ERR_UNSUPPORTED for nelem_global >= 2^27.

   caar_dss_pack / caar_dss_unpack take caar_dss's arguments, with its checks and selection rules. pack writes the send
   buffer: segment q (for every other part q) holds, for each local copy of a point that part q also holds a copy of,
   the copy's spheremp and its selected values at every level. unpack reads the receive buffer and performs the whole DSS
   of this handle in place, interior points included: the copies of every point, those held by other parts taken from
   the received segments, are ordered by (global e, p), and m, r = 1/m and S follow caar_dss's formulas in that order;
   every local copy gets S*r. The remote spheremp values come from the records, so a re-uploaded spheremp is used there
   too. The record layout and the order inside a segment are the library's, derived by both sides from the same global
   map; the caller moves segment p->q of part p's send buffer to segment p of part q's receive buffer, byte for byte.
   pack and unpack of one exchange must use the same field_mask, tl, qtl and qsize: mixing them is a caller error that
   is not detected. With nparts == 1 unpack equals caar_dss bit for bit.

   caar_dss_interior / caar_dss_boundary split caar_dss_unpack in two, with its arguments, checks and selection rules.
   The local groups (the points with a copy on this handle) are interior when every copy is on this handle and boundary
   when at least one copy is on another part. interior assembles the interior groups; it reads neither buffer and
   writes no copy that caar_dss_pack reads (a copy pack sends belongs to a point another part holds), so it may be
   queued before or after pack and may run while the segments are in flight. boundary assembles the boundary groups
   and reads the receive buffer, so it follows the transport. The two, in either order, give caar_dss_unpack's result
   bit for bit (the same operations in the same order per point), and so, over a block partition, the whole-mesh
   caar_dss. Each is at most one launch: none when nothing is selected, interior none when every local group has a
   remote copy, boundary none when there is no remote copy (nparts == 1, or a part that shares no point).

   caar_neighbor_minmax_pack / caar_neighbor_minmax_unpack: the same on the limiter bounds. Segment q holds the
   [qsize][L][2] bounds of every local element that has a neighbour in part q. unpack is caar_neighbor_minmax's rule over
   N(e) of the whole mesh: e's own value first, then every neighbour, local or remote, in ascending global element order
   (which also fixes which of -0.0 and +0.0 survives). It writes the second array as caar_neighbor_minmax does.

   caar_halo_segments: for op CAAR_HALO_DSS with (field_mask, qsize), or CAAR_HALO_MINMAX with qsize (the mask is then
   only checked), returns the device send and receive buffers and the offsets, in doubles, of every segment: segment q
   is [send_off[q], send_off[q+1]) of *send and [recv_off[q], recv_off[q+1]) of *recv. send_off of p->q on part p has
   the size of recv_off of q<-p on part q; the segments to and from this part itself are empty. Synchronous, launches
   nothing; CAAR_ERR_INVALID for null outputs or a bad op, mask or qsize.

   pack, unpack, interior and boundary are asynchronous on the handle's stream. The caller's transport must be ordered
   after pack, and unpack or boundary after the transport (with caar_set_stream on the transport's stream this is free). Before
   caar_set_partition every call here but caar_set_partition returns CAAR_ERR_STATE; a rejected call launches nothing
   and changes nothing. */
enum { CAAR_HALO_DSS = 0, CAAR_HALO_MINMAX = 1 };
int caar_set_partition(caar_handle h, const long long* gid, int nelem_global, const int* part_start, int nparts,
                       int part, int layout);
int caar_dss_pack(caar_handle h, unsigned field_mask, int tl, int qtl, int qsize, int weighting);
int caar_dss_unpack(caar_handle h, unsigned field_mask, int tl, int qtl, int qsize, int weighting);
int caar_dss_interior(caar_handle h, unsigned field_mask, int tl, int qtl, int qsize, int weighting);
int caar_dss_boundary(caar_handle h, unsigned field_mask, int tl, int qtl, int qsize, int weighting);
int caar_neighbor_minmax_pack(caar_handle h, int qsize);
int caar_neighbor_minmax_unpack(caar_handle h, int qsize);
int caar_halo_segments(caar_handle h, int op, unsigned field_mask, int qsize, double** send, double** recv,
                       size_t* send_off, size_t* recv_off);

/* ---- the weak-form operators behind hyperviscosity (SURVEY §8f rank 4) ----
   Level-local like the tracer step, on the same kernel skeleton, in the pointers_only index conventions
   (HOMMEXX view (igp,jgp) == pointers_only [jgp][igp]); uses the handle's Dinv / spheremp mirrors, Dvv, rrearth and
   three more handle-owned arrays moved with caar_extra_upload/download:
     CAAR_X_TENSORVISC  tensorVisc [E][4][4][2][2]  (like elem_D; LV/SphereOperators.hpp:560, input)
     CAAR_X_SCALAR_IN   scalar field [E][L][4][4]   (input of the laplace operators)
     CAAR_X_SCALAR_OUT  scalar field [E][L][4][4]   (output of every operator; input AND output of *_REPLACE)
     CAAR_OP_DIVERGENCE_WK           out = divergence_sphere_wk(CAAR_X_VSTAR)            LV/SphereOperators.hpp:493-535
     CAAR_OP_LAPLACE_SIMPLE          out = divergence_sphere_wk(gradient_sphere(in))     LV/SphereOperators.hpp:537-553
     CAAR_OP_LAPLACE_TENSOR          out = divergence_sphere_wk(tensorVisc.gradient_sphere(in))   :555-599
     CAAR_OP_LAPLACE_TENSOR_REPLACE  the same with in == out (CAAR_X_SCALAR_OUT)                   :601-636
   (the reference's accumulator `Scalar dd;` at :521 is zero-initialised by the vendored Vector's default constructor,
   LV/vector/KokkosKernels_Vector_SIMD.hpp:32-37: the sum starts from 0.) CAAR_MODE_STRICT is bit-identical to the
   reference's own code (which the tests run under a serial Kokkos stand-in), CAAR_MODE_FAST within 1e-12 of the field maximum.
   Asynchronous on the handle's stream. */
enum { CAAR_OP_DIVERGENCE_WK = 0, CAAR_OP_LAPLACE_SIMPLE = 1, CAAR_OP_LAPLACE_TENSOR = 2, CAAR_OP_LAPLACE_TENSOR_REPLACE = 3 };
int caar_sphere_wk(caar_handle h, int op, int nets, int nete, int mode);

/* Sum of squares of v, T, dp3d at time level `tl` over elements [nets,nete) — the three quantities
   print_results_2norm takes the sqrt of (PO/compute_and_apply_rhs.cpp:384-398). Returned as SUMS OF
   SQUARES so that ranks can all-reduce them before the sqrt. Synchronous. */
int caar_norms(caar_handle h, int tl, int nets, int nete, double sumsq[3]);

/* Checksums of every array compute_and_apply_rhs writes, and two energy norms, over elements [nets,nete) — what the
   ranks of a partitioned run all-reduce after the timed loop (north star: "final allreduce of field checksums and
   energy norms"); the reference's own protocol prints only the three norms above (PO/compute_and_apply_rhs.cpp:372-399).
   Field order: 0 dp3d(tl), 1 v(tl), 2 T(tl), 3 derived_eta_dot_dpdn, 4 derived_omega_p, 5 derived_phi, 6 derived_vn0.
     sum, sumsq  plain sums in a fixed order (all-reduce with SUM; compare at ~1e-13 relative)
     bits        sum of the IEEE-754 bit patterns mod 2^64: exact and order-independent, so two runs (or a run and the
                 bit-exact CPU reference) hold identical data iff these agree — all-reduce as 64-bit integers with SUM
     energy      { sum spheremp*0.5*(u^2+v^2)*dp3d, sum spheremp*cp*T*dp3d } at time level tl: the kinetic and internal
                 energy integrands of the reference's diagnostics (F/routine_extracted.F90:396-410)
   Synchronous. */
typedef struct caar_checksum {
  double sum[7];
  double sumsq[7];
  unsigned long long bits[7];
  double energy[2];
} caar_checksum;
int caar_checksums(caar_handle h, int tl, int nets, int nete, caar_checksum* out);

/* ---- the hot path on HOST arrays (what Homme::compute_and_apply_rhs(TestData&) means to its caller,
   PO/compute_and_apply_rhs.hpp:9, called from the timed loop PO/main.cpp:113-121) ---- */
/* ONE evaluation over [ctl->nets, ctl->nete) whose inputs are read from the caller's `host` arrays and whose
   results are in the `host` arrays (and in the device mirrors) when the call returns. Only the slices the
   routine actually reads travel host->device (time levels n0 and nm1 of dp3d/v/T, Qdp[qn0], vn0, pecnd,
   omega_p, the 2-D geometry: 13 level-fields + 1664 B per element) and only what it writes travels back
   (time level np1 of dp3d/v/T, vn0, phi, omega_p: 8 level-fields); every other host value is left
   untouched, as in the reference. The element range is cut into chunks of `chunk_elems` elements
   (0 = automatic) that flow through three CUDA streams — copy-in | kernel | copy-out — so that both PCIe
   directions and the SMs work concurrently. Page-locked host arrays (caar_host_register, or
   cudaMallocHost/torch pinned memory) are needed for the overlap; pageable memory works but serialises.
   Synchronous. STRICT mode additionally moves eta_dot_dpdn both ways (the += 0 update of PO:164-171). */
int caar_run_host(caar_handle h, const caar_arrays* host, const caar_control* ctl, int mode, int chunk_elems);
/* chunk_elems == CAAR_HOST_ZERO_COPY: no staging at all — the kernel reads the caller's arrays and writes the
   results over PCIe itself (TMA / LDG / bulk stores on mapped host memory), one launch for the whole range.
   Needs every array page-locked AND device-mapped (caar_host_register, cudaHostAlloc, torch pinned memory);
   fails with CAAR_ERR_INVALID otherwise. The device mirrors are NOT updated on this path. */
#define CAAR_HOST_ZERO_COPY (-1)
/* bytes one caar_run_host call with this control moves in each direction; CAAR_ERR_INVALID for a null argument, a
   bad control or a bad mode */
int caar_host_traffic(caar_handle h, const caar_control* ctl, int mode, size_t* h2d_bytes, size_t* d2h_bytes);

/* Reference-facing one-shot: create -> set_params -> caar_run_host -> destroy on `device`, i.e. exactly what
   Homme::compute_and_apply_rhs(TestData&) means for host arrays. */
int caar_compute_and_apply_rhs_host(const caar_dims* dims, const caar_arrays* host,
                                    const caar_control* ctl, const caar_constants* c,
                                    const double dvv[16], double ps0, const double* hyai, int device,
                                    int mode);

/* ---- saxpby bandwidth calibrator (saxpby_test/cxx/common.cpp:3-15): x = a*x + b*y ---- */
/* device pointers, asynchronous on `cuda_stream` (NULL = default stream) */
int caar_saxpby_device(double a, double b, double* x_dev, const double* y_dev, size_t n,
                       void* cuda_stream);
/* host pointers: H2D, `sweeps` sweeps, D2H on `device` */
int caar_saxpby_host(double a, double b, double* x, const double* y, size_t n, int sweeps, int device);

#ifdef __cplusplus
}
#endif
#endif /* CAAR_B200_H */
