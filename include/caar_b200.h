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

/* Constants + Derivative + HVCoord of TestData (PO/data_structures.cpp:117-163). hyai has nlev+1 entries. */
int caar_set_params(caar_handle h, const caar_constants* c, const double dvv[16], double ps0,
                    const double* hyai);

/* Vertical coordinate of the following caar_run* calls (SURVEY §8f rank 3). rsplit > 0 (default 1): vertically
   Lagrangian — eta_dot_dpdn = T_vadv = v_vadv = 0, the only branch the reference's C++ code runs
   (PO/compute_and_apply_rhs.cpp:164-171,222-231). rsplit == 0: Eulerian — eta_dot_dpdn at the interfaces from the
   running sum of div(v dp) and hybi, vertical advection of T and v (preq_vertadv), the dp3d update with the
   vertical flux difference, and derived_eta_dot_dpdn accumulates the real flux:
   F/routine_extracted.F90:227-262,270-277,325-334,515-517; LV/CaarFunctor.hpp:504-547. hybi has nlev+1 entries
   (F hvcoord%hybi; ignored when rsplit > 0). The reference holds no runnable implementation of this branch:
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
   levels that are not pairwise distinct, leaving *ctl unchanged. No DSS runs between stages. */
int caar_run_rk5(caar_handle h, caar_control* ctl, double dt, int nsteps, int mode);
int caar_sync(caar_handle h);
/* number of kernel launches issued through this handle since creation (caar_run, caar_run_rk5: 6 per step,
   caar_advect_tracers: 4 per step, caar_euler_step, caar_norms, ...) */
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
   double) on the kernel caar_euler_step uses in `mode` (CAAR_EULER_V1 included), storing into Qdp(np1) instead of
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
/* bytes one caar_run_host call with this control moves in each direction */
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
