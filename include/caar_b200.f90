! caar_b200.f90 — Fortran 2003 (ISO_C_BINDING) interface of the C-ABI in include/caar_b200.h, for the reference's
! Fortran test driver (compute_and_apply_rhs_test/fortran/main.F90:200-211 calls
! compute_and_apply_rhs(np1,nm1,n0,qn0,dt2,elem,hvcoord,deriv,nets,nete,eta_ave_w), fortran/routine_mod.F90:7).
!
! The Fortran arrays are handed over as they lie in memory (CAAR_LAYOUT_F90, the order HOMMEXX reads its F90 pointers
! in, level_vectorized_ppscan/Elements.cpp:48-99,154-292): one contiguous array per field with the element index
! slowest, e.g. real(c_double), target :: v(np,np,2,nlev,timelevels,nelemd). The reference keeps its fields inside
! the derived type elem(ie)%state%...; a caller copies them once into such arrays (or declares them so) — see
! INTEGRATION.md section 4 for the wrapper that gives routine_mod.F90's compute_and_apply_rhs signature.
!
! There is no Fortran compiler in the build image: this file is NOT compiled by the repository's tests. The C side
! guards the struct layouts it assumes with static_asserts (csrc/caar_capi.cu: sizeof / offsetof of caar_dims,
! caar_arrays, caar_constants, caar_control, caar_checksum); every bind(C) type below lists the same members in the same
! order, all of them interoperable scalars, so the Fortran processor lays them out as the companion C compiler does.
module caar_b200
  use, intrinsic :: iso_c_binding
  implicit none
  private

  ! ---- constants of include/caar_b200.h
  integer(c_int), parameter, public :: CAAR_OK = 0, CAAR_ERR_INVALID = 1, CAAR_ERR_CUDA = 2, CAAR_ERR_NOMEM = 3, &
                                       CAAR_ERR_UNSUPPORTED = 4, CAAR_ERR_STATE = 5
  integer(c_int), parameter, public :: CAAR_MODE_FAST = 0, CAAR_MODE_STRICT = 1
  integer(c_int), parameter, public :: CAAR_LAYOUT_CXX = 0, CAAR_LAYOUT_F90 = 1
  integer(c_int), parameter, public :: CAAR_F_D = 1, CAAR_F_DINV = 2, CAAR_F_FCOR = 4, CAAR_F_SPHEREMP = 8, &
       CAAR_F_METDET = 16, CAAR_F_RMETDET = 32, CAAR_F_DP3D = 64, CAAR_F_V = 128, CAAR_F_T = 256, CAAR_F_PHIS = 512, &
       CAAR_F_QDP = 1024, CAAR_F_ETA_DOT_DPDN = 2048, CAAR_F_OMEGA_P = 4096, CAAR_F_PHI = 8192, CAAR_F_PECND = 16384, &
       CAAR_F_VN0 = 32768, CAAR_F_ALL = 65535
  integer(c_int), parameter, public :: CAAR_F_MUTATED = 64 + 128 + 256 + 2048 + 4096 + 8192 + 32768
  integer(c_int), parameter, public :: CAAR_X_VSTAR = 0, CAAR_X_QTENS = 1, CAAR_X_TENSORVISC = 2, CAAR_X_SCALAR_IN = 3, &
                                       CAAR_X_SCALAR_OUT = 4
  integer(c_int), parameter, public :: CAAR_OP_DIVERGENCE_WK = 0, CAAR_OP_LAPLACE_SIMPLE = 1, CAAR_OP_LAPLACE_TENSOR = 2, &
                                       CAAR_OP_LAPLACE_TENSOR_REPLACE = 3

  ! ---- struct caar_dims (5 x int = 20 bytes)
  type, bind(C), public :: caar_dims
    integer(c_int) :: nelem, nlev, np, qsize_d, ntl
  end type caar_dims

  ! ---- struct caar_arrays (16 x double* = 128 bytes), the order of struct Arrays
  !      (compute_and_apply_rhs_test/cxx/pointers_only/data_structures.hpp:18-44); fill with c_loc(array)
  type, bind(C), public :: caar_arrays
    type(c_ptr) :: elem_D, elem_Dinv, elem_fcor, elem_spheremp, elem_metdet, elem_rmetdet
    type(c_ptr) :: elem_state_dp3d, elem_state_v, elem_state_T, elem_state_phis, elem_state_Qdp
    type(c_ptr) :: elem_derived_eta_dot_dpdn, elem_derived_omega_p, elem_derived_phi, elem_derived_pecnd, elem_derived_vn0
  end type caar_arrays

  ! ---- struct caar_constants (6 x double = 48 bytes): physical_constants.F90 + eta_ave_w
  type, bind(C), public :: caar_constants
    real(c_double) :: rrearth, eta_ave_w, cp, Rwater_vapor, Rgas, kappa
  end type caar_constants

  ! ---- struct caar_control (6 x int, 1 x double = 32 bytes). Time levels and qn0 are ZERO-based on the C side:
  !      pass n0-1, np1-1, nm1-1, qn0-1 (qn0 = -1 in Fortran means dry and stays -1); nets/nete: [nets-1, nete)
  type, bind(C), public :: caar_control
    integer(c_int) :: nets, nete, n0, np1, nm1, qn0
    real(c_double) :: dt2
  end type caar_control

  ! ---- struct caar_checksum (7 + 7 doubles, 7 x 64-bit integers, 2 doubles = 184 bytes)
  type, bind(C), public :: caar_checksum
    real(c_double) :: sum(7), sumsq(7)
    integer(c_int64_t) :: bits(7)     ! unsigned on the C side: compare for equality / add with wrap-around only
    real(c_double) :: energy(2)
  end type caar_checksum

  public :: caar_create, caar_destroy, caar_set_params_f90, caar_set_vertical_coordinate, caar_upload_layout, &
            caar_download_layout, caar_run, caar_run_stepping, caar_run_rk5, caar_update_time_levels, caar_sync, caar_norms, &
            caar_checksums, caar_euler_step, caar_advect_tracers, caar_sphere_wk, caar_extra_upload, caar_extra_download, caar_last_error, &
            caar_host_register, caar_host_unregister, caar_describe

  interface
    ! int caar_create(caar_handle* out, const caar_dims* dims, int device);
    function caar_create(handle, dims, device) bind(C, name="caar_create") result(rc)
      import :: c_ptr, c_int, caar_dims
      type(c_ptr), intent(out) :: handle
      type(caar_dims), intent(in) :: dims
      integer(c_int), value :: device
      integer(c_int) :: rc
    end function
    function caar_destroy(handle) bind(C, name="caar_destroy") result(rc)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: rc
    end function
    ! deriv%Dvv(np,np) as stored by Fortran; hyai(nlev+1) = hvcoord%hyai
    function caar_set_params_f90(handle, c, dvv, ps0, hyai) bind(C, name="caar_set_params_f90") result(rc)
      import :: c_ptr, c_int, c_double, caar_constants
      type(c_ptr), value :: handle
      type(caar_constants), intent(in) :: c
      real(c_double), intent(in) :: dvv(4, 4)
      real(c_double), value :: ps0
      real(c_double), intent(in) :: hyai(*)
      integer(c_int) :: rc
    end function
    ! rsplit > 0: vertically Lagrangian; rsplit = 0: Eulerian, hybi(nlev+1) = hvcoord%hybi
    function caar_set_vertical_coordinate(handle, rsplit, hybi) bind(C, name="caar_set_vertical_coordinate") result(rc)
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: handle
      integer(c_int), value :: rsplit
      real(c_double), intent(in) :: hybi(*)
      integer(c_int) :: rc
    end function
    function caar_upload_layout(handle, host, field_mask, layout) bind(C, name="caar_upload_layout") result(rc)
      import :: c_ptr, c_int, caar_arrays
      type(c_ptr), value :: handle
      type(caar_arrays), intent(in) :: host
      integer(c_int), value :: field_mask, layout
      integer(c_int) :: rc
    end function
    function caar_download_layout(handle, host, field_mask, layout) bind(C, name="caar_download_layout") result(rc)
      import :: c_ptr, c_int, caar_arrays
      type(c_ptr), value :: handle
      type(caar_arrays), intent(in) :: host
      integer(c_int), value :: field_mask, layout
      integer(c_int) :: rc
    end function
    function caar_run(handle, ctl, nsteps, mode) bind(C, name="caar_run") result(rc)
      import :: c_ptr, c_int, caar_control
      type(c_ptr), value :: handle
      type(caar_control), intent(in) :: ctl
      integer(c_int), value :: nsteps, mode
      integer(c_int) :: rc
    end function
    function caar_run_stepping(handle, ctl, nsteps, mode) bind(C, name="caar_run_stepping") result(rc)
      import :: c_ptr, c_int, caar_control
      type(c_ptr), value :: handle
      type(caar_control), intent(inout) :: ctl
      integer(c_int), value :: nsteps, mode
      integer(c_int) :: rc
    end function
    ! int caar_run_rk5(caar_handle h, caar_control* ctl, double dt, int nsteps, int mode); tstep_type == 5
    function caar_run_rk5(handle, ctl, dt, nsteps, mode) bind(C, name="caar_run_rk5") result(rc)
      import :: c_ptr, c_int, c_double, caar_control
      type(c_ptr), value :: handle
      type(caar_control), intent(inout) :: ctl
      real(c_double), value :: dt
      integer(c_int), value :: nsteps, mode
      integer(c_int) :: rc
    end function
    subroutine caar_update_time_levels(ctl) bind(C, name="caar_update_time_levels")
      import :: caar_control
      type(caar_control), intent(inout) :: ctl
    end subroutine
    function caar_sync(handle) bind(C, name="caar_sync") result(rc)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: rc
    end function
    ! sums of squares of v, T, dp3d at (zero-based) time level tl over elements [nets, nete)
    function caar_norms(handle, tl, nets, nete, sumsq) bind(C, name="caar_norms") result(rc)
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: handle
      integer(c_int), value :: tl, nets, nete
      real(c_double), intent(out) :: sumsq(3)
      integer(c_int) :: rc
    end function
    function caar_checksums(handle, tl, nets, nete, cs) bind(C, name="caar_checksums") result(rc)
      import :: c_ptr, c_int, caar_checksum
      type(c_ptr), value :: handle
      integer(c_int), value :: tl, nets, nete
      type(caar_checksum), intent(out) :: cs
      integer(c_int) :: rc
    end function
    function caar_euler_step(handle, nets, nete, qn0, qsize, dt, mode) bind(C, name="caar_euler_step") result(rc)
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: handle
      integer(c_int), value :: nets, nete, qn0, qsize
      real(c_double), value :: dt
      integer(c_int), value :: mode
      integer(c_int) :: rc
    end function
    ! int caar_advect_tracers(caar_handle h, int nets, int nete, int* qn0, int qsize, double dt, int nsteps, int mode);
    ! HOMME's three-stage tracer step (rkstage = 3); qn0 (zero-based n0_qdp) comes back toggled once per step
    function caar_advect_tracers(handle, nets, nete, qn0, qsize, dt, nsteps, mode) bind(C, name="caar_advect_tracers") &
        result(rc)
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: handle
      integer(c_int), value :: nets, nete
      integer(c_int), intent(inout) :: qn0
      integer(c_int), value :: qsize
      real(c_double), value :: dt
      integer(c_int), value :: nsteps, mode
      integer(c_int) :: rc
    end function
    function caar_sphere_wk(handle, op, nets, nete, mode) bind(C, name="caar_sphere_wk") result(rc)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int), value :: op, nets, nete, mode
      integer(c_int) :: rc
    end function
    ! the arrays beyond struct Arrays (vstar, qtens, tensorVisc, scalar in / out) travel in the C++ layout
    function caar_extra_upload(handle, which, host) bind(C, name="caar_extra_upload") result(rc)
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: handle
      integer(c_int), value :: which
      real(c_double), intent(in) :: host(*)
      integer(c_int) :: rc
    end function
    function caar_extra_download(handle, which, host) bind(C, name="caar_extra_download") result(rc)
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: handle
      integer(c_int), value :: which
      real(c_double), intent(out) :: host(*)
      integer(c_int) :: rc
    end function
    function caar_host_register(ptr, bytes) bind(C, name="caar_host_register") result(rc)
      import :: c_ptr, c_int, c_size_t
      type(c_ptr), value :: ptr
      integer(c_size_t), value :: bytes
      integer(c_int) :: rc
    end function
    function caar_host_unregister(ptr) bind(C, name="caar_host_unregister") result(rc)
      import :: c_ptr, c_int
      type(c_ptr), value :: ptr
      integer(c_int) :: rc
    end function
    function caar_describe(handle, mode, buf, len, is_fused) bind(C, name="caar_describe") result(rc)
      import :: c_ptr, c_int, c_char, c_size_t
      type(c_ptr), value :: handle
      integer(c_int), value :: mode
      character(kind=c_char), intent(out) :: buf(*)
      integer(c_size_t), value :: len
      integer(c_int), intent(out) :: is_fused
      integer(c_int) :: rc
    end function
    ! const char* caar_last_error(void): convert with c_f_pointer to a character(kind=c_char) array up to c_null_char
    function caar_last_error() bind(C, name="caar_last_error") result(msg)
      import :: c_ptr
      type(c_ptr) :: msg
    end function
  end interface
end module caar_b200
