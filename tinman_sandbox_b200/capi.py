"""ctypes binding of include/caar_b200.h (libcaar_b200.so).

This is the Python stand-in for the reference-side binding (INTEGRATION.md shows the C++ one): it mirrors
the reference's TestData members by name (compute_and_apply_rhs_test/cxx/pointers_only/data_structures.hpp)
and calls straight through the C-ABI. Arrays are numpy float64 in the reference's host layout.
No CPU fallback: a missing library or a missing device raises CaarError.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

FIELD_NAMES = (
    "elem_D", "elem_Dinv", "elem_fcor", "elem_spheremp", "elem_metdet", "elem_rmetdet",
    "elem_state_dp3d", "elem_state_v", "elem_state_T", "elem_state_phis", "elem_state_Qdp",
    "elem_derived_eta_dot_dpdn", "elem_derived_omega_p", "elem_derived_phi", "elem_derived_pecnd",
    "elem_derived_vn0",
)
FIELD_BIT = {n: 1 << i for i, n in enumerate(FIELD_NAMES)}
MUTATED_FIELDS = ("elem_state_dp3d", "elem_state_v", "elem_state_T", "elem_derived_eta_dot_dpdn",
                  "elem_derived_omega_p", "elem_derived_phi", "elem_derived_vn0")
F_ALL = 0xFFFF
F_MUTATED = sum(FIELD_BIT[n] for n in MUTATED_FIELDS)
MODE_FAST, MODE_STRICT = 0, 1
LAYOUT_CXX, LAYOUT_F90 = 0, 1
X_VSTAR, X_QTENS, X_TENSORVISC, X_SCALAR_IN, X_SCALAR_OUT = 0, 1, 2, 3, 4
OP_DIVERGENCE_WK, OP_LAPLACE_SIMPLE, OP_LAPLACE_TENSOR, OP_LAPLACE_TENSOR_REPLACE = 0, 1, 2, 3

# every symbol include/caar_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = (
    "caar_last_error", "caar_version", "caar_field_count", "caar_device_count", "caar_create",
    "caar_destroy", "caar_set_params", "caar_set_stream", "caar_upload", "caar_download",
    "caar_device_arrays", "caar_host_register", "caar_host_unregister", "caar_run", "caar_run_host",
    "caar_host_traffic", "caar_upload_layout", "caar_download_layout", "caar_set_params_f90", "caar_set_vertical_coordinate", "caar_run_stepping",
    "caar_update_time_levels", "caar_extra_count", "caar_extra_upload", "caar_extra_download", "caar_euler_step",
    "caar_sync", "caar_launch_count", "caar_timer_start",
    "caar_timer_stop", "caar_norms", "caar_compute_and_apply_rhs_host", "caar_saxpby_device",
    "caar_saxpby_host", "caar_checksums", "caar_upload_range", "caar_download_range", "caar_describe",
    "caar_sphere_wk", "caar_run_rk5", "caar_advect_tracers",
)
CHECKSUM_FIELDS = ("elem_state_dp3d", "elem_state_v", "elem_state_T", "elem_derived_eta_dot_dpdn",
                   "elem_derived_omega_p", "elem_derived_phi", "elem_derived_vn0")


class CaarError(RuntimeError):
    pass


class Dims(C.Structure):
    _fields_ = [("nelem", C.c_int), ("nlev", C.c_int), ("np", C.c_int), ("qsize_d", C.c_int), ("ntl", C.c_int)]


class Arrays(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_double)) for n in FIELD_NAMES]


class Constants(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("rrearth", "eta_ave_w", "cp", "Rwater_vapor", "Rgas", "kappa")]


class Checksum(C.Structure):
    _fields_ = [("sum", C.c_double * 7), ("sumsq", C.c_double * 7), ("bits", C.c_ulonglong * 7),
                ("energy", C.c_double * 2)]


class Control(C.Structure):
    _fields_ = [("nets", C.c_int), ("nete", C.c_int), ("n0", C.c_int), ("np1", C.c_int), ("nm1", C.c_int),
                ("qn0", C.c_int), ("dt2", C.c_double)]


def field_shape(name, E, L, Q=1, ntl=3):
    """Host shapes of struct Arrays, PO/data_structures.cpp:14-31."""
    return {
        "elem_D": (E, 4, 4, 2, 2), "elem_Dinv": (E, 4, 4, 2, 2),
        "elem_fcor": (E, 4, 4), "elem_spheremp": (E, 4, 4), "elem_metdet": (E, 4, 4),
        "elem_rmetdet": (E, 4, 4), "elem_state_phis": (E, 4, 4),
        "elem_state_dp3d": (E, ntl, L, 4, 4), "elem_state_T": (E, ntl, L, 4, 4),
        "elem_state_v": (E, ntl, L, 4, 4, 2),
        "elem_state_Qdp": (E, Q, 2, L, 4, 4),
        "elem_derived_eta_dot_dpdn": (E, L + 1, 4, 4),
        "elem_derived_omega_p": (E, L, 4, 4), "elem_derived_phi": (E, L, 4, 4),
        "elem_derived_pecnd": (E, L, 4, 4), "elem_derived_vn0": (E, L, 4, 4, 2),
    }[name]


def lib_path():
    return os.path.join(HERE, "libcaar_b200.so")


_LIB = None


def load_library():
    """Loads libcaar_b200.so. Raises CaarError if it has not been built (python -m tinman_sandbox_b200.build)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise CaarError(f"{path} is missing: build it with `python -m tinman_sandbox_b200.build` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(path)
    lib.caar_last_error.restype = C.c_char_p
    lib.caar_version.restype = C.c_char_p
    lib.caar_field_count.restype = C.c_size_t
    lib.caar_field_count.argtypes = [C.POINTER(Dims), C.c_int]
    lib.caar_launch_count.restype = C.c_longlong
    lib.caar_launch_count.argtypes = [C.c_void_p]
    lib.caar_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(Dims), C.c_int]
    lib.caar_destroy.argtypes = [C.c_void_p]
    lib.caar_set_params.argtypes = [C.c_void_p, C.POINTER(Constants), C.POINTER(C.c_double), C.c_double,
                                    C.POINTER(C.c_double)]
    lib.caar_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.caar_upload.argtypes = [C.c_void_p, C.POINTER(Arrays), C.c_uint]
    lib.caar_download.argtypes = [C.c_void_p, C.POINTER(Arrays), C.c_uint]
    lib.caar_device_arrays.argtypes = [C.c_void_p, C.POINTER(Arrays)]
    lib.caar_host_register.argtypes = [C.c_void_p, C.c_size_t]
    lib.caar_host_unregister.argtypes = [C.c_void_p]
    lib.caar_run.argtypes = [C.c_void_p, C.POINTER(Control), C.c_int, C.c_int]
    lib.caar_run_host.argtypes = [C.c_void_p, C.POINTER(Arrays), C.POINTER(Control), C.c_int, C.c_int]
    lib.caar_host_traffic.argtypes = [C.c_void_p, C.POINTER(Control), C.c_int, C.POINTER(C.c_size_t),
                                      C.POINTER(C.c_size_t)]
    lib.caar_set_vertical_coordinate.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    lib.caar_run_stepping.argtypes = [C.c_void_p, C.POINTER(Control), C.c_int, C.c_int]
    lib.caar_run_rk5.argtypes = [C.c_void_p, C.POINTER(Control), C.c_double, C.c_int, C.c_int]
    lib.caar_update_time_levels.argtypes = [C.POINTER(Control)]
    lib.caar_update_time_levels.restype = None
    lib.caar_extra_count.restype = C.c_size_t
    lib.caar_extra_count.argtypes = [C.POINTER(Dims), C.c_int]
    lib.caar_extra_upload.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    lib.caar_extra_download.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    lib.caar_sphere_wk.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.caar_euler_step.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int]
    lib.caar_advect_tracers.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int, C.c_double, C.c_int,
                                        C.c_int]
    lib.caar_upload_layout.argtypes = [C.c_void_p, C.POINTER(Arrays), C.c_uint, C.c_int]
    lib.caar_download_layout.argtypes = [C.c_void_p, C.POINTER(Arrays), C.c_uint, C.c_int]
    lib.caar_set_params_f90.argtypes = [C.c_void_p, C.POINTER(Constants), C.POINTER(C.c_double), C.c_double,
                                        C.POINTER(C.c_double)]
    lib.caar_sync.argtypes = [C.c_void_p]
    lib.caar_timer_start.argtypes = [C.c_void_p]
    lib.caar_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    lib.caar_norms.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    lib.caar_describe.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_int)]
    lib.caar_checksums.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(Checksum)]
    lib.caar_upload_range.argtypes = [C.c_void_p, C.POINTER(Arrays), C.c_uint, C.c_int, C.c_int]
    lib.caar_download_range.argtypes = [C.c_void_p, C.POINTER(Arrays), C.c_uint, C.c_int, C.c_int]
    lib.caar_compute_and_apply_rhs_host.argtypes = [C.POINTER(Dims), C.POINTER(Arrays), C.POINTER(Control),
                                                    C.POINTER(Constants), C.POINTER(C.c_double), C.c_double,
                                                    C.POINTER(C.c_double), C.c_int, C.c_int]
    lib.caar_saxpby_device.argtypes = [C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.caar_saxpby_host.argtypes = [C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                     C.c_size_t, C.c_int, C.c_int]
    _LIB = lib
    return lib


def _check(lib, rc, what):
    if rc != 0:
        raise CaarError(f"{what} failed (code {rc}): {lib.caar_last_error().decode()}")


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _arrays_struct(arrays: dict, names=FIELD_NAMES, dims=None):
    st = Arrays()
    for n in names:
        a = arrays[n]
        if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"]:
            raise CaarError(f"{n}: need a C-contiguous float64 array")
        if dims is not None and a.size != int(np.prod(field_shape(n, *dims))):
            raise CaarError(f"{n}: has {a.size} values, dims need {int(np.prod(field_shape(n, *dims)))}")
        setattr(st, n, _dp(a))
    return st


def _mask(names):
    if names is None:
        return F_ALL
    m = 0
    for n in names:
        m |= FIELD_BIT[n]
    return m


class Caar:
    """One handle = the device-resident mirror of a TestData (PO/data_structures.hpp:78-89) for a slice of
    elements on one GPU. Method names follow the reference: ``compute_and_apply_rhs`` is
    Homme::compute_and_apply_rhs (PO/compute_and_apply_rhs.hpp:9), ``norms`` is print_results_2norm."""

    def __init__(self, nelem, nlev=72, qsize_d=1, ntl=3, device=0):
        self.lib = load_library()
        self.dims = Dims(nelem, nlev, 4, qsize_d, ntl)
        self.shape_args = (nelem, nlev, qsize_d, ntl)
        self.h = C.c_void_p()
        _check(self.lib, self.lib.caar_create(C.byref(self.h), C.byref(self.dims), device), "caar_create")
        self.control = Control(0, nelem, 0, 1, 2, 0, 1.0)

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.caar_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- TestData members -------------------------------------------------------------------------
    def set_params(self, consts, dvv, ps0, hyai):
        """consts = (rrearth, eta_ave_w, cp, Rwater_vapor, Rgas, kappa); dvv (4,4) row-major; hyai (nlev+1,)."""
        c = Constants(*[float(x) for x in consts])
        dvv = np.ascontiguousarray(dvv, dtype=np.float64).reshape(16)
        hyai = np.ascontiguousarray(hyai, dtype=np.float64)
        if hyai.size != self.dims.nlev + 1:
            raise CaarError("hyai needs nlev+1 entries")
        _check(self.lib, self.lib.caar_set_params(self.h, C.byref(c), _dp(dvv), float(ps0), _dp(hyai)),
               "caar_set_params")

    def set_vertical_coordinate(self, rsplit, hybi=None):
        """rsplit > 0: vertically Lagrangian (default); rsplit == 0: Eulerian, needs hybi (nlev+1,)
        (F/routine_extracted.F90:227-262)."""
        if hybi is not None:
            hybi = np.ascontiguousarray(hybi, dtype=np.float64)
            if hybi.size != self.dims.nlev + 1:
                raise CaarError("hybi needs nlev+1 entries")
        _check(self.lib, self.lib.caar_set_vertical_coordinate(self.h, int(rsplit), _dp(hybi) if hybi is not None else None),
               "caar_set_vertical_coordinate")

    def set_control(self, nets=None, nete=None, n0=None, np1=None, nm1=None, qn0=None, dt2=None):
        c = self.control
        for k, v in dict(nets=nets, nete=nete, n0=n0, np1=np1, nm1=nm1, qn0=qn0).items():
            if v is not None:
                setattr(c, k, int(v))
        if dt2 is not None:
            c.dt2 = float(dt2)

    def set_stream(self, cuda_stream_ptr):
        _check(self.lib, self.lib.caar_set_stream(self.h, C.c_void_p(cuda_stream_ptr)), "caar_set_stream")

    def upload(self, arrays: dict, names=None):
        names = FIELD_NAMES if names is None else names
        st = _arrays_struct(arrays, names, self.shape_args)
        _check(self.lib, self.lib.caar_upload(self.h, C.byref(st), _mask(names)), "caar_upload")

    def upload_f90(self, arrays: dict, names=None):
        """Upload arrays held in Fortran memory order (CAAR_LAYOUT_F90, see include/caar_b200.h); only the flat
        sizes are checked. `elem_rmetdet` may be absent: it is then computed on the device as 1/metdet."""
        names = FIELD_NAMES if names is None else names
        st = Arrays()
        for n in names:
            if n == "elem_rmetdet" and n not in arrays:
                continue
            a = arrays[n]
            if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"] or a.size != int(np.prod(field_shape(n, *self.shape_args))):
                raise CaarError(f"{n}: need a contiguous float64 array of the field's size")
            setattr(st, n, _dp(a))
        _check(self.lib, self.lib.caar_upload_layout(self.h, C.byref(st), _mask(names), LAYOUT_F90), "caar_upload_layout")

    def download_f90(self, arrays: dict, names=MUTATED_FIELDS):
        names = FIELD_NAMES if names is None else names
        st = Arrays()
        for n in names:
            a = arrays[n]
            if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"] or a.size != int(np.prod(field_shape(n, *self.shape_args))):
                raise CaarError(f"{n}: need a contiguous float64 array of the field's size")
            setattr(st, n, _dp(a))
        _check(self.lib, self.lib.caar_download_layout(self.h, C.byref(st), _mask(names), LAYOUT_F90), "caar_download_layout")

    def set_params_f90(self, consts, dvv_f90, ps0, hyai):
        c = Constants(*[float(x) for x in consts])
        dvv = np.ascontiguousarray(dvv_f90, dtype=np.float64).reshape(16)
        hyai = np.ascontiguousarray(hyai, dtype=np.float64)
        _check(self.lib, self.lib.caar_set_params_f90(self.h, C.byref(c), _dp(dvv), float(ps0), _dp(hyai)),
               "caar_set_params_f90")

    def download(self, arrays: dict, names=MUTATED_FIELDS):
        names = FIELD_NAMES if names is None else names
        st = _arrays_struct(arrays, names, self.shape_args)
        _check(self.lib, self.lib.caar_download(self.h, C.byref(st), _mask(names)), "caar_download")

    def _range_struct(self, arrays, names, e0, e1):
        E, L, Q, ntl = self.shape_args
        return _arrays_struct(arrays, names, (e1 - e0, L, Q, ntl))

    def upload_range(self, arrays: dict, e0, e1, names=None):
        """arrays hold ONLY elements [e0,e1) of each field (caar_upload_range)."""
        names = FIELD_NAMES if names is None else names
        st = self._range_struct(arrays, names, e0, e1)
        _check(self.lib, self.lib.caar_upload_range(self.h, C.byref(st), _mask(names), e0, e1), "caar_upload_range")

    def download_range(self, e0, e1, names=MUTATED_FIELDS, arrays=None):
        """-> dict of arrays holding elements [e0,e1) of the named fields (caar_download_range)."""
        names = FIELD_NAMES if names is None else names
        E, L, Q, ntl = self.shape_args
        if arrays is None:
            arrays = {n: np.empty(field_shape(n, e1 - e0, L, Q, ntl)) for n in names}
        st = self._range_struct(arrays, names, e0, e1)
        _check(self.lib, self.lib.caar_download_range(self.h, C.byref(st), _mask(names), e0, e1), "caar_download_range")
        return arrays

    def checksums(self, tl=None, nets=None, nete=None):
        """caar_checksums -> dict(sum, sumsq: float64[7]; bits: uint64[7]; energy: float64[2]); field order
        CHECKSUM_FIELDS. All-reduce sum/sumsq/energy with SUM and bits as 64-bit integers with SUM."""
        out = Checksum()
        tl = self.control.np1 if tl is None else tl
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        _check(self.lib, self.lib.caar_checksums(self.h, tl, nets, nete, C.byref(out)), "caar_checksums")
        return {"sum": np.array(out.sum[:]), "sumsq": np.array(out.sumsq[:]),
                "bits": np.array(out.bits[:], dtype=np.uint64), "energy": np.array(out.energy[:])}

    def describe(self, mode=MODE_FAST):
        """-> (text, is_fused): which kernel compute_and_apply_rhs launches in `mode` (caar_describe)."""
        buf, flag = C.create_string_buffer(256), C.c_int()
        _check(self.lib, self.lib.caar_describe(self.h, mode, buf, 256, C.byref(flag)), "caar_describe")
        return buf.value.decode(), bool(flag.value)

    def device_pointers(self):
        st = Arrays()
        _check(self.lib, self.lib.caar_device_arrays(self.h, C.byref(st)), "caar_device_arrays")
        return {n: C.cast(getattr(st, n), C.c_void_p).value for n in FIELD_NAMES}

    # -- the hot path -------------------------------------------------------------------------------
    def compute_and_apply_rhs(self, nsteps=1, mode=MODE_FAST, sync=True):
        _check(self.lib, self.lib.caar_run(self.h, C.byref(self.control), nsteps, mode), "caar_run")
        if sync:
            self.sync()

    def run_stepping(self, nsteps, mode=MODE_FAST, sync=True):
        """nsteps evaluations with TestData::update_time_levels (PO/data_structures.cpp:174-180) after each;
        self.control holds the rotated time levels afterwards."""
        _check(self.lib, self.lib.caar_run_stepping(self.h, C.byref(self.control), nsteps, mode), "caar_run_stepping")
        if sync:
            self.sync()

    def run_rk5(self, nsteps, dt, mode=MODE_FAST, sync=True):
        """nsteps steps of HOMME's five-stage Runge-Kutta dynamics step (tstep_type 5, caar_run_rk5) of length dt;
        self.control holds the rotated time levels afterwards and its dt2 is not used."""
        _check(self.lib, self.lib.caar_run_rk5(self.h, C.byref(self.control), float(dt), int(nsteps), mode),
               "caar_run_rk5")
        if sync:
            self.sync()

    # -- the step after CAAR: tracer advection RHS (LV/EulerStepFunctor.hpp:33-66) ------------------------
    def upload_vstar(self, vstar):
        E, L, Q, _ = self.shape_args
        if vstar.dtype != np.float64 or not vstar.flags["C_CONTIGUOUS"] or vstar.size != E * L * 32:
            raise CaarError("vstar: need a C-contiguous float64 array [E][L][4][4][2]")
        _check(self.lib, self.lib.caar_extra_upload(self.h, X_VSTAR, _dp(vstar)), "caar_extra_upload")

    def euler_step(self, qn0, qsize, dt, mode=MODE_FAST, nets=None, nete=None, sync=True):
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        _check(self.lib, self.lib.caar_euler_step(self.h, nets, nete, int(qn0), int(qsize), float(dt), mode),
               "caar_euler_step")
        if sync:
            self.sync()

    def advect_tracers(self, qn0, qsize, dt, nsteps=1, mode=MODE_FAST, nets=None, nete=None, sync=True):
        """nsteps steps of HOMME's three-stage tracer step (rkstage = 3, caar_advect_tracers) of length dt on the
        resident Qdp, starting from time level qn0 (0 or 1) -> the qn0 of the new state."""
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        q = C.c_int(int(qn0))
        _check(self.lib, self.lib.caar_advect_tracers(self.h, nets, nete, C.byref(q), int(qsize), float(dt),
                                                      int(nsteps), mode), "caar_advect_tracers")
        if sync:
            self.sync()
        return q.value

    def download_qtens(self, qtens=None):
        E, L, Q, _ = self.shape_args
        if qtens is None:
            qtens = np.zeros((E, Q, L, 4, 4))
        if qtens.dtype != np.float64 or not qtens.flags["C_CONTIGUOUS"] or qtens.size != E * Q * L * 16:
            raise CaarError("qtens: need a C-contiguous float64 array [E][qsize_d][L][4][4]")
        _check(self.lib, self.lib.caar_extra_download(self.h, X_QTENS, _dp(qtens)), "caar_extra_download")
        return qtens

    # -- the weak-form operators behind hyperviscosity (LV/SphereOperators.hpp:493-636) ---------------------
    def upload_extra(self, which, a):
        n = int(self.lib.caar_extra_count(C.byref(self.dims), which))
        if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"] or a.size != n:
            raise CaarError(f"extra array {which}: need a C-contiguous float64 array of {n} values")
        _check(self.lib, self.lib.caar_extra_upload(self.h, which, _dp(a)), "caar_extra_upload")

    def download_extra(self, which, shape):
        a = np.zeros(shape)
        if a.size != int(self.lib.caar_extra_count(C.byref(self.dims), which)):
            raise CaarError(f"extra array {which}: wrong shape {shape}")
        _check(self.lib, self.lib.caar_extra_download(self.h, which, _dp(a)), "caar_extra_download")
        return a

    def sphere_wk(self, op, mode=MODE_FAST, nets=None, nete=None, sync=True):
        """caar_sphere_wk: OP_DIVERGENCE_WK (of X_VSTAR), OP_LAPLACE_SIMPLE / OP_LAPLACE_TENSOR (of X_SCALAR_IN),
        OP_LAPLACE_TENSOR_REPLACE (X_SCALAR_OUT in place) -> X_SCALAR_OUT."""
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        _check(self.lib, self.lib.caar_sphere_wk(self.h, int(op), nets, nete, mode), "caar_sphere_wk")
        if sync:
            self.sync()

    def compute_and_apply_rhs_host(self, arrays: dict, mode=MODE_FAST, chunk_elems=0):
        """Homme::compute_and_apply_rhs(TestData&) on HOST arrays (PO/main.cpp:113-121 calls it this way):
        inputs are read from `arrays`, results are in `arrays` on return; copy-in, kernel and copy-out are
        pipelined over element chunks (caar_run_host)."""
        st = _arrays_struct(arrays, FIELD_NAMES, self.shape_args)
        _check(self.lib, self.lib.caar_run_host(self.h, C.byref(st), C.byref(self.control), mode, chunk_elems),
               "caar_run_host")

    def host_traffic(self, mode=MODE_FAST):
        """(h2d_bytes, d2h_bytes) one compute_and_apply_rhs_host call moves with the current control."""
        a, b = C.c_size_t(), C.c_size_t()
        _check(self.lib, self.lib.caar_host_traffic(self.h, C.byref(self.control), mode, C.byref(a), C.byref(b)),
               "caar_host_traffic")
        return int(a.value), int(b.value)

    def sync(self):
        _check(self.lib, self.lib.caar_sync(self.h), "caar_sync")

    def timer_start(self):
        _check(self.lib, self.lib.caar_timer_start(self.h), "caar_timer_start")

    def timer_stop(self) -> float:
        ms = C.c_float()
        _check(self.lib, self.lib.caar_timer_stop(self.h, C.byref(ms)), "caar_timer_stop")
        return ms.value

    def launch_count(self) -> int:
        return int(self.lib.caar_launch_count(self.h))

    def sumsq(self, tl=None, nets=None, nete=None):
        """Sums of squares of (v, T, dp3d) at time level tl over [nets,nete) — all-reduce these across
        ranks, then sqrt, to get the reference's printed norms."""
        out = np.zeros(3)
        tl = self.control.np1 if tl is None else tl
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        _check(self.lib, self.lib.caar_norms(self.h, tl, nets, nete, _dp(out)), "caar_norms")
        return out

    def norms(self, tl=None):
        return np.sqrt(self.sumsq(tl))


def compute_and_apply_rhs(state, mode=MODE_FAST, device=0):
    """Reference-facing one-shot on HOST arrays: the meaning of Homme::compute_and_apply_rhs(TestData&).
    `state` is anything with .nelem .nlev .qsize_d .ntl .arrays .ctl .dt2 .consts .dvv .ps0 .hyai
    (e.g. oracle.harness.State). Mutates state.arrays in place, like the reference."""
    lib = load_library()
    dims = Dims(state.nelem, state.nlev, 4, state.qsize_d, state.ntl)
    st = _arrays_struct(state.arrays, FIELD_NAMES, (state.nelem, state.nlev, state.qsize_d, state.ntl))
    ctl = Control(*[int(x) for x in state.ctl], float(state.dt2))
    c = Constants(*[float(x) for x in state.consts])
    dvv = np.ascontiguousarray(state.dvv, dtype=np.float64).reshape(16)
    hyai = np.ascontiguousarray(state.hyai, dtype=np.float64)
    rc = lib.caar_compute_and_apply_rhs_host(C.byref(dims), C.byref(st), C.byref(ctl), C.byref(c), _dp(dvv),
                                             float(state.ps0), _dp(hyai), device, mode)
    _check(lib, rc, "caar_compute_and_apply_rhs_host")


HOST_ZERO_COPY = -1  # chunk_elems value selecting the zero-copy path of caar_run_host


def host_register(arrays: dict):
    """Page-locks and device-maps caller-owned numpy arrays in place (caar_host_register)."""
    lib = load_library()
    for n, a in arrays.items():
        _check(lib, lib.caar_host_register(C.c_void_p(a.ctypes.data), a.nbytes), f"caar_host_register({n})")


def host_unregister(arrays: dict):
    lib = load_library()
    for n, a in arrays.items():
        _check(lib, lib.caar_host_unregister(C.c_void_p(a.ctypes.data)), f"caar_host_unregister({n})")


def saxpby_host(a, b, x, y, sweeps=1, device=0):
    lib = load_library()
    if x.dtype != np.float64 or y.dtype != np.float64 or x.size != y.size:
        raise CaarError("saxpby: x and y must be float64 of equal size")
    _check(lib, lib.caar_saxpby_host(float(a), float(b), _dp(x), _dp(y), x.size, sweeps, device),
           "caar_saxpby_host")
