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
DSS_ASSEMBLE, DSS_PROJECT = 0, 1
DSS_FIELDS = ("elem_state_dp3d", "elem_state_v", "elem_state_T", "elem_state_Qdp")   # what caar_dss can select
HALO_DSS, HALO_MINMAX = 0, 1

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
    "caar_sphere_wk", "caar_run_rk5", "caar_advect_tracers", "caar_bounds_upload", "caar_bounds_download",
    "caar_tracer_bounds", "caar_limit_tracers", "caar_set_connectivity", "caar_dss", "caar_neighbor_minmax",
    "caar_run_rk5_dss", "caar_set_partition", "caar_dss_pack", "caar_dss_unpack", "caar_neighbor_minmax_pack",
    "caar_neighbor_minmax_unpack", "caar_halo_segments", "caar_rk5_stage", "caar_dss_interior", "caar_dss_boundary",
    "caar_vertical_remap",
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
    lib.caar_rk5_stage.argtypes = [C.c_void_p, C.POINTER(Control), C.c_double, C.c_int, C.c_int, C.POINTER(C.c_int)]
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
    lib.caar_bounds_upload.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    lib.caar_bounds_download.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    lib.caar_tracer_bounds.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.caar_limit_tracers.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.caar_vertical_remap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.caar_set_connectivity.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.c_int]
    lib.caar_dss.argtypes = [C.c_void_p, C.c_uint, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.caar_neighbor_minmax.argtypes = [C.c_void_p, C.c_int]
    lib.caar_run_rk5_dss.argtypes = [C.c_void_p, C.POINTER(Control), C.c_double, C.c_int, C.c_int]
    lib.caar_set_partition.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.c_int, C.POINTER(C.c_int), C.c_int,
                                       C.c_int, C.c_int]
    lib.caar_dss_pack.argtypes = lib.caar_dss.argtypes
    lib.caar_dss_unpack.argtypes = lib.caar_dss.argtypes
    lib.caar_dss_interior.argtypes = lib.caar_dss.argtypes
    lib.caar_dss_boundary.argtypes = lib.caar_dss.argtypes
    lib.caar_neighbor_minmax_pack.argtypes = [C.c_void_p, C.c_int]
    lib.caar_neighbor_minmax_unpack.argtypes = [C.c_void_p, C.c_int]
    lib.caar_halo_segments.argtypes = [C.c_void_p, C.c_int, C.c_uint, C.c_int, C.POINTER(C.c_void_p),
                                       C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
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
        self.device = device

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

    def rk5_stage(self, stage, dt, mode=MODE_FAST, sync=True):
        """Stage `stage` (0..4) of run_rk5's step on self.control's levels (caar_rk5_stage) -> the level it wrote, which
        a DSS after the stage assembles; self.control is not rotated (update_time_levels after stage 4)."""
        tl = C.c_int(-1)
        _check(self.lib, self.lib.caar_rk5_stage(self.h, C.byref(self.control), float(dt), int(stage), mode,
                                                 C.byref(tl)), "caar_rk5_stage")
        if sync:
            self.sync()
        return tl.value

    def update_time_levels(self):
        """caar_update_time_levels on self.control."""
        self.lib.caar_update_time_levels(C.byref(self.control))

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

    # -- the tracer limiter (limiter_option 8): element-local bounds and limiter_optim_iter_full --------------------
    def upload_bounds(self, bounds):
        """bounds [E][qsize_d][L][2] = (qmin, qmax): the whole handle-owned array (caar_bounds_upload)."""
        E, L, Q, _ = self.shape_args
        if bounds.dtype != np.float64 or not bounds.flags["C_CONTIGUOUS"] or bounds.size != E * Q * L * 2:
            raise CaarError("bounds: need a C-contiguous float64 array [E][qsize_d][L][2]")
        _check(self.lib, self.lib.caar_bounds_upload(self.h, _dp(bounds)), "caar_bounds_upload")

    def download_bounds(self, bounds=None):
        E, L, Q, _ = self.shape_args
        if bounds is None:
            bounds = np.zeros((E, Q, L, 2))
        if bounds.dtype != np.float64 or not bounds.flags["C_CONTIGUOUS"] or bounds.size != E * Q * L * 2:
            raise CaarError("bounds: need a C-contiguous float64 array [E][qsize_d][L][2]")
        _check(self.lib, self.lib.caar_bounds_download(self.h, _dp(bounds)), "caar_bounds_download")
        return bounds

    def tracer_bounds(self, qtl, qsize, dp_tl, nets=None, nete=None, sync=True):
        """caar_tracer_bounds: bounds of Qdp(qtl)/dp3d(dp_tl) per element, tracer iq < qsize and level, qmin >= 0."""
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        _check(self.lib, self.lib.caar_tracer_bounds(self.h, nets, nete, int(qtl), int(qsize), int(dp_tl)),
               "caar_tracer_bounds")
        if sync:
            self.sync()

    def limit_tracers(self, qtl, qsize, dp_tl, nets=None, nete=None, sync=True):
        """caar_limit_tracers: HOMME's limiter_optim_iter_full on Qdp(qtl) with weights spheremp * dp3d(dp_tl), within
        the handle's bounds (relaxed bounds are written back)."""
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        _check(self.lib, self.lib.caar_limit_tracers(self.h, nets, nete, int(qtl), int(qsize), int(dp_tl)),
               "caar_limit_tracers")
        if sync:
            self.sync()

    # -- the vertical remap (rsplit > 0) -----------------------------------------------------------------------------
    def vertical_remap(self, tl=None, qtl=0, qsize=0, nets=None, nete=None, sync=True):
        """caar_vertical_remap: HOMME's PPM remap of T, v at time level tl (default control.np1) and Qdp(qtl) of tracers
        iq < qsize from dp3d(tl) to the reference levels of hyai (set_params) and hybi (set_vertical_coordinate), then
        dp3d(tl) = dp."""
        tl = self.control.np1 if tl is None else tl
        nets = self.control.nets if nets is None else nets
        nete = self.control.nete if nete is None else nete
        _check(self.lib, self.lib.caar_vertical_remap(self.h, int(nets), int(nete), int(tl), int(qtl), int(qsize)),
               "caar_vertical_remap")
        if sync:
            self.sync()

    # -- the direct stiffness summation over shared element-boundary points -------------------------------------------
    def set_connectivity(self, gid, layout=LAYOUT_CXX):
        """caar_set_connectivity: gid [E][4][4] int64, the global id of every GLL point ([igp][jgp] with LAYOUT_CXX, the
        memory order of HOMME's gdofP(np,np,nelemd) with LAYOUT_F90)."""
        E = self.shape_args[0]
        gid = np.ascontiguousarray(gid, dtype=np.int64)
        if gid.size != E * 16:
            raise CaarError(f"gid: need {E * 16} ids, got {gid.size}")
        _check(self.lib, self.lib.caar_set_connectivity(self.h, gid.ctypes.data_as(C.POINTER(C.c_longlong)), int(layout)),
               "caar_set_connectivity")

    def dss(self, names, tl=None, qtl=0, qsize=0, weighting=DSS_ASSEMBLE, sync=True):
        """caar_dss in place on the named fields of DSS_FIELDS: dp3d, v, T at time level tl (default control.np1) and
        Qdp(qtl) of tracers < qsize."""
        tl = self.control.np1 if tl is None else tl
        for n in names:
            if n not in DSS_FIELDS:
                raise CaarError(f"{n}: caar_dss assembles only {DSS_FIELDS}")
        _check(self.lib, self.lib.caar_dss(self.h, _mask(names) if names else 0, int(tl), int(qtl), int(qsize),
                                           int(weighting)), "caar_dss")
        if sync:
            self.sync()

    def neighbor_minmax(self, qsize, sync=True):
        """caar_neighbor_minmax: widen the handle's limiter bounds of tracers < qsize over neighbouring elements."""
        _check(self.lib, self.lib.caar_neighbor_minmax(self.h, int(qsize)), "caar_neighbor_minmax")
        if sync:
            self.sync()

    def run_rk5_dss(self, nsteps, dt, mode=MODE_FAST, sync=True):
        """run_rk5 with caar_dss of v, T and dp3d after every stage (caar_run_rk5_dss); needs set_connectivity and the
        control's range [0, nelem)."""
        _check(self.lib, self.lib.caar_run_rk5_dss(self.h, C.byref(self.control), float(dt), int(nsteps), mode),
               "caar_run_rk5_dss")
        if sync:
            self.sync()

    # -- the DSS and neighbor_minmax across partitioned handles --------------------------------------------------------
    def set_partition(self, gid, part_start, part, layout=LAYOUT_CXX):
        """caar_set_partition: gid [nelem_global][4][4] int64 of the whole mesh; this handle holds the elements
        [part_start[part], part_start[part + 1])."""
        gid = np.ascontiguousarray(gid, dtype=np.int64)
        ps = np.ascontiguousarray(part_start, dtype=np.int32)
        if gid.size % 16:
            raise CaarError(f"gid: need 16 ids per element, got {gid.size}")
        _check(self.lib, self.lib.caar_set_partition(self.h, gid.ctypes.data_as(C.POINTER(C.c_longlong)), gid.size // 16,
                                                     ps.ctypes.data_as(C.POINTER(C.c_int)), len(ps) - 1, int(part),
                                                     int(layout)), "caar_set_partition")
        self.nparts = len(ps) - 1

    def _dss_call(self, fn, what, names, tl, qtl, qsize, weighting, sync):
        tl = self.control.np1 if tl is None else tl
        for n in names:
            if n not in DSS_FIELDS:
                raise CaarError(f"{n}: {what} selects only {DSS_FIELDS}")
        _check(self.lib, fn(self.h, _mask(names) if names else 0, int(tl), int(qtl), int(qsize), int(weighting)), what)
        if sync:
            self.sync()

    def dss_pack(self, names, tl=None, qtl=0, qsize=0, weighting=DSS_ASSEMBLE, sync=True):
        """caar_dss_pack: the records of the named fields for every other part into the send buffer."""
        self._dss_call(self.lib.caar_dss_pack, "caar_dss_pack", names, tl, qtl, qsize, weighting, sync)

    def dss_unpack(self, names, tl=None, qtl=0, qsize=0, weighting=DSS_ASSEMBLE, sync=True):
        """caar_dss_unpack: the whole DSS of the handle in place, remote copies from the receive buffer."""
        self._dss_call(self.lib.caar_dss_unpack, "caar_dss_unpack", names, tl, qtl, qsize, weighting, sync)

    def dss_interior(self, names, tl=None, qtl=0, qsize=0, weighting=DSS_ASSEMBLE, sync=True):
        """caar_dss_interior: the points whose copies are all on this handle; reads neither exchange buffer."""
        self._dss_call(self.lib.caar_dss_interior, "caar_dss_interior", names, tl, qtl, qsize, weighting, sync)

    def dss_boundary(self, names, tl=None, qtl=0, qsize=0, weighting=DSS_ASSEMBLE, sync=True):
        """caar_dss_boundary: the points with a copy on another part, remote copies from the receive buffer."""
        self._dss_call(self.lib.caar_dss_boundary, "caar_dss_boundary", names, tl, qtl, qsize, weighting, sync)

    def neighbor_minmax_pack(self, qsize, sync=True):
        _check(self.lib, self.lib.caar_neighbor_minmax_pack(self.h, int(qsize)), "caar_neighbor_minmax_pack")
        if sync:
            self.sync()

    def neighbor_minmax_unpack(self, qsize, sync=True):
        _check(self.lib, self.lib.caar_neighbor_minmax_unpack(self.h, int(qsize)), "caar_neighbor_minmax_unpack")
        if sync:
            self.sync()

    def halo_segments(self, op, names=(), qsize=0):
        """caar_halo_segments -> (send, recv, send_off, recv_off): torch float64 CUDA tensors viewing the handle's
        two exchange buffers (valid until the handle is closed or its map replaced) and the segment offsets in doubles,
        numpy int64 [nparts + 1] each; segment q is send[send_off[q]:send_off[q + 1]]."""
        import torch
        n = self.nparts + 1
        sp, rp = C.c_void_p(), C.c_void_p()
        so, ro = (C.c_size_t * n)(), (C.c_size_t * n)()
        _check(self.lib, self.lib.caar_halo_segments(self.h, int(op), _mask(names) if names else 0, int(qsize),
                                                     C.byref(sp), C.byref(rp), so, ro), "caar_halo_segments")
        so, ro = np.array(so[:], dtype=np.int64), np.array(ro[:], dtype=np.int64)
        dev = torch.device("cuda", self.device)
        return _device_view(sp.value, int(so[-1]), dev), _device_view(rp.value, int(ro[-1]), dev), so, ro

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


class _CudaArray:
    """__cuda_array_interface__ of n float64 at a device pointer, for torch.as_tensor"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3,
                                         "strides": None}


def _device_view(ptr, n, device):
    import torch
    if n == 0:
        return torch.empty(0, dtype=torch.float64, device=device)
    return torch.as_tensor(_CudaArray(ptr, n), device=device)


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
