"""tinman_sandbox_b200 — B200-native compute_and_apply_rhs (HOMME "CAAR" as extracted in
E3SM-Project/tinman_sandbox) behind a C-ABI shared library of hand-written sm_100a CUDA kernels.

Layout of the package (only what the hot path needs):

  csrc/            CUDA kernels + the C-ABI (include/caar_b200.h)      -> libcaar_b200.so
  host/            C++ host side: Homme::compute_and_apply_rhs(TestData&) shim + driver
  capi.py          ctypes binding of the C-ABI (used by tests/, bench.py, smoke())
  build.py         nvcc build of everything above (sm_100a only)

There is no CPU fallback anywhere in this package: importing works without a GPU (so the C-ABI can be
loaded and its symbols checked), but every compute call fails loudly without a CUDA device or without
the built extension.
"""
from .capi import (  # noqa: F401
    Caar, CaarError, FIELD_NAMES, MUTATED_FIELDS, MODE_FAST, MODE_STRICT, lib_path, load_library,
    field_shape, compute_and_apply_rhs, saxpby_host, EXPORTED_SYMBOLS, HOST_ZERO_COPY, host_register,
    host_unregister, CHECKSUM_FIELDS, X_VSTAR, X_QTENS, X_TENSORVISC, X_SCALAR_IN, X_SCALAR_OUT, OP_DIVERGENCE_WK,
    OP_LAPLACE_SIMPLE, OP_LAPLACE_TENSOR, OP_LAPLACE_TENSOR_REPLACE, DSS_ASSEMBLE, DSS_PROJECT, DSS_FIELDS,
    HALO_DSS, HALO_MINMAX,
)

__all__ = [
    "Caar", "CaarError", "FIELD_NAMES", "MUTATED_FIELDS", "MODE_FAST", "MODE_STRICT", "lib_path",
    "load_library", "field_shape", "compute_and_apply_rhs", "saxpby_host", "EXPORTED_SYMBOLS",
    "HOST_ZERO_COPY", "host_register", "host_unregister", "CHECKSUM_FIELDS",
]
