"""ctypes binding of libblmm_b200.so — the same C-ABI (include/blmm_b200.h) the Julia shim
`ccall`s.  There is no fallback: if the library is missing or no B200 is present the calls raise."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# BLMM_B200_LIB (the variable the Julia shim reads too) points at another build of the same library
LIB_PATH = os.environ.get("BLMM_B200_LIB") or os.path.join(HERE, "lib", "libblmm_b200.so")

# status codes / enums of include/blmm_b200.h
OK, E_INVALID, E_DIM, E_H2_ONE, E_ZERO_NORM, E_ONE_TRAIT, E_CUDA, E_NOT_SPD, E_NO_DEVICE, E_WEIGHTS = range(10)
MEM_HOST, MEM_DEVICE = 0, 1
METHOD_NULL_GRID, METHOD_ALT_GRID, METHOD_NULL_EXACT = 0, 1, 2
H2PANEL_REFERENCE, H2PANEL_ARGMAX = 0, 1
DECOMP_EIGEN, DECOMP_SVD = 0, 1
ABI_VERSION = 3

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)


class Problem(C.Structure):
    _fields_ = [("n", C.c_int64), ("p", C.c_int64), ("m", C.c_int64), ("c", C.c_int64),
                ("Y", C.c_void_p), ("G", C.c_void_p), ("Covar", C.c_void_p), ("U", C.c_void_p),
                ("lam", C.c_void_p), ("obs_weights", C.c_void_p)]


class Opts(C.Structure):
    _fields_ = [("method", C.c_int32), ("reml", C.c_int32), ("prior_variance", C.c_double),
                ("prior_sample_size", C.c_double), ("h2_grid", c_double_p), ("ngrid", C.c_int32),
                ("optim_interval", C.c_int32), ("h2_panel_mode", C.c_int32), ("mem_space", C.c_int32),
                ("ld_out", C.c_int64), ("chisq_df", C.c_int32), ("reserved", C.c_int32),
                ("log10p_out", C.c_void_p)]


# every symbol include/blmm_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "blmm_abi_version": (C.c_int, []),
    "blmm_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "blmm_create_multi": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int]),
    "blmm_device_count": (C.c_int, [C.c_void_p]),
    "blmm_destroy": (None, [C.c_void_p]),
    "blmm_last_error": (C.c_char_p, [C.c_void_p]),
    "blmm_sync": (C.c_int, [C.c_void_p]),
    "blmm_stream": (C.c_uint64, [C.c_void_p]),
    "blmm_launch_count": (C.c_int64, [C.c_void_p]),
    "blmm_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "blmm_last_scan_ms": (C.c_double, [C.c_void_p]),
    "blmm_last_gather_ms": (C.c_double, [C.c_void_p]),
    "blmm_host_write_gbs": (C.c_double, [C.c_int, C.c_int64]),
    "blmm_kinship": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int]),
    "blmm_decompose": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                 C.POINTER(C.c_int), C.c_int]),
    "blmm_rotate": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.c_void_p, C.c_void_p, C.c_int]),
    "blmm_bulkscan": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Opts), C.c_void_p, C.c_void_p]),
    "blmm_bulkscan_peaks": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Opts), C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "blmm_grid_loglik": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Opts), C.c_void_p]),
    "blmm_fit_h2": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Opts), C.c_void_p, C.c_void_p,
                              C.c_void_p]),
    "blmm_scan_perms": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Opts), C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "blmm_scan_null": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Opts), C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "blmm_scan_alt": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Opts), C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
    "blmm_lod2log10p": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                  C.c_void_p, C.c_int]),
    "blmm_thresholds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "blmm_read_csv": (C.c_int, [C.c_char_p, C.c_char, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_void_p)]),
    "blmm_free_matrix": (None, [C.c_void_p, C.c_int]),
    "blmm_io_last_error": (C.c_char_p, []),
    "blmm_weight_kinship": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library and declare every entry point (fails loudly if it is not built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python bulklmm.jl_b200/build.py` "
            "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.blmm_abi_version() != ABI_VERSION:
        raise RuntimeError("libblmm_b200.so ABI version mismatch")
    _lib = lib
    return lib
