"""ctypes binding of libspart_b200.so (C ABI declared in include/spart_b200.h).

There is deliberately no fallback: if the shared library has not been built, or there is no
CUDA device, every compute entry point raises.  Build with `python __graft_entry__.py build`
(or `python spart-python_b200/build.py`).
"""
import ctypes
from ctypes import POINTER, Structure, byref, c_char_p, c_double, c_int32, c_int64, c_size_t, c_uint32, c_uint64, c_void_p
from pathlib import Path

import os

# SPART_B200_LIB lets kernel-tuning scripts load an alternative build of the same library
LIB_PATH = Path(os.environ.get("SPART_B200_LIB") or Path(__file__).resolve().parent / "lib" / "libspart_b200.so")
ABI_VERSION = 5
FLAG_SOIL_SPECTRUM = 2
FLAG_SRF_BANDS = 4
FLAG_REUSE_RECORD = 8
FLAG_F32_IO = 16
FLAG_COMPACT_OUT = 32
FLAG_USER_LIDF = 64
FLAG_SOIL_LIBRARY = 128
NKERNELS = 3
NPAR = 27
# rows 19..21 (sun zenith, observer zenith, relative azimuth) as broadcast rows = one geometry for
# the whole batch by construction; the library then folds it once per thread block
GEOMETRY_ROWS = (1 << 19) | (1 << 20) | (1 << 21)

FP64 = 64
FP32 = 32

EXPORTS = (
    "spart_abi_version", "spart_last_error", "spart_device_count", "spart_create", "spart_create_with_soils",
    "spart_destroy",
    "spart_workspace_bytes", "spart_forward_bands", "spart_forward_bands_bc", "spart_forward_bands_host", "spart_forward_spectrum",
    "spart_smac", "spart_sailh", "spart_lut_workspace_bytes", "spart_lut_nearest", "spart_lut_nearest_tc", "spart_lut_unpack",
    "spart_lut_topk_workspace_bytes", "spart_lut_topk", "spart_lut_topk_merge", "spart_lut_moments_accumulate",
    "spart_lut_moments_finish", "spart_sobol_design", "spart_sobol_acc_elems", "spart_sobol_accumulate",
    "spart_sobol_finish", "spart_invert_state_rows", "spart_invert_design", "spart_invert_step", "spart_invert_finish",
    "spart_leafangles", "spart_set_lidf", "spart_profile_enable", "spart_profile_read", "spart_measure_peaks", "spart_measure_fp64_chain", "spart_launch_count",
)


class SpartError(RuntimeError):
    """Raised for every non-zero return of the C ABI (and for a missing library)."""


class SpartTables(Structure):
    _fields_ = [("n_wl", c_int32), ("lc", POINTER(c_double))]


class SpartSensor(Structure):
    _fields_ = [
        ("n_bands", c_int32),
        ("wl_lo", POINTER(c_int32)),
        ("wl_hi", POINTER(c_int32)),
        ("wl_frac", POINTER(c_double)),
        ("smac", POINTER(c_double)),
        ("conv_ea", POINTER(c_double)),
        ("srf_len", POINTER(c_int32)),
        ("srf_idx", POINTER(c_int32)),
        ("srf_w", POINTER(c_double)),
    ]


_lib = None


def load():
    """Load (once) and type the shared library."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise SpartError(
            f"{LIB_PATH} is missing: the CUDA library has not been built "
            "(run `python __graft_entry__.py build`); spart_b200 has no CPU fallback")
    lib = ctypes.CDLL(str(LIB_PATH))
    lib.spart_abi_version.restype = ctypes.c_int
    lib.spart_last_error.restype = c_char_p
    lib.spart_device_count.restype = ctypes.c_int
    lib.spart_create.argtypes = [POINTER(SpartTables), POINTER(SpartSensor), c_int32, c_int32, POINTER(c_void_p)]
    lib.spart_create_with_soils.argtypes = [POINTER(SpartTables), POINTER(SpartSensor), c_int32, POINTER(c_double),
                                            c_int32, c_int32, POINTER(c_void_p)]
    lib.spart_destroy.argtypes = [c_void_p]
    lib.spart_workspace_bytes.argtypes = [c_void_p, c_int64]
    lib.spart_workspace_bytes.restype = c_size_t
    lib.spart_forward_bands.argtypes = [c_void_p, c_int32, c_void_p, c_int64, c_int64, c_uint32, c_int32, c_int32,
                                        c_void_p, c_void_p, c_void_p]
    lib.spart_forward_bands_bc.argtypes = [c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_int64, c_uint32, c_int32,
                                           c_int32, c_void_p, c_void_p, c_void_p]
    lib.spart_forward_bands_host.argtypes = [c_void_p, c_int32, c_void_p, c_int64, c_int64, c_uint32, c_int32,
                                             c_int32, c_void_p]
    lib.spart_forward_spectrum.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_int32, c_double, c_double,
                                           c_void_p, c_void_p, c_void_p]
    lib.spart_smac.argtypes = [c_void_p, c_int32, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]
    lib.spart_sailh.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                c_void_p, c_void_p]
    lib.spart_lut_workspace_bytes.argtypes = [c_int64]
    lib.spart_lut_workspace_bytes.restype = c_size_t
    lib.spart_lut_nearest.argtypes = [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_void_p]
    lib.spart_lut_nearest_tc.argtypes = lib.spart_lut_nearest.argtypes
    lib.spart_lut_unpack.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]
    lib.spart_lut_topk_workspace_bytes.argtypes = [c_int64, c_int64, c_int32]
    lib.spart_lut_topk_workspace_bytes.restype = c_size_t
    lib.spart_lut_topk.argtypes = [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32, c_void_p, c_int64, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p]
    lib.spart_lut_topk_merge.argtypes = [c_void_p, c_int64, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.spart_lut_moments_accumulate.argtypes = [c_void_p, c_int32, c_int64, c_int64, c_int32, c_int64, c_int64,
                                                 c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p]
    lib.spart_lut_moments_finish.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p,
                                             c_void_p]
    lib.spart_sobol_design.argtypes = [POINTER(c_int32), POINTER(c_double), POINTER(c_double), c_int32, c_uint64,
                                       c_int32, c_int64, c_int64, c_int32, c_void_p, c_int64, c_void_p]
    lib.spart_sobol_acc_elems.argtypes = [c_int32, c_int32]
    lib.spart_sobol_acc_elems.restype = c_size_t
    lib.spart_sobol_accumulate.argtypes = [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]
    lib.spart_sobol_finish.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_int32] + [c_void_p] * 7
    lib.spart_invert_state_rows.argtypes = [c_int32]
    lib.spart_invert_state_rows.restype = c_size_t
    lib.spart_invert_design.argtypes = [POINTER(c_int32), POINTER(c_double), POINTER(c_double), c_int32,
                                        POINTER(c_int32), c_int32, c_void_p, c_int64, POINTER(c_double), c_int32,
                                        c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p]
    lib.spart_invert_step.argtypes = [POINTER(c_double), POINTER(c_double), c_int32, c_int32, c_void_p, c_int32,
                                      c_int32, c_void_p, c_void_p, c_double, c_double, c_int32, c_void_p, c_int64,
                                      c_void_p, c_int64, c_void_p]
    lib.spart_invert_finish.argtypes = [POINTER(c_double), POINTER(c_double), c_int32, c_int32, c_int32, c_int32,
                                        c_void_p, c_int64] + [c_void_p] * 8
    lib.spart_leafangles.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_void_p]
    lib.spart_set_lidf.argtypes = [c_void_p, c_int64, c_void_p, c_void_p]
    lib.spart_profile_enable.argtypes = [c_void_p, c_int32]
    lib.spart_profile_read.argtypes = [c_void_p, POINTER(c_double), POINTER(c_int64)]
    lib.spart_measure_peaks.argtypes = [c_int32, POINTER(c_double), POINTER(c_double)]
    lib.spart_measure_fp64_chain.argtypes = [c_int32, POINTER(c_double)]
    lib.spart_launch_count.restype = c_int64
    if lib.spart_abi_version() != ABI_VERSION:
        raise SpartError(f"libspart_b200.so ABI {lib.spart_abi_version()} != expected {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().spart_last_error().decode("utf-8", "replace")
        kind = "argument error" if rc < 0 else "CUDA error"
        raise SpartError(f"{what}: {kind} {rc}: {msg}")


def row_mask(rows):
    """Bit mask of `broadcast_rows` from an int mask or an iterable of row indices (0..26)."""
    if rows is None:
        return 0
    if isinstance(rows, int):
        mask = rows
    else:
        mask = 0
        for r in rows:
            mask |= 1 << int(r)
    if mask < 0 or mask >> NPAR:
        raise ValueError("broadcast_rows: rows are 0..26")
    return mask


def as_double_ptr(a):
    return a.ctypes.data_as(POINTER(c_double))


def as_int32_ptr(a):
    return a.ctypes.data_as(POINTER(c_int32))


__all__ = ["load", "check", "SpartError", "SpartTables", "SpartSensor", "FP64", "FP32", "EXPORTS", "row_mask",
           "as_double_ptr", "as_int32_ptr", "byref", "c_void_p", "c_double", "c_int64"]
