"""ctypes binding of libgbm_b200.so -- exactly the symbols declared in include/gbm_b200.h.

The Julia shim (../julia/GenomicBreedingModelsB200.jl) binds the same symbols with `ccall`;
this module is the harness that can run in an image without Julia.  There is no fallback:
if the shared library is missing or no B200 is present, every compute call raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, byref, c_char_p, c_double, c_int, c_int64, c_uint8, c_uint64, c_void_p

import numpy as np

_PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG_DIR, "libgbm_b200.so")
CSRC_DIR = os.path.join(_PKG_DIR, "csrc")

ABI_VERSION = 3  # GBM_ABI_VERSION of include/gbm_b200.h
GBM_OK = 0
GBM_ERR_ARGUMENT = 1
GBM_ERR_RUNTIME = 2
GBM_ERR_CUDA = 3
GBM_ERR_NOT_INITIALISED = 4

GRM_SIMPLE, GRM_PLOIDY_AWARE = 0, 1
GRM_NO_CENTRE = 1
MODEL_OLS, MODEL_LMM = 0, 1
PVALUE_TWO_SIDED = 1
SCAN_HOST_NO_PACK = 4
LMM_REFERENCE_OBJECTIVE = 8
KIND_DIPLOID, KIND_TETRAPLOID, KIND_CONTINUOUS = 0, 1, 2


class ArgumentError(ValueError):
    """Julia ``ArgumentError`` (GBM_ERR_ARGUMENT)."""


class ErrorException(RuntimeError):
    """Julia ``ErrorException`` (GBM_ERR_RUNTIME)."""


class CudaError(RuntimeError):
    """CUDA / cuSOLVER failure, or no usable B200 (GBM_ERR_CUDA / NOT_INITIALISED)."""


class GwasTiming(ctypes.Structure):
    """gbm_gwas_timing of include/gbm_b200.h"""
    _fields_ = [("colstats_ms", c_double), ("grm_ms", c_double), ("allreduce_ms", c_double), ("kstd_pc1_ms", c_double),
                ("eig_ms", c_double), ("scan_ms", c_double), ("gather_ms", c_double), ("total_ms", c_double),
                ("grm_tflops", c_double), ("scan_kernel_ms", c_double), ("launches", c_int64),
                ("ploidy", ctypes.c_int32), ("lanczos_steps", ctypes.c_int32)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class RemlTiming(ctypes.Structure):
    """gbm_reml_timing of include/gbm_b200.h"""
    _fields_ = [("colstats_ms", c_double), ("grm_ms", c_double), ("allreduce_ms", c_double), ("kprep_ms", c_double),
                ("eig_ms", c_double), ("broadcast_ms", c_double), ("scan_ms", c_double), ("gather_ms", c_double),
                ("total_ms", c_double), ("rotation_ms", c_double), ("search_ms", c_double), ("rotation_tflops", c_double),
                ("grm_tflops", c_double), ("launches", c_int64), ("ploidy", ctypes.c_int32), ("n_gpus", ctypes.c_int32)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Timing(ctypes.Structure):
    _fields_ = [("h2d_ms", c_double), ("kernel_ms", c_double), ("main_ms", c_double), ("d2h_ms", c_double),
                ("launches", c_int64), ("packed_blocks", c_int64), ("host_packed_blocks", c_int64), ("h2d_bytes", c_int64)]


# every exported symbol of include/gbm_b200.h: name -> (restype, argtypes)
_P = c_void_p  # data pointers may be host or device addresses
SIGNATURES = {
    "gbm_abi_version": (c_int, []),
    "gbm_last_error": (c_char_p, []),
    "gbm_init": (c_int, [c_int]),
    "gbm_shutdown": (c_int, []),
    "gbm_set_stream": (c_int, [c_void_p]),
    "gbm_synchronize": (c_int, []),
    "gbm_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int64), c_char_p, c_int]),
    "gbm_last_timing": (c_int, [POINTER(Timing)]),
    "gbm_matrix_upload": (c_int, [_P, c_int64, c_int64, c_int64, POINTER(c_void_p)]),
    "gbm_matrix_upload_compact": (c_int, [_P, c_int64, c_int64, c_int64, POINTER(c_void_p), POINTER(c_int)]),
    "gbm_matrix_upload_indexed": (c_int, [_P, c_int64, c_int64, c_int64, _P, c_int64, _P, c_int64, POINTER(c_void_p)]),
    "gbm_matrix_wrap": (c_int, [_P, c_int64, c_int64, c_int64, POINTER(c_void_p)]),
    "gbm_matrix_generate": (c_int, [c_uint64, c_int64, c_int64, c_int64, c_int, POINTER(c_void_p)]),
    "gbm_matrix_pack": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_int64)]),
    "gbm_matrix_upload_packed": (c_int, [_P, c_int64, c_int64, c_int64, POINTER(c_void_p)]),
    "gbm_pack_host": (c_int, [_P, c_int64, c_int64, c_int64, _P, c_int64, POINTER(c_int64)]),
    "gbm_pack_host_check": (c_int, [_P, c_int64, c_int64, c_int64, c_int, _P]),
    "gbm_side_vector_digits": (c_int, [_P, c_int64, c_int, c_int64, _P, c_int64, POINTER(c_double)]),
    "gbm_tridiag_top": (c_int, [_P, _P, c_int64, POINTER(c_double), _P]),
    "gbm_matrix_download": (c_int, [c_void_p, c_int64, c_int64, _P, c_int64]),
    "gbm_matrix_download_cols": (c_int, [c_void_p, _P, c_int64, c_int, _P, c_int64]),
    "gbm_matrix_info": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64), POINTER(c_void_p)]),
    "gbm_matrix_free": (c_int, [c_void_p]),
    "gbm_colstats": (c_int, [c_void_p, _P, _P, _P, _P, _P, POINTER(c_int64), POINTER(c_double)]),
    "gbm_grm": (c_int, [c_void_p, c_int, c_int, c_int, _P, POINTER(c_double)]),
    "gbm_grm_accumulate": (c_int, [c_void_p, c_int, _P, POINTER(c_double), POINTER(c_double)]),
    "gbm_grm_finalize": (c_int, [_P, c_int64, c_double]),
    "gbm_kstd_pc1": (c_int, [_P, c_int64, _P, _P, POINTER(c_double)]),
    "gbm_scan": (c_int, [c_void_p, _P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, _P, _P, _P, _P, _P, _P, _P]),
    "gbm_scan_plan_create": (c_int, [c_void_p, _P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, POINTER(c_void_p)]),
    "gbm_scan_plan_run": (c_int, [c_void_p, _P, _P, _P, _P, _P, _P, _P]),
    "gbm_scan_plan_free": (c_int, [c_void_p]),
    "gbm_scan_host": (c_int, [_P, c_int64, c_int64, c_int64, _P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int,
                              _P, _P, _P, _P, _P, _P, _P]),
    "gbm_lmm_plan_create": (c_int, [_P, c_int64, _P, _P, c_int64, c_int64, POINTER(c_void_p), POINTER(c_double),
                                    POINTER(c_double)]),
    "gbm_lmm_plan_run": (c_int, [c_void_p, c_void_p, c_int, _P, _P, _P, _P, _P, POINTER(c_double), POINTER(c_double)]),
    "gbm_lmm_plan_free": (c_int, [c_void_p]),
    "gbm_gemm_tn": (c_int, [_P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int64, c_int64, POINTER(c_double)]),
    "gbm_transform1_screen": (c_int, [c_void_p, _P, c_int, c_double, c_int, c_double, c_int64, _P, _P, POINTER(c_int64)]),
    "gbm_transform2_screen": (c_int, [c_void_p, _P, c_int, c_double, c_int, c_double, c_int, c_int64, _P, _P, _P,
                                      POINTER(c_int64)]),
    "gbm_transform2_screen_rows": (c_int, [c_void_p, _P, c_int, c_double, c_int, c_double, c_int, c_int64, c_int64, c_int64,
                                           _P, _P, _P, POINTER(c_int64)]),
    "gbm_transform1_apply": (c_int, [c_void_p, c_int, c_double, c_int, _P, c_int64, _P, c_int64]),
    "gbm_transform2_apply": (c_int, [c_void_p, c_int, c_double, c_int, _P, c_int64, _P, c_int64]),
    "gbm_group_create_local": (c_int, [c_int, POINTER(c_int), POINTER(c_void_p)]),
    "gbm_group_unique_id": (c_int, [_P]),
    "gbm_group_create_rank": (c_int, [_P, c_int, c_int, POINTER(c_void_p)]),
    "gbm_group_info": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "gbm_group_free": (c_int, [c_void_p]),
    "gbm_sharded_upload": (c_int, [c_void_p, _P, c_int64, c_int64, c_int64, c_int, POINTER(c_void_p), POINTER(c_int)]),
    "gbm_sharded_generate": (c_int, [c_void_p, c_uint64, c_int64, c_int64, c_int, c_int, POINTER(c_void_p), POINTER(c_int)]),
    "gbm_sharded_adopt": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p)]),
    "gbm_sharded_info": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64),
                                 POINTER(c_int)]),
    "gbm_sharded_free": (c_int, [c_void_p]),
    "gbm_sharded_colstats": (c_int, [c_void_p, _P, _P, _P, _P, _P, POINTER(c_int64), POINTER(c_double)]),
    "gbm_sharded_grm": (c_int, [c_void_p, c_int, c_int, c_int, _P, POINTER(c_double)]),
    "gbm_sharded_kstd_pc1": (c_int, [c_void_p, _P, _P, POINTER(c_double)]),
    "gbm_sharded_scan": (c_int, [c_void_p, _P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, _P, _P, _P, _P, _P, _P,
                                 _P]),
    "gbm_sharded_gwas": (c_int, [c_void_p, _P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, POINTER(c_int64), _P,
                                 POINTER(GwasTiming)]),
    "gbm_sharded_lmm_plan_create": (c_int, [c_void_p, _P, _P, _P, c_int64, c_int64, POINTER(c_void_p), POINTER(c_double),
                                            POINTER(c_double)]),
    "gbm_sharded_lmm_plan_run": (c_int, [c_void_p, c_void_p, c_int, _P, _P, _P, _P, _P, POINTER(RemlTiming)]),
    "gbm_sharded_lmm_plan_free": (c_int, [c_void_p]),
    "gbm_sharded_gwasreml": (c_int, [c_void_p, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, POINTER(c_int64), POINTER(c_double),
                                     POINTER(RemlTiming)]),
    "gbm_neglog10_sf": (c_int, [_P, c_int64, c_int, c_double, _P]),
    "gbm_measure_copy_bandwidth": (c_int, [c_int64, c_int, POINTER(c_double)]),
}

_lib = None
_initialised_device = None


def build(force: bool = False) -> str:
    """Compile libgbm_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC_DIR, f) for f in os.listdir(CSRC_DIR) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(os.path.dirname(_PKG_DIR), "include", "gbm_b200.h"))
    stale = force or not os.path.exists(LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if stale:
        subprocess.check_call(["make", "-C", CSRC_DIR, "-j8"], stdout=subprocess.DEVNULL)
    return LIB_PATH


def load():
    """dlopen the library and declare every prototype.  Raises if the .so is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CudaError(
                f"{LIB_PATH} is missing: build it with `make -C {CSRC_DIR}` (there is no CPU fallback)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.gbm_abi_version() != ABI_VERSION:
            raise CudaError("libgbm_b200.so ABI version mismatch")
        _lib = lib
    return _lib


def check(code: int):
    if code == GBM_OK:
        return
    msg = (load().gbm_last_error() or b"").decode("utf-8", "replace")
    if code == GBM_ERR_ARGUMENT:
        raise ArgumentError(msg)
    if code == GBM_ERR_RUNTIME:
        raise ErrorException(msg)
    raise CudaError(msg)


def init(device: int | None = None):
    """Select the GPU (default: LOCAL_RANK or 0).  Raises CudaError without a B200."""
    global _initialised_device
    lib = load()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if _initialised_device != device:
        check(lib.gbm_init(device))
        _initialised_device = device
    return lib


def lib():
    if _initialised_device is None:
        return init()
    return load()


def ptr(x):
    """Address of a NumPy array (host), a torch tensor (host or CUDA), an int address or None."""
    if x is None:
        return None
    if isinstance(x, int):
        return c_void_p(x)
    if isinstance(x, np.ndarray):
        return c_void_p(x.ctypes.data)
    if hasattr(x, "data_ptr"):
        return c_void_p(x.data_ptr())
    raise TypeError(f"cannot take the address of {type(x)}")


def last_timing() -> dict:
    t = Timing()
    check(load().gbm_last_timing(byref(t)))
    return {"h2d_ms": t.h2d_ms, "kernel_ms": t.kernel_ms, "main_ms": t.main_ms, "d2h_ms": t.d2h_ms,
            "launches": int(t.launches), "packed_blocks": int(t.packed_blocks),
            "host_packed_blocks": int(t.host_packed_blocks), "h2d_bytes": int(t.h2d_bytes)}


def device_info() -> dict:
    sm, maj, mnr, mem = c_int(), c_int(), c_int(), c_int64()
    name = ctypes.create_string_buffer(128)
    check(lib().gbm_device_info(byref(sm), byref(maj), byref(mnr), byref(mem), name, 128))
    return {"sm_count": sm.value, "cc": (maj.value, mnr.value), "hbm_bytes": mem.value, "name": name.value.decode()}
