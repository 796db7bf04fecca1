"""CPU checks of the sharded gwasreml entry points (gbm_sharded_lmm_plan_* / gbm_sharded_gwasreml): the timing
struct is the same in the header, the ctypes binding and the Julia shim, and without a GPU every new path fails with
a clear error instead of falling back."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "gbm_b200.h")
SHIM = os.path.join(ROOT, "genomicbreedingmodels.jl_b200", "julia", "GenomicBreedingModelsB200.jl")
KIND = {"double": "f64", "int64_t": "i64", "int32_t": "i32", "Float64": "f64", "Int64": "i64", "Int32": "i32"}


def header_fields():
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"typedef struct gbm_reml_timing \{(.*?)\} gbm_reml_timing;", src, flags=re.S).group(1)
    fields = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if decl:
            ctype, names = decl.split(" ", 1)
            fields += [(name.strip(), KIND[ctype]) for name in names.split(",")]
    return fields


def test_julia_shim_reml_timing_matches_the_header():
    """`RemlTiming` (passed by reference to gbm_sharded_gwasreml) has gbm_reml_timing's fields in order and width."""
    text = open(SHIM).read()
    jbody = re.search(r"struct RemlTiming[^\n]*\n(.*?)\nend", text, flags=re.S).group(1)
    j_fields = [(name, KIND[t]) for name, t in re.findall(r"([a-z_0-9]+)::([A-Za-z0-9]+)", jbody)]
    assert j_fields == header_fields()


def test_ctypes_reml_timing_matches_the_header():
    from gbm_b200 import _lib

    kinds = {ctypes.c_double: "f64", ctypes.c_int64: "i64", ctypes.c_int32: "i32"}
    assert [(name, kinds[t]) for name, t in _lib.RemlTiming._fields_] == header_fields()
    assert ctypes.sizeof(_lib.RemlTiming) == 13 * 8 + 8 + 2 * 4


def _has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU failure mode")
def test_sharded_gwasreml_fails_loudly_without_gpu(monkeypatch):
    import gbm_b200
    from gbm_b200 import _lib, multigpu

    lib = _lib.load()
    out = np.empty(4)
    with pytest.raises(_lib.ArgumentError, match="null sharded-matrix handle"):
        _lib.check(lib.gbm_sharded_gwasreml(None, _lib.ptr(out), 0, 0, None, None, None, None, None, None, None, None,
                                            None))
    with pytest.raises(_lib.ArgumentError, match="null sharded-matrix handle"):
        _lib.check(lib.gbm_sharded_lmm_plan_create(None, _lib.ptr(out), _lib.ptr(out), None, 0, 2,
                                                   ctypes.byref(ctypes.c_void_p()), None, None))
    with pytest.raises(_lib.ArgumentError, match="null sharded-matrix handle"):
        _lib.check(lib.gbm_sharded_lmm_plan_run(None, None, 0, None, None, None, None, None, None))
    with pytest.raises(_lib.CudaError, match="no CUDA device"):
        multigpu.Group.local(1)
    # the keyword API under GBM_NUM_GPUS: the group cannot be formed, and that is an error, not a CPU run
    A = np.asfortranarray(np.random.default_rng(0).integers(0, 3, size=(10, 6)) / 2.0)
    g = gbm_b200.Genomes.from_matrix(A)
    ph = gbm_b200.Phenomes.from_matrix(np.arange(10.0), entries=g.entries)
    monkeypatch.setenv("GBM_NUM_GPUS", "2")
    with pytest.raises(_lib.CudaError):
        gbm_b200.gwasreml(genomes=g, phenomes=ph)
