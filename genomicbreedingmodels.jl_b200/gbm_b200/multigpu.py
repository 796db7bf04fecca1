"""Multi-GPU layer over the C ABI's ``gbm_group`` / ``gbm_sharded`` entry points
(include/gbm_b200.h, section "multi-GPU"): markers sharded by contiguous column block over
the GPUs of one box, every collective (GRM all-reduce, PC1 all-reduces, result gathers)
inside libgbm_b200.so over NCCL.

The reference's parallel axis is ``Threads.@threads for j = 1:l``
(/root/reference/src/gwas.jl:239, :363); a group of GPUs is its B200 equivalent.

Two ways to form a group:

* ``Group.local(n_gpus)`` -- this process drives all GPUs (what a Julia session does through
  the shim's ``GBM_NUM_GPUS``);
* ``Group.from_torch_distributed()`` -- one process per GPU under ``torchrun``; the 128-byte
  NCCL id is handed out with ``torch.distributed`` (any transport works: gloo, nccl, MPI, a file).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import byref, c_double, c_int, c_int64, c_void_p

import numpy as np

from . import _lib
from ._lib import check, ptr
from .core import DeviceMatrix, _f64

GROUP_ID_BYTES = 128


def _prefer_torch_nccl():
    """libgbm_b200.so binds NCCL at its first group creation and prefers a libnccl.so.2 that the process already
    holds.  PyTorch bundles its own (newer) NCCL; if the system's copy were loaded first, a later `import torch` in
    the same process would fail to resolve its symbols.  So when PyTorch is installed, load it (and with it its NCCL)
    before the first group is made.  A Julia process has no such concern: it gets the system's libnccl.so.2."""
    try:
        import torch  # noqa: F401
        import torch.distributed  # noqa: F401
    except Exception:
        pass


class Group:
    def __init__(self, handle: c_void_p):
        self._h = handle
        w, nl, fr = c_int(), c_int(), c_int()
        check(_lib.load().gbm_group_info(self._h, byref(w), byref(nl), byref(fr)))
        self.world, self.n_local, self.first_rank = w.value, nl.value, fr.value

    @classmethod
    def local(cls, n_gpus: int, devices=None) -> "Group":
        """All ``n_gpus`` GPUs driven by this process (``gbm_group_create_local``)."""
        _prefer_torch_nccl()
        h = c_void_p()
        dev = None
        if devices is not None:
            dev = (c_int * n_gpus)(*[int(d) for d in devices])
        check(_lib.load().gbm_group_create_local(int(n_gpus), dev, byref(h)))
        return cls(h)

    @staticmethod
    def unique_id() -> bytes:
        _prefer_torch_nccl()
        buf = ctypes.create_string_buffer(GROUP_ID_BYTES)
        check(_lib.load().gbm_group_unique_id(buf))
        return buf.raw

    @classmethod
    def from_rank(cls, uid: bytes, world: int, rank: int) -> "Group":
        """One process per GPU; the GPU is the one of ``gbm_b200.init`` (``gbm_group_create_rank``)."""
        if len(uid) != GROUP_ID_BYTES:
            raise _lib.ArgumentError("the group id must be 128 bytes")
        _prefer_torch_nccl()
        _lib.lib()  # gbm_init(LOCAL_RANK)
        h = c_void_p()
        check(_lib.load().gbm_group_create_rank(ctypes.c_char_p(uid), int(world), int(rank), byref(h)))
        return cls(h)

    @classmethod
    def from_torch_distributed(cls, group=None) -> "Group":
        """Collective over an initialised ``torch.distributed`` process group (any backend): rank 0 makes the
        id, everybody receives it, every rank joins."""
        import torch.distributed as dist

        world, rank = dist.get_world_size(group), dist.get_rank(group)
        box = [cls.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, group=group)
        return cls.from_rank(box[0], world, rank)

    def free(self):
        if self._h is not None:
            check(_lib.load().gbm_group_free(self._h))
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ShardedMatrix:
    """n x p genotype matrix resident as column blocks on the GPUs of a group (``gbm_sharded``)."""

    def __init__(self, group: Group, handle: c_void_p, packed: bool, keepalive=None):
        self.group, self._h, self.packed = group, handle, bool(packed)
        self._keepalive = keepalive
        n, p = c_int64(), c_int64()
        fc, nc = (c_int64 * group.n_local)(), (c_int64 * group.n_local)()
        check(_lib.load().gbm_sharded_info(self._h, byref(n), byref(p), fc, nc, None))
        self.n, self.p = n.value, p.value
        self.first_col, self.ncols = list(fc), list(nc)

    @classmethod
    def upload(cls, group: Group, A, compact: bool = True) -> "ShardedMatrix":
        """``A``: the whole host matrix (NumPy n x p, or a torch CPU tensor of shape (p, n) == n x p column-major);
        every process passes the same matrix and uploads the blocks of its own GPUs."""
        if isinstance(A, np.ndarray):
            A = _f64(A)
            n, p = A.shape
        else:
            p, n = A.shape
        h, pk = c_void_p(), c_int()
        check(_lib.load().gbm_sharded_upload(group._h, ptr(A), n, p, n, int(compact), byref(h), byref(pk)))
        return cls(group, h, pk.value)

    @classmethod
    def generate(cls, group: Group, seed: int, n: int, p: int, kind: int, pack: bool = False) -> "ShardedMatrix":
        h, pk = c_void_p(), c_int()
        check(_lib.load().gbm_sharded_generate(group._h, seed, n, p, kind, int(pack), byref(h), byref(pk)))
        return cls(group, h, pk.value)

    @classmethod
    def adopt(cls, group: Group, blocks) -> "ShardedMatrix":
        """Wrap resident ``DeviceMatrix`` blocks (one per local GPU, rank order); they stay owned by the caller."""
        arr = (c_void_p * group.n_local)(*[b._h for b in blocks])
        h = c_void_p()
        check(_lib.load().gbm_sharded_adopt(group._h, arr, byref(h)))
        return cls(group, h, all(b.packed for b in blocks), keepalive=list(blocks))

    def free(self):
        if self._h is not None:
            check(_lib.load().gbm_sharded_free(self._h))
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # ---- gwasprep pieces ---------------------------------------------------------------
    def colstats(self):
        p = self.p
        mean, sd, mnz = np.empty(p), np.empty(p), np.empty(p)
        keep = np.empty(p, dtype=np.uint8)
        idx = np.empty(p, dtype=np.int64)
        nk, mk = c_int64(), c_double()
        check(_lib.load().gbm_sharded_colstats(self._h, ptr(mean), ptr(sd), ptr(mnz), ptr(keep), ptr(idx), byref(nk),
                                               byref(mk)))
        return {"mean": mean, "sd": sd, "min_nonzero": mnz, "keep": keep.astype(bool),
                "idx_cols": idx[: nk.value].copy(), "min_nonzero_kept": mk.value}

    def grm(self, grm_type: int = _lib.GRM_SIMPLE, ploidy: int = 2, flags: int = 0, want_host: bool = True):
        """Per-GPU partials + one all-reduce + scale/mirror.  Returns (K or None, aggregate TFLOP/s); the GRM
        also stays resident on the GPUs for ``kstd_pc1``."""
        K = np.empty((self.n, self.n), dtype=np.float64, order="F") if want_host else None
        tf = c_double()
        check(_lib.load().gbm_sharded_grm(self._h, grm_type, ploidy, flags, ptr(K), byref(tf)))
        return K, tf.value

    def kstd_pc1(self, K=None):
        """PC1 of the column-standardised GRM (gwas.jl:130, :234): columns of K sharded, one n-vector all-reduce
        per Lanczos step.  ``K`` None: the GRM left resident by ``grm``."""
        pc = np.empty(self.n)
        ms = c_double()
        Kh = None if K is None else _f64(K)
        check(_lib.load().gbm_sharded_kstd_pc1(self._h, ptr(Kh), ptr(pc), byref(ms)))
        return pc, ms.value

    def scan(self, Y, C=None, model: int = _lib.MODEL_OLS, flags: int = 0):
        Y = _f64(np.asarray(Y, dtype=np.float64).reshape(self.n, -1))
        T = Y.shape[1]
        Cm = None if C is None else _f64(np.asarray(C, dtype=np.float64).reshape(self.n, -1))
        k = 0 if Cm is None else Cm.shape[1]
        p = self.p
        out = {name: np.empty((p, T), dtype=np.float64, order="F") for name in ("beta", "se", "stat", "neglog10p")}
        mean, sd = np.empty(p), np.empty(p)
        keep = np.empty(p, dtype=np.uint8)
        check(_lib.load().gbm_sharded_scan(self._h, ptr(Y), T, self.n, ptr(Cm), k, self.n, model, flags, ptr(out["beta"]),
                                           ptr(out["se"]), ptr(out["stat"]), ptr(out["neglog10p"]), ptr(mean), ptr(sd),
                                           ptr(keep)))
        out.update(mean=mean, sd=sd, keep=keep.astype(bool))
        return out

    def gwas(self, y, model: int = _lib.MODEL_LMM, grm_type: int = _lib.GRM_SIMPLE, flags: int = 0,
             want=("stat", "beta", "se", "neglog10p"), out=None):
        """Whole gwasols / gwaslmm after extractxyetc in ONE collective call (``gbm_sharded_gwas``): filter + ploidy
        probe, GRM + all-reduce, K standardisation, PC1, marker scan, gather.  ``y`` is used as given.
        ``out``: a dict from a previous call whose arrays are reused (no fresh allocations: a fresh NumPy array is
        page-faulted in while the results are copied into it)."""
        y = np.ascontiguousarray(y, dtype=np.float64)
        if y.shape != (self.n,):
            raise _lib.ArgumentError("phenotype length does not match the number of entries")
        p = self.p
        if out is None:
            out = {k: np.zeros(p) for k in want}
            out["_keep"] = np.zeros(p, dtype=np.uint8)
            out["_idx"] = np.zeros(p, dtype=np.int64)
            out["pc1"] = np.zeros(self.n)
        nk = c_int64()
        tm = _lib.GwasTiming()
        check(_lib.load().gbm_sharded_gwas(self._h, ptr(y), model, grm_type, flags, ptr(out.get("stat")), ptr(out.get("beta")),
                                           ptr(out.get("se")), ptr(out.get("neglog10p")), None, None, ptr(out["_keep"]),
                                           ptr(out["_idx"]), byref(nk), ptr(out["pc1"]), byref(tm)))
        out.update(keep=out["_keep"].view(bool), idx_cols=out["_idx"][: nk.value], timing=tm.asdict())
        return out

    def lmm_plan(self, K, y, C=None) -> "ShardedLmmPlan":
        """The GRM-covariance LMM of ``LmmPlan`` over the shards (``gbm_sharded_lmm_plan_create``): K is factored once,
        on rank 0, and U is broadcast to every GPU.  Every process passes the same K, y and C."""
        return ShardedLmmPlan(self, K, y, C)

    def gwasreml(self, y, grm_type: int = _lib.GRM_SIMPLE, objective: str = "reml", two_sided: bool = False):
        """Whole gwasreml after extractxyetc in ONE collective call (``gbm_sharded_gwasreml``): filter + ploidy probe,
        GRM + all-reduce, for ``objective="reference"`` the symmetric part of the column-standardised K, the
        eigendecomposition on rank 0 and its broadcast, rotation + delta search per GPU, gather.  ``y`` is used as
        given."""
        if objective not in ("reml", "reference"):
            raise _lib.ArgumentError("objective must be \"reml\" or \"reference\"")
        y = np.ascontiguousarray(y, dtype=np.float64)
        if y.shape != (self.n,):
            raise _lib.ArgumentError("phenotype length does not match the number of entries")
        flags = (_lib.LMM_REFERENCE_OBJECTIVE if objective == "reference" else 0) | (
            _lib.PVALUE_TWO_SIDED if two_sided else 0)
        p = self.p
        out = {k: np.empty(p) for k in ("stat", "beta", "se", "neglog10p", "log_delta")}
        idx = np.empty(p, dtype=np.int64)
        nk, lam0 = c_int64(), c_double()
        tm = _lib.RemlTiming()
        check(_lib.load().gbm_sharded_gwasreml(self._h, ptr(y), grm_type, flags, ptr(out["stat"]), ptr(out["beta"]),
                                               ptr(out["se"]), ptr(out["neglog10p"]), ptr(out["log_delta"]), ptr(idx),
                                               byref(nk), byref(lam0), byref(tm)))
        out.update(idx_cols=idx[: nk.value].copy(), null_log_delta=lam0.value, timing=tm.asdict())
        return out


class ShardedLmmPlan:
    """``gbm_sharded_lmm_plan``: the same interface as ``LmmPlan``, for a ``ShardedMatrix``."""

    def __init__(self, sm: ShardedMatrix, K, y, C=None):
        n = sm.n
        y = np.ascontiguousarray(y, dtype=np.float64)
        if y.shape != (n,):
            raise _lib.ArgumentError("phenotype length does not match the number of entries")
        K = _f64(K)
        if K.shape != (n, n):
            raise _lib.ArgumentError("GRM must be n x n")
        Cm = None if C is None else _f64(np.asarray(C, dtype=np.float64).reshape(n, -1))
        h = c_void_p()
        eig, lam0 = c_double(), c_double()
        check(_lib.load().gbm_sharded_lmm_plan_create(sm._h, ptr(K), ptr(y), ptr(Cm), 0 if Cm is None else Cm.shape[1], n,
                                                      byref(h), byref(eig), byref(lam0)))
        self._h, self.n, self._sm = h, n, sm
        self.eig_ms, self.null_log_delta = eig.value, lam0.value

    def run(self, flags: int = 0):
        p = self._sm.p
        out = {k: np.empty(p) for k in ("beta", "se", "stat", "neglog10p", "log_delta")}
        tm = _lib.RemlTiming()
        check(_lib.load().gbm_sharded_lmm_plan_run(self._h, self._sm._h, flags, ptr(out["beta"]), ptr(out["se"]),
                                                   ptr(out["stat"]), ptr(out["neglog10p"]), ptr(out["log_delta"]),
                                                   byref(tm)))
        out["timing"] = tm.asdict()
        return out

    def free(self):
        if self._h is not None:
            check(_lib.load().gbm_sharded_lmm_plan_free(self._h))
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


_default_group = None


def default_group():
    """The group the host mirror's gwasols / gwaslmm / gwasreml use: ``GBM_NUM_GPUS`` GPUs of this process (None when the
    variable is unset or 1)."""
    global _default_group
    n = int(os.environ.get("GBM_NUM_GPUS", "1") or "1")
    if n <= 1:
        return None
    if _default_group is None or _default_group.world != n:
        _default_group = Group.local(n)
    return _default_group
