"""The rotation LMM of gwasreml (gbm_sharded_lmm_plan_* / gbm_sharded_gwasreml, include/gbm_b200.h) with the markers
sharded over a group of GPUs: bit-identity with the single-GPU engine for a given K, the one-call pipeline against the
CPU oracle, the keyword API under GBM_NUM_GPUS, and argument errors.  Every test runs on a group of ONE GPU (NCCL with
a single rank: the whole code path); the `multigpu` cases add 2, 4 and 8 GPUs when the box has them."""
import os
import signal
import subprocess
import sys

import numpy as np
import pytest

from oracle import gwas_oracle as go, lmm_oracle as lo, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUTPUTS = ("beta", "se", "stat", "neglog10p", "log_delta")


def visible_gpus():
    import ctypes

    try:
        rt = ctypes.CDLL("libcudart.so.12")
        c = ctypes.c_int()
        return c.value if rt.cudaGetDeviceCount(ctypes.byref(c)) == 0 else 0
    except OSError:
        return 0


def group_sizes():
    n = visible_gpus()
    sizes = [1] + [g for g in (2, 4, 8) if g <= n]
    return [pytest.param(g, marks=[pytest.mark.multigpu] if g > 1 else []) for g in sizes]


@pytest.fixture(scope="module", params=group_sizes())
def grp(request, gbm):
    from gbm_b200 import multigpu

    g = multigpu.Group.local(request.param)
    yield g
    g.free()


def _structured(seed, n, p, kind, h2=0.5):
    A = synth.block(seed, n, 0, p, kind)
    rng = np.random.default_rng(seed)
    g = (A - A.mean(axis=0)) @ rng.normal(size=p)
    g /= g.std()
    y = np.sqrt(h2) * g + np.sqrt(1 - h2) * rng.normal(size=n)
    return A, (y - y.mean()) / y.std(ddof=1)


@pytest.mark.parametrize("p", [97, 1301])
@pytest.mark.parametrize("objective", ["reml", "reference"])
@pytest.mark.parametrize("k", [0, 1])
@pytest.mark.parametrize("packed", [False, True])
def test_plan_with_a_given_K_equals_the_single_gpu_engine_bit_for_bit(gbm, grp, packed, k, objective, p):
    """U is broadcast (the same bits on every GPU), the rotation GEMM has no split-K and the delta search's arithmetic
    per marker does not depend on the grid: every output equals LmmPlan(K, y, C).run(dm), NaN positions included.
    p = 97 puts every shard below one 128-column tile; p = 1301 gives ragged shards."""
    from gbm_b200 import multigpu

    n = 203
    A, y = _structured(31 + k, n, p, synth.KIND_DIPLOID)
    A[:, 5] = A[0, 5]  # a fixed locus: NaN in every output
    K = go.grm_simple(A)
    flags = 0
    if objective == "reference":
        Ks, _, _ = gbm.kstd_pc1(K, want_pc1=False)
        K = 0.5 * (Ks + Ks.T)
        flags = gbm._lib.LMM_REFERENCE_OBJECTIVE
    C = np.random.default_rng(7).normal(size=(n, k)) if k else None
    dm = gbm.DeviceMatrix.upload(A)
    if packed:
        f64, dm = dm, dm.pack()
        f64.free()
    sm = multigpu.ShardedMatrix.upload(grp, A, compact=packed)
    one = gbm.LmmPlan(K, y, C)
    many = sm.lmm_plan(K, y, C)
    try:
        assert sm.packed == packed and dm.packed == packed
        assert many.null_log_delta == one.null_log_delta
        for f in (flags, flags | gbm._lib.PVALUE_TWO_SIDED):
            r0, r1 = one.run(dm, flags=f), many.run(flags=f)
            assert np.isnan(r1["stat"][5])
            for key in OUTPUTS:
                assert np.array_equal(r1[key], r0[key], equal_nan=True), (key, f)
            tm = r1["timing"]
            assert tm["n_gpus"] == grp.world and tm["rotation_ms"] > 0 and tm["rotation_tflops"] > 0
    finally:
        many.free()
        one.free()
        sm.free()
        dm.free()


@pytest.mark.parametrize("grm_type,kind,n,p", [("simple", synth.KIND_DIPLOID, 300, 1001),
                                               ("ploidy-aware", synth.KIND_TETRAPLOID, 256, 700),
                                               ("simple", synth.KIND_CONTINUOUS, 240, 500)])
def test_one_call_gwasreml_matches_the_oracle(gbm, grp, grm_type, kind, n, p):
    """gbm_sharded_gwasreml == oracle lmm_scan on the oracle's GRM, with the tolerances of test_gpu_lmm.py; the filter
    indices exact; the ploidy-aware GRM infers ploidy 4."""
    from gbm_b200 import multigpu

    A = synth.block(23, n, 0, p, kind)
    y = synth.phenotype(23, n, p, kind)
    ys = (y - y.mean()) / y.std(ddof=1)
    K = go.grm_simple(A) if grm_type == "simple" else go.grm_ploidy_aware(A, 4)
    ref = lo.lmm_scan(A, ys, K)
    keep = ref["keep"]
    sm = multigpu.ShardedMatrix.generate(grp, 23, n, p, kind, pack=True)
    try:
        assert sm.packed == (kind != synth.KIND_CONTINUOUS)
        res = sm.gwasreml(ys, grm_type=gbm._lib.GRM_PLOIDY_AWARE if grm_type == "ploidy-aware" else gbm._lib.GRM_SIMPLE)
    finally:
        sm.free()
    _, v = go.column_std(A)
    assert np.array_equal(res["idx_cols"], go.fixed_locus_filter(v))
    assert np.array_equal(np.flatnonzero(keep) + 1, res["idx_cols"])
    assert np.all(np.isnan(res["stat"][~keep]))
    assert abs(res["null_log_delta"] - ref["lam0"]) < 1e-8
    assert np.max(np.abs(res["log_delta"][keep] - ref["log_delta"][keep])) < 1e-7
    zs = np.abs(ref["z"][keep]).max()
    assert np.max(np.abs(res["stat"][keep] - ref["z"][keep])) < 1e-9 * max(1.0, zs)
    sd = A.std(axis=0, ddof=1)
    np.testing.assert_allclose(res["beta"][keep], ref["beta"][keep] * sd[keep], rtol=1e-7, atol=1e-10)
    np.testing.assert_allclose(res["se"][keep], ref["se"][keep] * sd[keep], rtol=1e-8)
    want_p = go.neglog10_sf_normal(res["stat"][keep])
    assert np.max(np.abs(res["neglog10p"][keep] - want_p)) < 1e-6
    tm = res["timing"]
    assert tm["ploidy"] == (4 if grm_type == "ploidy-aware" else 2) and tm["n_gpus"] == grp.world
    assert tm["total_ms"] > 0 and tm["eig_ms"] > 0 and tm["rotation_tflops"] > 0 and tm["grm_tflops"] > 0
    assert tm["launches"] > 0


def test_one_call_reference_objective_matches_its_oracle(gbm, grp):
    """GBM_LMM_REFERENCE_OBJECTIVE in one call: K column-standardised and symmetrised on the device, against
    oracle refobj_scan on NumPy's (K + K')/2 -- 1e-6 as test_gwasreml_reference_objective_end_to_end: the device's
    and NumPy's standardised K differ in the last bits, which the unprofiled s2u amplifies."""
    from gbm_b200 import multigpu

    n, p = 100, 400
    A, y = _structured(42, n, p, synth.KIND_TETRAPLOID)
    ent = [str(i) for i in range(n)]
    prep = go.gwasprep(A, ent, y[:, None], ent, standardise=True)
    z_ref, _, _ = lo.refobj_scan(prep.G, prep.y, 0.5 * (prep.K + prep.K.T))
    sm = multigpu.ShardedMatrix.upload(grp, A, compact=True)
    try:
        res = sm.gwasreml(prep.y, objective="reference", two_sided=True)
    finally:
        sm.free()
    assert np.array_equal(res["idx_cols"], prep.idx_cols)
    z = res["stat"][res["idx_cols"] - 1]
    assert np.max(np.abs(z - z_ref)) < 1e-6 * max(1.0, np.abs(z_ref).max())
    want_p = go.neglog10_sf_normal(z) - np.log10(2.0)
    assert np.max(np.abs(res["neglog10p"][res["idx_cols"] - 1] - want_p)) < 1e-6
    assert res["timing"]["kprep_ms"] > 0


@pytest.mark.parametrize("objective", ["reml", "reference"])
@pytest.mark.parametrize("n_gpus", group_sizes())
def test_gwasreml_uses_the_group_when_gbm_num_gpus_is_set(gbm, n_gpus, objective, monkeypatch):
    """gwasreml of the host mirror (keyword API of /root/reference/src/gwas.jl:549-613) with GBM_NUM_GPUS: the Fit
    equals the single-GPU one."""
    from gbm_b200 import multigpu

    n, p = 320, 1500
    A = synth.block(3, n, 0, p, synth.KIND_TETRAPLOID)
    y = synth.phenotype(3, n, p, synth.KIND_TETRAPLOID)
    g = gbm.Genomes.from_matrix(A)
    ph = gbm.Phenomes.from_matrix(y, entries=g.entries)
    monkeypatch.delenv("GBM_NUM_GPUS", raising=False)
    one = gbm.gwasreml(genomes=g, phenomes=ph, GRM_type="ploidy-aware", objective=objective)
    monkeypatch.setenv("GBM_NUM_GPUS", str(max(n_gpus, 2) if visible_gpus() >= 2 else 1))
    if visible_gpus() < 2:  # a single visible GPU: exercise the group path with a group of one
        monkeypatch.setattr(multigpu, "default_group", lambda: multigpu.Group.local(1))
    many = gbm.gwasreml(genomes=g, phenomes=ph, GRM_type="ploidy-aware", objective=objective)
    assert many.model == one.model == "GWAS_REML" and many.b_hat_labels == one.b_hat_labels
    assert many.entries == one.entries and many.trait == one.trait
    assert many.extras["ploidy"] == one.extras["ploidy"] == 4 and many.extras["objective"] == objective
    assert many.extras["n_gpus"] >= 1 and many.extras["storage"] == "u8 dosage codes" and "timing" in many.extras
    assert set(one.extras) <= set(many.extras)
    assert np.array_equal(np.isnan(many.b_hat), np.isnan(one.b_hat))  # NaN is kept, as on one GPU
    np.testing.assert_allclose(many.b_hat, one.b_hat, rtol=1e-9, atol=1e-9 * np.nanmax(np.abs(one.b_hat)))
    for key in ("beta", "se", "neglog10p", "log_delta"):
        np.testing.assert_allclose(many.extras[key], one.extras[key], rtol=1e-9,
                                   atol=1e-9 * np.nanmax(np.abs(one.extras[key])))
    assert np.array_equal(many.extras["idx_cols"], one.extras["idx_cols"])


def test_argument_errors_return_without_a_hang(gbm, grp):
    """Checks that every rank makes before any collective: each call returns an ArgumentError, and the group is
    usable afterwards."""
    from ctypes import byref, c_double, c_int64, c_void_p

    from gbm_b200 import _lib, multigpu

    n, p = 64, 200
    A, y = _structured(5, n, p, synth.KIND_DIPLOID)
    K = go.grm_simple(A)
    sm = multigpu.ShardedMatrix.upload(grp, A)
    lib = _lib.load()
    out = np.empty(p)
    try:
        with pytest.raises(_lib.ArgumentError, match="flags"):  # GBM_GRM_NO_CENTRE-style bits are not scan flags
            _lib.check(lib.gbm_sharded_gwasreml(sm._h, _lib.ptr(y), _lib.GRM_SIMPLE, 4, _lib.ptr(out), None, None, None,
                                                None, None, None, None, None))
        with pytest.raises(_lib.ArgumentError, match="GRM_type"):
            sm.gwasreml(y, grm_type=7)
        with pytest.raises(_lib.ArgumentError):
            sm.lmm_plan(np.eye(n + 1), y)
        with pytest.raises(_lib.ArgumentError, match="covariates"):
            sm.lmm_plan(K, y, C=np.ones((n, 3)))
        h = c_void_p()
        with pytest.raises(_lib.ArgumentError):
            _lib.check(lib.gbm_sharded_lmm_plan_create(sm._h, _lib.ptr(K), None, None, 0, n, byref(h), None, None))
        with pytest.raises(_lib.ArgumentError):
            _lib.check(lib.gbm_sharded_gwasreml(sm._h, None, _lib.GRM_SIMPLE, 0, _lib.ptr(out), None, None, None, None,
                                                None, None, None, None))
        with pytest.raises(_lib.ArgumentError, match="null plan"):
            _lib.check(lib.gbm_sharded_lmm_plan_run(None, sm._h, 0, None, None, _lib.ptr(out), None, None, None))
        _lib.check(lib.gbm_sharded_lmm_plan_free(None))
        res = sm.gwasreml(y)  # the group still works
        assert np.isfinite(res["stat"][res["idx_cols"] - 1]).all()
    finally:
        sm.free()


@pytest.mark.multigpu
@pytest.mark.skipif(visible_gpus() < 2, reason="needs at least 2 GPUs on the box")
def test_gwasreml_one_process_per_gpu_under_torchrun(gbm):
    """tests/dist_reml_check.py on every visible GPU: the one-call gwasreml and the plan on a RANK group
    (gbm_group_create_rank) against the oracle."""
    n = visible_gpus()
    port = 29900 + os.getpid() % 90
    # own session: if a rank dies the others wait in NCCL for ever -- the whole process group is killed at the timeout
    proc = subprocess.Popen([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                             "--master-addr", "127.0.0.1", "--master-port", str(port),
                             os.path.join(ROOT, "tests", "dist_reml_check.py")], stdout=subprocess.PIPE,
                            stderr=subprocess.STDOUT, text=True, start_new_session=True)
    try:
        log, _ = proc.communicate(timeout=300)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, signal.SIGKILL)
        log, _ = proc.communicate()
        log += "\n[killed at the 300 s timeout]"
    print(log)  # the ranks' log: shown by pytest with the test's captured output (-rP, or on failure)
    assert proc.returncode == 0, log[-3000:]
    assert log.count("-> OK") == 1 and "FAIL" not in log, log[-3000:]
