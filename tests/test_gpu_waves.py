"""The persistent kernels past their first wave.

Every hot kernel launches min(work items, SMs) CTAs and loops over items, carrying state from one item to the next:
the TMA ring's stage / phase, the double-buffered TMEM accumulator of the tcgen05 kernels, the end-of-work sentinel of
grm_i8.cu, and the LMM engine's column blocks and grid-stride rounds.  None of it runs until a CTA takes its second
item, so each case here takes its shape from the device's SM count, asserts that every CTA gets several items (with the
kernel's own tiling formula, constants quoted from the .cu file), and only then compares all outputs with a reference
that shares no code with the kernel: exact integer products, the NumPy oracle, or the independent CUDA-core kernel."""
import os
from ctypes import byref, c_double

import numpy as np
import pytest

from oracle import gwas_oracle as go, lmm_oracle as lo, synth

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def sm(gbm):
    """SM count as the launchers see it (State::sm_count = multiProcessorCount)."""
    return gbm._lib.device_info()["sm_count"]


def _coverage(name, items, k, sm):
    print(f"{name}: {items} work items on {sm} SMs ({items / sm:.2f} per CTA)")
    assert items >= k * sm, f"{name}: {items} work items no longer give every CTA {k} of them on {sm} SMs"


def _rel_err(a, b, floor=1e-4):
    """max |a-b| / max(|b|, floor * max|b|): relative, with the floor the parity tests use for statistics near 0."""
    a, b = np.asarray(a), np.asarray(b)
    scale = max(float(np.nanmax(np.abs(b))), 1e-300)
    return float(np.nanmax(np.abs(a - b) / np.maximum(np.abs(b), floor * scale)))


def _heavy_tailed(n, seed):
    """Trait and covariate with a wide dynamic range, as in the tensor-core code scan test."""
    rng = np.random.default_rng(seed)
    y = rng.normal(size=n) * np.exp(rng.normal(size=n) * 3.0)
    pc = rng.normal(size=n)
    pc[rng.integers(0, n, 5)] *= 1e3
    return (y - y.mean()) / y.std(ddof=1), pc


def _closed_form(cols_fn, ncols, ys, pc, chunk=4096):
    """go.scan_closed_form over column chunks (columns are independent): beta, se_lmm, stat_lmm, mean, sd."""
    out = {k: np.empty(ncols) for k in ("beta", "se_lmm", "stat_lmm", "mean", "sd")}
    for c0 in range(0, ncols, chunk):
        c1 = min(c0 + chunk, ncols)
        r = go.scan_closed_form(cols_fn(c0, c1), ys, pc)
        for k in out:
            out[k][c0:c1] = r[k]
    return out


# ---------------------------------------------------------------------------------------------------------------------
# 1. grm_i8_kernel: dynamic fetch over (tile, slice) items, 4-slot ring, two TMEM accumulators, sentinel
# ---------------------------------------------------------------------------------------------------------------------
def test_int8_grm_past_the_first_wave_is_exact(gbm, sm):
    # grm_i8.cu: kI8Tile = 128 rows i, kI8TileN = 256 rows i', tiles(nb) = sum_{bi < nb} (bi / 2 + 1);
    # kI8KB = 128 markers per step, kI8SliceStages = 256 steps (32,768 markers) per item
    assert os.environ.get("GBM_GRM_INT8", "1") != "0", "GBM_GRM_INT8=0 routes packed GRMs away from grm_i8.cu"
    n, p = 24 * 128 + 1, 32768 + 200  # last row block holds one row; last slice: 2 steps, the second 72 markers
    nb = (n + 127) // 128
    tiles = sum(bi // 2 + 1 for bi in range(nb))
    steps = (p + 127) // 128
    slices = (steps + 255) // 256
    assert (tiles, slices) == (169, 2)
    # the last column block (bj = 12, rows 3072..3327): its second 128-row box starts at 3200 >= n
    assert ((nb - 1) // 2) * 256 + 128 >= n
    _coverage("grm_i8", tiles * slices, 2, sm)

    src = gbm.DeviceMatrix.generate(31, n, p, synth.KIND_DIPLOID)
    A = src.download()
    src.free()
    A[5] = 0.0  # a row of zeros: G[5, :] = 0, so Ku[5, :] must be exactly 0
    dm = gbm.DeviceMatrix.upload(A)
    pk = dm.pack()
    assert pk is not None
    Ks, _ = pk.grm(0, 2, 0)
    Ks2, _ = pk.grm(0, 2, 0)
    Ku, _ = pk.grm(0, 2, 1)
    Ku2, _ = pk.grm(0, 2, 1)
    Kp, _ = pk.grm(1, 2, 0)
    Kf, _ = dm.grm(0, 2, 0)  # the Float64 DMMA route (grm.cu) on the same data
    dm.free()
    pk.free()

    # exact integer parts.  Every product of codes is <= 240^2 and every partial sum of G = C C' is an integer below
    # 57600 p < 2^53, so the float64 BLAS product is exact whatever its summation order; likewise U = C S
    # (partial sums <= 240 * 240 n * p < 2^53).  M2 = sum_j S_j^2 can pass 2^53 in general: Python integers.
    C = np.rint(240.0 * A)
    G = C @ C.T
    S = C.sum(axis=0)
    U = (C @ S).astype(np.int64)
    del C
    M2 = sum(int(s) * int(s) for s in S.astype(np.int64))
    Gi = G.astype(np.int64)

    for K in (Ks, Ks2, Ku, Ku2, Kp, Kf):
        assert np.array_equal(K, K.T)
    # the header's claim: a deterministic function of the codes, whatever order the CTAs fetched the items in
    assert np.array_equal(Ks, Ks2) and np.array_equal(Ku, Ku2)

    # uncentred: G / (57600 p) to a few roundings per element, exact zeros where G is zero
    want_u = G / (57600.0 * p)
    assert np.all(np.abs(Ku - want_u) <= 4 * EPS * np.abs(want_u))
    assert np.all(Ku[G == 0] == 0.0) and np.all(Ku[5] == 0.0)

    # centred: 57600 p n^2 Kc = n^2 G - n (U_i + U_i') + M2, an integer below 2^63 here
    assert 4 * 57600 * n * n * p < 2**63  # |n^2 G|, |n U_i|, M2 <= 57600 n^2 p
    num = n * n * Gi - n * (U[:, None] + U[None, :]) + M2
    want_c = num / float(n * n * 57600 * p)
    scale = np.abs(want_c).max()
    assert np.max(np.abs(Ks - want_c)) < 1e-12 * scale
    assert np.max(np.abs(Ks - go.grm_simple(A))) < 1e-11 * scale
    assert np.max(np.abs(Kp - go.grm_ploidy_aware(A, 2))) < 1e-11 * np.abs(Kp).max()
    # the int8 route and the DMMA route
    assert np.max(np.abs(Ks - Kf)) < 1e-11 * np.abs(Kf).max()


# ---------------------------------------------------------------------------------------------------------------------
# 2. scan_sums_u8_tc_kernel: static tiles (tile += gridDim.x), 10-slot ring, two TMEM accumulators per segment
# ---------------------------------------------------------------------------------------------------------------------
def _tc_scans(pk, ys, pc, monkeypatch):
    """M = 2 (model 1 with the covariate) and M = 1 (model 0, no covariate) on the tcgen05 kernel and on the
    CUDA-core code kernel of scan_u8.cu."""
    out = {}
    for tc in ("1", "0"):
        monkeypatch.setenv("GBM_U8_TC", tc)
        out["tc" if tc == "1" else "cc", 2] = pk.scan(ys, pc[:, None], model=1)
        out["tc" if tc == "1" else "cc", 1] = pk.scan(ys, None, model=0)
    monkeypatch.delenv("GBM_U8_TC")
    return out


def _tc_equals_cuda_cores(res):
    for m in (2, 1):
        tc, cc = res["tc", m], res["cc", m]
        keep = cc["keep"]
        assert np.array_equal(tc["keep"], keep)
        for key in ("mean", "sd"):  # integer sums in both code kernels: bit for bit
            assert np.array_equal(tc[key], cc[key]), (m, key)
        for key in ("beta", "se", "stat"):
            x, z = tc[key][keep], cc[key][keep]
            assert np.nanmax(np.abs(x - z)) <= 1e-10 * max(1.0, np.nanmax(np.abs(z))), (m, key)
            assert np.all(np.isfinite(x)) and np.all(np.isnan(tc[key][~keep])), (m, key)


# scan_u8_tc.cu: kTcMarkers = 128 markers per tile, kTcRows = 128 rows per ring slot (chunk), kTcStages = 10,
# kTcSegChunks = 512 chunks (65,536 rows) per accumulation segment
def test_code_scan_many_tiles_per_cta(gbm, sm, monkeypatch):
    """Case A: every CTA takes >= 3 tiles, the last round is partial and ragged; n = 833 is 7 chunks per tile, coprime
    with the 10-slot ring, so consecutive tiles start on different slots and phases.  Also: a copy of the columns
    from a j0 that is not a multiple of 128 scans to the same bits (tile assignment does not matter)."""
    n, p = 833, 3 * 128 * sm + 77
    chunks = (n + 127) // 128
    assert chunks == 7 and np.gcd(chunks, 10) == 1
    tiles = (p + 127) // 128
    _coverage("scan_u8_tc (case A)", tiles, 3, sm)
    src = gbm.DeviceMatrix.generate(23, n, p, synth.KIND_TETRAPLOID)
    A = src.download()
    src.free()
    const = {3: 0.75, 128 * sm + 5: 0.0, 2 * 128 * sm + 200: 1.0 / 3.0, p - 1: 1.0}  # CTA 0's first, 2nd, 3rd, last tile
    for j, v in const.items():
        A[:, j] = v
    codes = np.asfortranarray(np.rint(A * 240.0).astype(np.uint8))
    assert np.array_equal(codes / 240.0, A)
    ys, pc = _heavy_tailed(n, 1)
    pk = gbm.DeviceMatrix.upload_packed(codes)
    res = _tc_scans(pk, ys, pc, monkeypatch)
    pk.free()
    _tc_equals_cuda_cores(res)

    tc = res["tc", 2]
    keep = tc["keep"]
    assert not keep[list(const)].any() and np.all(tc["sd"][list(const)] == 0.0)
    kept = np.flatnonzero(keep)
    pcn = pc - pc.mean()
    ref = _closed_form(lambda c0, c1: A[:, kept[c0:c1]], kept.size, ys, pcn / np.linalg.norm(pcn))
    assert _rel_err(tc["stat"][keep, 0], ref["stat_lmm"]) < 1e-9
    assert _rel_err(tc["beta"][keep, 0], ref["beta"]) < 1e-9
    assert _rel_err(tc["se"][keep, 0], ref["se_lmm"], floor=0) < 1e-9
    np.testing.assert_allclose(tc["mean"][keep], ref["mean"], rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(tc["sd"][keep], ref["sd"], rtol=1e-11)

    # the same markers in other tiles and other TMEM lanes: columns [j0, p) as a matrix of their own
    j0 = 128 * sm + 45
    sub = gbm.DeviceMatrix.upload_packed(codes[:, j0:])
    part = _tc_scans(sub, ys, pc, monkeypatch)
    sub.free()
    for m in (2, 1):
        full, mine = res["tc", m], part["tc", m]
        assert np.array_equal(mine["keep"], full["keep"][j0:])
        for key in ("mean", "sd", "beta", "se", "stat"):
            assert np.array_equal(mine[key], full[key][j0:], equal_nan=True), (m, key)


def test_code_scan_two_segments_per_tile(gbm, sm, monkeypatch):
    """Case B: n = 65,536 + 1,000 rows is two s32 accumulation segments per tile, and p = 2 * 128 * sm + 5 gives every
    CTA >= 2 tiles, so both TMEM accumulators are reused after a tempty wait (>= 4 segments per CTA)."""
    n, p = 65536 + 1000, 2 * 128 * sm + 5
    chunks = (n + 127) // 128
    segments = (chunks + 511) // 512
    assert segments == 2
    tiles = (p + 127) // 128
    _coverage("scan_u8_tc (case B) tiles", tiles, 2, sm)
    _coverage("scan_u8_tc (case B) segments", tiles * segments, 4, sm)
    kind, seed = synth.KIND_TETRAPLOID, 29
    dm = gbm.DeviceMatrix.generate(seed, n, p, kind)
    pk = dm.pack()
    dm.free()
    assert pk is not None
    ys, pc = _heavy_tailed(n, 2)
    res = _tc_scans(pk, ys, pc, monkeypatch)
    pk.free()
    _tc_equals_cuda_cores(res)

    # the oracle on every CTA's second tile (tiles sm .. 2 sm - 1, a different lane in each), the last column and the
    # generator's constant columns among them
    fixed = synth.column_params(seed, np.arange(p, dtype=np.uint64))[1]
    second = np.arange(128 * sm, 256 * sm)
    cols = np.unique(np.concatenate([
        np.arange(sm, 2 * sm) * 128 + (np.arange(sm) * 37) % 128,
        second[fixed[second]][:8], [p - 1]]))
    assert fixed[cols].any()
    A = np.column_stack([synth.block(seed, n, int(j), 1, kind)[:, 0] for j in cols])
    tc = res["tc", 2]
    mu, v = go.column_std(A)
    keep = v > go.EPS
    assert np.array_equal(tc["keep"][cols], keep) and np.array_equal(keep, ~fixed[cols])
    assert np.all(np.isnan(tc["stat"][cols[~keep], 0]))
    pcn = pc - pc.mean()
    ref = go.scan_closed_form(A[:, keep], ys, pcn / np.linalg.norm(pcn))
    sel = cols[keep]
    assert _rel_err(tc["stat"][sel, 0], ref["stat_lmm"]) < 1e-9
    assert _rel_err(tc["beta"][sel, 0], ref["beta"]) < 1e-9
    assert _rel_err(tc["se"][sel, 0], ref["se_lmm"], floor=0) < 1e-9
    np.testing.assert_allclose(tc["mean"][cols], mu, rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(tc["sd"][sel], v[keep], rtol=1e-11)


# ---------------------------------------------------------------------------------------------------------------------
# 3. scan_sums_mt_kernel: V = 0 (128 markers per tile), V = 1 and V = 2 (256 markers per tile), static tiles
# ---------------------------------------------------------------------------------------------------------------------
def test_multi_trait_scan_all_variants_past_the_first_wave(gbm, sm):
    # scan_mt.cu: MtCfg<NT, V>::MARKERS = 128 (V = 0) or 256 (V = 1, 2); NT = (M + 1 + 7) / 8;
    # mt_variant(nt) = nt >= 2 ? 1 : 0 for Float64, V = 2 for codes
    for var in ("GBM_MT_VARIANT", "GBM_SCAN_NO_DMMA"):
        assert var not in os.environ, f"{var} changes which scan_mt.cu variant these shapes select"
    n, p = 1001, 3 * 256 * sm + 33
    _coverage("scan_mt V=0 tiles", (p + 127) // 128, 6, sm)
    _coverage("scan_mt V=1/2 tiles", (p + 255) // 256, 3, sm)
    src = gbm.DeviceMatrix.generate(37, n, p, synth.KIND_TETRAPLOID)
    A = src.download()
    src.free()
    const = {256 * sm + 7: 0.25, 2 * 256 * sm + 300: 1.0 / 3.0, p - 1: 0.3}  # dyadic and non-dyadic, later tiles
    for j, v in const.items():
        A[:, j] = v
    dm = gbm.DeviceMatrix.upload(A)
    pk = dm.pack()
    assert pk is not None
    rng = np.random.default_rng(n)
    Y = rng.normal(size=(n, 30)) + 3.0
    C = rng.normal(size=(n, 1))
    runs = []
    for T, m, V in ((5, dm, 0), (20, dm, 1), (30, dm, 1), (20, pk, 2)):
        M = 1 + T
        nt = (M + 1 + 7) // 8
        assert (V == 2) == m.packed and (m.packed or V == (1 if nt >= 2 else 0)) and M <= 31
        runs.append((T, V, m.scan(Y[:, :T], C, model=0)))
    dm.free()
    pk.free()

    # reference: the projection formula over all markers and all 30 traits, column chunk by column chunk
    Qo, _ = np.linalg.qr(np.hstack([np.ones((n, 1)), C]))
    My = Y - Qo @ (Qo.T @ Y)
    mu, sd = np.empty(p), np.empty(p)
    ref = np.full((p, 30), np.nan)
    for c0 in range(0, p, 8192):
        a = A[:, c0:c0 + 8192]
        mu[c0:c0 + a.shape[1]], sd[c0:c0 + a.shape[1]] = go.column_std(a)
        d = a - mu[c0:c0 + a.shape[1]]
        Md = d - Qo @ (Qo.T @ d)
        with np.errstate(invalid="ignore", divide="ignore"):
            ref[c0:c0 + a.shape[1]] = (My.T @ Md / np.sqrt(np.einsum("ij,ij->j", Md, Md))).T
    keep = sd > go.EPS
    assert not keep[list(const)].any()
    for T, V, res in runs:
        assert np.array_equal(res["keep"], keep), V
        assert np.all(res["sd"][list(const)] == 0.0), V
        np.testing.assert_allclose(res["mean"], mu, rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(res["sd"][keep], sd[keep], rtol=1e-11)
        for key in ("beta", "se", "stat", "neglog10p"):
            assert np.all(np.isnan(res[key][~keep])), (T, V, key)
            assert np.all(np.isfinite(res[key][keep])), (T, V, key)
        for t in range(T):
            assert _rel_err(res["stat"][keep, t], ref[keep, t]) < 1e-9, (T, V, t)


# ---------------------------------------------------------------------------------------------------------------------
# 4. the LMM engine: column blocks of gbm_lmm_plan_run, grid-stride rounds of lmm_delta_kernel
# ---------------------------------------------------------------------------------------------------------------------
def _lmm_run_into_sentinels(gbm, plan, m):
    """gbm_lmm_plan_run into device outputs pre-filled with +inf: an entry no block wrote stays +inf."""
    import torch

    p = m.p
    outs = [torch.full((p,), float("inf"), dtype=torch.float64, device="cuda:0") for _ in range(5)]
    torch.cuda.synchronize()  # the library works on its own non-blocking stream
    tf, sms = c_double(), c_double()
    gbm._lib.check(gbm._lib.lib().gbm_lmm_plan_run(plan._h, m._h, 0, *[gbm._lib.ptr(o) for o in outs], byref(tf),
                                                   byref(sms)))
    return dict(zip(("beta", "se", "stat", "neglog10p", "log_delta"), (o.cpu().numpy() for o in outs)))


def test_lmm_engine_across_blocks_and_rounds(gbm, sm):
    n = 2003
    # gbm_lmm_plan_run: ldr = round_up(n, 16), PB = max(128, 2^30 / (8 ldr) rounded down to 128) markers per block;
    # lmm_delta_kernel: min(ceil(pb / 8), 6 sm) blocks of 8 warps, one warp per marker, grid-stride
    ldr = (n + 15) // 16 * 16
    PB = max(128, ((1 << 30) // (8 * ldr)) // 128 * 128)
    assert (ldr, PB) == (2016, 66560)
    p = 2 * PB + 1001
    nblocks = (p + PB - 1) // PB
    W = min((PB + 7) // 8, 6 * sm) * 8  # warps per grid-stride round in a full block
    rounds = (PB + W - 1) // W
    assert nblocks == 3
    # markers of one column block against the 6 x 8 warps per SM: every warp takes >= 2 markers of every full block
    _coverage("lmm_delta markers per column block", PB, 2 * 6 * 8, sm)
    print(f"lmm: {nblocks} column blocks of {PB} markers, {rounds} grid-stride rounds of {W} warps per full block")

    kind, seed = synth.KIND_DIPLOID, 43
    A0 = synth.block(seed, n, 0, 4000, kind)
    K = go.grm_simple(A0)
    rng = np.random.default_rng(seed)
    g = (A0 - A0.mean(axis=0)) @ rng.normal(size=A0.shape[1])
    g /= g.std()
    y = np.sqrt(0.5) * g + np.sqrt(0.5) * rng.normal(size=n)
    del A0

    # sampled markers: first and last of each block, ten in every grid-stride round, the generator's constant columns
    # of the second block
    fixed = synth.column_params(seed, np.arange(p, dtype=np.uint64))[1]
    picks = []
    for b in range(nblocks):
        s, pb = b * PB, min(PB, p - b * PB)
        picks += [s, s + pb - 1]
        for r in range((pb + W - 1) // W):
            lo_, hi_ = r * W, min((r + 1) * W, pb)
            picks += list(s + rng.integers(lo_, hi_, 10))
    blk2 = np.arange(PB, 2 * PB)
    picks += list(blk2[fixed[blk2]][:4])
    cols = np.unique(np.array(picks, dtype=np.int64))
    assert cols.size >= 190 and fixed[cols[(cols >= PB) & (cols < 2 * PB)]].any()
    As = np.column_stack([synth.block(seed, n, int(j), 1, kind)[:, 0] for j in cols])
    ref = lo.lmm_scan(As, y, K)

    dm = gbm.DeviceMatrix.generate(seed, n, p, kind)
    pk = dm.pack()
    assert pk is not None
    keep = dm.colstats()["keep"]
    assert np.array_equal(keep, ~fixed)
    assert np.array_equal(ref["keep"], keep[cols])
    plan = gbm.LmmPlan(K, y)
    assert abs(plan.null_log_delta - ref["lam0"]) < 1e-8
    results = {"float64": _lmm_run_into_sentinels(gbm, plan, dm), "codes": _lmm_run_into_sentinels(gbm, plan, pk)}
    plan.free()
    dm.free()
    pk.free()

    sdv = As.std(axis=0, ddof=1)
    k = ref["keep"]
    zs = max(1.0, np.abs(ref["z"][k]).max())
    for name, res in results.items():
        for key, v in res.items():  # every marker written: finite when kept, NaN when filtered
            assert np.all(np.isfinite(v[keep])) and np.all(np.isnan(v[~keep])), (name, key)
        got = {key: v[cols] for key, v in res.items()}
        assert np.max(np.abs(got["log_delta"][k] - ref["log_delta"][k])) < 1e-7, name
        assert np.max(np.abs(got["stat"][k] - ref["z"][k])) < 1e-9 * zs, name
        np.testing.assert_allclose(got["beta"][k], ref["beta"][k] * sdv[k], rtol=1e-7, atol=1e-10)
        np.testing.assert_allclose(got["se"][k], ref["se"][k] * sdv[k], rtol=1e-8)
