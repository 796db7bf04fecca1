"""Host-side mirror of the reference's GWAS API for the hot path, same names, keyword
arguments and error behaviour:

    gwasprep   /root/reference/src/gwas.jl:77-142
    gwasols    /root/reference/src/gwas.jl:206-259
    gwaslmm    /root/reference/src/gwas.jl:329-399
    extractxyetc (row filter + validation)  /root/reference/src/prediction.jl:53-139
    grmsimple / grmploidyaware (GenomicBreedingCore; call sites gwas.jl:120, :124)

The Julia shim (../julia/GenomicBreedingModelsB200.jl) has the same structure over the same
C ABI; this module is the one that can run in an image without Julia.  Only O(n) and
label bookkeeping happens here -- every O(n*p) / O(n^2*p) / O(n^3) step is a call into
libgbm_b200.so, and there is no CPU fallback.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from ._lib import ArgumentError, ErrorException
from .core import DeviceMatrix, LmmPlan, kstd_pc1
from .structs import GRM, Fit, Genomes, Phenomes

GRM_TYPES = ("simple", "ploidy-aware")
_EPS = float(np.finfo(np.float64).eps)


# --------------------------------------------------------------------------------------
def _validate_and_select(genomes: Genomes, phenomes: Phenomes, idx_entries, idx_loci_alleles, idx_trait: int):
    """Argument checks and the phenotype row filter of extractxyetc
    (/root/reference/src/prediction.jl:67-127).  Returns (rows1, cols1, y): 1-based row and
    column index vectors (None = all) and the filtered phenotype vector."""
    if not genomes.checkdims() and not phenomes.checkdims():  # :67-69
        raise ArgumentError("The Genomes and Phenomes structs are corrupted ☹.")
    if not genomes.checkdims():  # :70-72
        raise ArgumentError("The Genomes struct is corrupted ☹.")
    if not phenomes.checkdims():  # :73-75
        raise ArgumentError("The Phenomes struct is corrupted ☹.")
    if list(genomes.entries) != list(phenomes.entries):  # :76-78
        raise ArgumentError("The genomes and phenomes input need to have been merged to have consitent entries.")
    n0, p0 = genomes.allele_frequencies.shape
    all_rows = idx_entries is None
    if all_rows:  # :79-80
        idx_entries = np.arange(1, n0 + 1, dtype=np.int64)
    else:
        idx_entries = np.asarray(idx_entries, dtype=np.int64)
        if idx_entries.size == 0 or idx_entries.min() < 1 or idx_entries.max() > n0:  # :82-94
            raise ArgumentError(
                "The indexes of the entries, `idx_entries` are out of bounds. Expected range: from 1 to "
                f"{n0} while the supplied range is from "
                f"{idx_entries.min() if idx_entries.size else 'n/a'} to {idx_entries.max() if idx_entries.size else 'n/a'}.")
    if idx_loci_alleles is not None:  # :96-111
        idx_loci_alleles = np.asarray(idx_loci_alleles, dtype=np.int64)
        if idx_loci_alleles.size == 0 or idx_loci_alleles.min() < 1 or idx_loci_alleles.max() > p0:
            raise ArgumentError(
                "The indexes of the loci_alleles, `idx_loci_alleles` are out of bounds. Expected range: from 1 to "
                f"{p0} while the supplied range is from "
                f"{idx_loci_alleles.min() if idx_loci_alleles.size else 'n/a'} to "
                f"{idx_loci_alleles.max() if idx_loci_alleles.size else 'n/a'}.")
    if not (1 <= idx_trait <= phenomes.phenotypes.shape[1]):
        raise ArgumentError("`idx_trait` is out of bounds.")  # Julia: BoundsError at :114
    phi = np.asarray(phenomes.phenotypes, dtype=np.float64)[idx_entries - 1, idx_trait - 1]  # :114
    idx = np.flatnonzero(np.isfinite(phi))  # :116
    if idx.size < 2:  # :117-123
        raise ArgumentError(
            "There are less than 2 entries with non-missing phenotype data after merging with the genotype data.")
    y = phi[idx].copy()  # :124
    if np.var(y, ddof=1) < 1e-20:  # :125-127
        raise ErrorException("Very low or zero variance in trait: `" + phenomes.traits[idx_trait - 1] + "`.")
    rows1 = idx_entries[idx]
    if all_rows and idx.size == n0:
        rows1 = None
    return rows1, idx_loci_alleles, y


def extractxyetc(genomes: Genomes, phenomes: Phenomes, idx_entries=None, idx_loci_alleles=None, idx_trait: int = 1,
                 add_intercept: bool = True):
    """extractxyetc (/root/reference/src/prediction.jl:53-139).  Returns
    (X, y, entries, populations, loci_alleles) with X a host array; the GWAS functions below
    do not call this (they keep G on the device) -- it exists for API completeness."""
    rows1, cols1, y = _validate_and_select(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)
    A = np.asarray(genomes.allele_frequencies, dtype=np.float64)
    r0 = np.arange(A.shape[0]) if rows1 is None else rows1 - 1
    c0 = np.arange(A.shape[1]) if cols1 is None else cols1 - 1
    G = np.asfortranarray(A[np.ix_(r0, c0)])
    if np.isnan(G).any():
        raise ErrorException("cannot convert a value of type Missing to Float64")  # :129
    entries = [genomes.entries[i] for i in r0]
    populations = [genomes.populations[i] for i in r0]
    loci_alleles = [genomes.loci_alleles[j] for j in c0]
    if add_intercept:
        G = np.asfortranarray(np.hstack([np.ones((G.shape[0], 1)), G]))
    return G, y, entries, populations, loci_alleles


# --------------------------------------------------------------------------------------
def _grm_of(dm: DeviceMatrix, GRM_type: str, ploidy: int | None, centre: bool = True) -> np.ndarray:
    if GRM_type == "ploidy-aware":
        K, _ = dm.grm(_lib.GRM_PLOIDY_AWARE, int(ploidy), 0)
    else:
        K, _ = dm.grm(_lib.GRM_SIMPLE, 2, 0 if centre else _lib.GRM_NO_CENTRE)
    return K


def grmsimple(genomes: Genomes, idx_entries=None, idx_loci_alleles=None, centre: bool = True, verbose: bool = False) -> GRM:
    """grmsimple(genomes) (call site /root/reference/src/gwas.jl:124).  PARITY UNPINNED:
    GenomicBreedingCore source is absent; defined as (A - 1 mu')(A - 1 mu')'/p
    (``centre=False``: A A'/p, the recalled upstream variant)."""
    if not genomes.checkdims():
        raise ArgumentError("The Genomes struct is corrupted ☹.")
    A = np.asarray(genomes.allele_frequencies, dtype=np.float64)
    dm = DeviceMatrix.upload(A, idx_entries, idx_loci_alleles)
    try:
        K = _grm_of(dm, "simple", None, centre)
    finally:
        dm.free()
    if np.isnan(K).any():
        raise ErrorException("cannot convert a value of type Missing to Float64")
    ent = genomes.entries if idx_entries is None else [genomes.entries[i - 1] for i in idx_entries]
    loc = genomes.loci_alleles if idx_loci_alleles is None else [genomes.loci_alleles[j - 1] for j in idx_loci_alleles]
    return GRM(list(ent), list(loc), K)


def grmploidyaware(genomes: Genomes, ploidy: int = 2, idx_entries=None, idx_loci_alleles=None, verbose: bool = False) -> GRM:
    """grmploidyaware(genomes; ploidy) (call site /root/reference/src/gwas.jl:120).
    PARITY UNPINNED; defined as ploidy (A - 1 q')(A - 1 q')' / sum_j q_j (1 - q_j)."""
    if not genomes.checkdims():
        raise ArgumentError("The Genomes struct is corrupted ☹.")
    A = np.asarray(genomes.allele_frequencies, dtype=np.float64)
    dm = DeviceMatrix.upload(A, idx_entries, idx_loci_alleles)
    try:
        K = _grm_of(dm, "ploidy-aware", ploidy)
    finally:
        dm.free()
    if np.isnan(K).any():
        raise ErrorException("cannot convert a value of type Missing to Float64")
    ent = genomes.entries if idx_entries is None else [genomes.entries[i - 1] for i in idx_entries]
    loc = genomes.loci_alleles if idx_loci_alleles is None else [genomes.loci_alleles[j - 1] for j in idx_loci_alleles]
    return GRM(list(ent), list(loc), K)


# --------------------------------------------------------------------------------------
class _Prep:
    """Device-resident state shared by gwasprep / gwasols / gwaslmm."""

    __slots__ = ("dm", "packed", "scan_dm", "y", "K", "pc1", "stats", "idx_cols", "entries", "populations",
                 "loci_alleles", "trait", "ploidy", "rows1", "cols1", "eig_ms")

    def free(self):
        if getattr(self, "packed", None) is not None:
            self.packed.free()
        if getattr(self, "dm", None) is not None:
            self.dm.free()


def _prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, standardise, need_kstd,
             need_pc1, use_packed: bool = True) -> _Prep:
    rows1, cols1, y = _validate_and_select(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)  # gwas.jl:93-100
    if GRM_type not in GRM_TYPES:  # :101-107
        raise ArgumentError("Unrecognised `GRM_type`. Please select from:\n\t‣ " + "\n\t‣ ".join(GRM_TYPES))
    trait = phenomes.traits[idx_trait - 1]
    if np.var(y, ddof=1) < _EPS:  # :109-111
        raise ArgumentError("No variance in the trait: " + trait + ".")
    A = np.asarray(genomes.allele_frequencies, dtype=np.float64)
    pr = _Prep()
    pr.rows1, pr.cols1 = rows1, cols1
    subset = rows1 is not None or cols1 is not None
    # G = allele_frequencies[rows, cols] goes straight to the device (prediction.jl:129).  Dosage data (every
    # element an exact ploidy level) is stored as one byte per genotype: the scan then reads 1/8 of the bytes
    # and the GRM runs exactly on the INT8 tensor cores.  Without subsetting the host cores pack on the way
    # (gbm_matrix_upload_compact: the Float64 matrix never crosses PCIe); with subsetting the gather runs on
    # the device and the gathered matrix is packed there.
    if not subset and use_packed:
        m = DeviceMatrix.upload_compact(A)
        pr.dm, pr.packed = (None, m) if m.packed else (m, None)
    else:
        pr.dm = DeviceMatrix.upload(A, rows1, cols1)
        pr.packed = pr.dm.pack() if use_packed else None
    try:
        return _prepare_resident(pr, genomes, phenomes, A, rows1, cols1, y, trait, subset, use_packed, GRM_type,
                                 standardise, need_kstd, need_pc1)
    except BaseException:
        pr.free()  # nothing of a failed preparation stays resident
        raise


def _prepare_resident(pr: _Prep, genomes, phenomes, A, rows1, cols1, y, trait, subset, use_packed, GRM_type, standardise,
                      need_kstd, need_pc1) -> _Prep:
    pr.scan_dm = pr.packed if pr.packed is not None else pr.dm
    pr.stats = pr.scan_dm.colstats()  # v = std(G, dims=1); idx_cols (:112-113)
    if np.isnan(pr.stats["sd"]).any():
        # Matrix{Float64}(::Matrix{Union{Float64,Missing}}) throws on a missing genotype
        # (prediction.jl:129); a NaN/Inf genotype shows up here as a NaN column sd.
        raise ErrorException("cannot convert a value of type Missing to Float64")
    pr.idx_cols = pr.stats["idx_cols"]
    r0 = np.arange(A.shape[0]) if rows1 is None else rows1 - 1
    c0 = np.arange(A.shape[1]) if cols1 is None else cols1 - 1
    pr.entries = [genomes.entries[i] for i in r0]
    pr.populations = [genomes.populations[i] for i in r0]
    pr.loci_alleles = [genomes.loci_alleles[c0[j - 1]] for j in pr.idx_cols]  # :115
    pr.trait = trait
    # GRM on the FULL genomes (:117-126; SURVEY.md F6)
    pr.ploidy = None
    full = pr.scan_dm if not subset else DeviceMatrix.upload(A)
    full_packed = None
    if subset and use_packed:
        full_packed = full.pack()
    try:
        if GRM_type == "ploidy-aware":
            pr.ploidy = int(round(1.0 / pr.stats["min_nonzero_kept"]))  # :119
        K = _grm_of(full_packed if full_packed is not None else full, GRM_type, pr.ploidy)
    finally:
        if full_packed is not None:
            full_packed.free()
        if full is not pr.scan_dm:
            full.free()
    pr.pc1, pr.eig_ms = None, 0.0
    if standardise:  # :127-131
        y = (y - y.mean()) / np.std(y, ddof=1)
        Ks, pc1, eig_ms = kstd_pc1(K, want_kstd=need_kstd, want_pc1=need_pc1)
        K = Ks if need_kstd else None
        pr.pc1, pr.eig_ms = pc1, eig_ms
    pr.y, pr.K = y, K
    return pr


def _new_fit(pr: _Prep) -> Fit:
    n, l = len(pr.entries), int(pr.idx_cols.size)  # :133
    fit = Fit.new(n, l)  # :134
    fit.model = ""
    fit.trait = pr.trait
    fit.b_hat_labels = list(pr.loci_alleles)
    fit.entries = list(pr.entries)
    fit.populations = list(pr.populations)
    fit.metrics = {"": 0.0}  # :140
    return fit


def gwasprep(*, genomes: Genomes, phenomes: Phenomes, idx_entries=None, idx_loci_alleles=None, idx_trait: int = 1,
             GRM_type: str = "simple", standardise: bool = True, verbose: bool = False):
    """gwasprep (/root/reference/src/gwas.jl:77-142): returns (G, y, GRM, fit) as host arrays
    like the reference.  G is materialised on the host only here (the scan functions below
    never do that)."""
    pr = _prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, standardise,
                  need_kstd=True, need_pc1=False)
    try:
        G = pr.scan_dm.download_cols(pr.idx_cols, standardise=standardise)  # :114, :129 on the device
        K = pr.K
        fit = _new_fit(pr)
    finally:
        pr.free()
    return np.asfortranarray(G), pr.y, K, fit


def _gwas_multigpu(group, model_name: str, model: int, genomes, phenomes, idx_trait, GRM_type, y, verbose) -> Fit:
    """gwasols / gwaslmm on a group of GPUs (GBM_NUM_GPUS > 1): markers sharded by column block, ONE collective
    call into the library (gbm_sharded_upload + gbm_sharded_gwas); same Fit as the single-GPU path."""
    from .multigpu import ShardedMatrix

    A = np.asarray(genomes.allele_frequencies, dtype=np.float64)
    sm = ShardedMatrix.upload(group, A, compact=True)
    try:
        ys = (y - y.mean()) / np.std(y, ddof=1)  # gwas.jl:128
        res = sm.gwas(ys, model=model,
                      grm_type=_lib.GRM_PLOIDY_AWARE if GRM_type == "ploidy-aware" else _lib.GRM_SIMPLE)
        packed = sm.packed
    finally:
        sm.free()
    idx_cols = res["idx_cols"].copy()
    sel = idx_cols - 1
    if np.isnan(res["stat"][sel]).all() and np.isnan(A).any():
        raise ErrorException("cannot convert a value of type Missing to Float64")
    fit = Fit.new(A.shape[0], int(idx_cols.size))  # gwas.jl:133-140
    fit.model = model_name
    fit.trait = phenomes.traits[idx_trait - 1]
    fit.b_hat_labels = [genomes.loci_alleles[j] for j in sel]
    fit.entries = list(genomes.entries)
    fit.populations = list(genomes.populations)
    fit.metrics = {"": 0.0}
    b = res["stat"][sel]
    if model == _lib.MODEL_LMM:
        b = np.where(np.isnan(b), 0.0, b)  # failed fits leave 0.0 (:367-382)
    fit.b_hat = np.ascontiguousarray(b)
    tm = res["timing"]
    fit.extras = {"beta": res["beta"][sel], "se": res["se"][sel], "neglog10p": res["neglog10p"][sel],
                  "pvalue": np.power(10.0, -res["neglog10p"][sel]), "idx_cols": idx_cols, "pc1": res["pc1"].copy(),
                  "ploidy": tm["ploidy"] if GRM_type == "ploidy-aware" else None, "eig_ms": tm["eig_ms"], "timing": tm,
                  "storage": "u8 dosage codes" if packed else "float64", "n_gpus": group.world}
    if not fit.checkdims():
        raise ErrorException(f"Error performing GWAS via {model_name[5:]} using the {GRM_type} GRM.")
    return fit


def _gwas(model_name: str, model: int, genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type,
          verbose) -> Fit:
    from .multigpu import default_group

    group = default_group()  # GBM_NUM_GPUS > 1
    if group is not None:
        rows1, cols1, y = _validate_and_select(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)
        if GRM_type not in GRM_TYPES:
            raise ArgumentError("Unrecognised `GRM_type`. Please select from:\n\t‣ " + "\n\t‣ ".join(GRM_TYPES))
        if np.var(y, ddof=1) < _EPS:
            raise ArgumentError("No variance in the trait: " + phenomes.traits[idx_trait - 1] + ".")
        if rows1 is None and cols1 is None and np.shape(genomes.allele_frequencies)[1] >= group.world:
            return _gwas_multigpu(group, model_name, model, genomes, phenomes, idx_trait, GRM_type, y, verbose)
    pr = _prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, True, need_kstd=False,
                  need_pc1=True)  # gwas.jl:221-230 / :344-353, PCA :234 / :357
    try:
        if len(pr.entries) != pr.pc1.shape[0]:
            # SURVEY.md F6: the reference's hcat (:241) throws when entries were dropped
            raise ArgumentError(
                "The GRM is computed on all entries of `genomes` (gwas.jl:120,:124) but some entries were dropped "
                "(idx_entries or missing phenotypes): the covariate PC1 and G have different numbers of rows.")
        fit = _new_fit(pr)
        fit.model = model_name  # :231 / :354
        res = pr.scan_dm.scan(pr.y, pr.pc1[:, None], model=model)  # marker loop :239-249 / :363-389
        sel = pr.idx_cols - 1
        b = res["stat"][sel, 0]
        if model == _lib.MODEL_LMM:
            b = np.where(np.isnan(b), 0.0, b)  # failed fits leave 0.0 (:367-382)
        fit.b_hat = np.ascontiguousarray(b)
        fit.extras = {
            "beta": res["beta"][sel, 0], "se": res["se"][sel, 0], "neglog10p": res["neglog10p"][sel, 0],
            "pvalue": np.power(10.0, -res["neglog10p"][sel, 0]), "idx_cols": pr.idx_cols, "pc1": pr.pc1,
            "ploidy": pr.ploidy, "eig_ms": pr.eig_ms, "timing": _lib.last_timing(),
            "storage": "u8 dosage codes" if pr.packed is not None else "float64",
        }
        if verbose:
            lod = fit.extras["neglog10p"]
            thr = -np.log10(0.05 / max(len(lod), 1))
            print(f"{model_name} using {GRM_type} GRM: {len(lod)} loci-alleles, max -log10(p) = {np.nanmax(lod):.3f}, "
                  f"{int(np.sum(lod > thr))} above the Bonferroni threshold {thr:.3f}")
        if not fit.checkdims():  # :255-257 / :395-397
            raise ErrorException(f"Error performing GWAS via {model_name[5:]} using the {GRM_type} GRM.")
        return fit
    finally:
        pr.free()


def gwasols(*, genomes: Genomes, phenomes: Phenomes, idx_entries=None, idx_loci_alleles=None, idx_trait: int = 1,
            GRM_type: str = "simple", verbose: bool = False) -> Fit:
    """gwasols (/root/reference/src/gwas.jl:206-259): fit.b_hat[j] = b[end]/sqrt(Vinv[end,end])."""
    return _gwas("GWAS_OLS", _lib.MODEL_OLS, genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type,
                 verbose)


def gwaslmm(*, genomes: Genomes, phenomes: Phenomes, idx_entries=None, idx_loci_alleles=None, idx_trait: int = 1,
            GRM_type: str = "simple", verbose: bool = False) -> Fit:
    """gwaslmm (/root/reference/src/gwas.jl:329-399): fit.b_hat[j] = z of `x` in
    y ~ 1 + PC1 + x + (1|entries) fitted by REML (closed form, SURVEY.md Appendix A.3)."""
    return _gwas("GWAS_LMM", _lib.MODEL_LMM, genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type,
                 verbose)


def _gwasreml_multigpu(group, genomes, phenomes, idx_trait, GRM_type, y, objective) -> Fit:
    """gwasreml on a group of GPUs (GBM_NUM_GPUS > 1): markers sharded by column block, ONE collective call into the
    library (gbm_sharded_upload + gbm_sharded_gwasreml); the same Fit as the single-GPU path, plus timing, n_gpus and
    storage in extras."""
    from .multigpu import ShardedMatrix

    A = np.asarray(genomes.allele_frequencies, dtype=np.float64)
    # the single-GPU path's y: standardised once for REML; for the reference objective gwasprep standardises it
    # (gwas.jl:128) and gwasreml once more
    ys = (y - y.mean()) / np.std(y, ddof=1)
    if objective == "reference":
        ys = (ys - ys.mean()) / np.std(ys, ddof=1)
    sm = ShardedMatrix.upload(group, A, compact=True)
    try:
        res = sm.gwasreml(ys, grm_type=_lib.GRM_PLOIDY_AWARE if GRM_type == "ploidy-aware" else _lib.GRM_SIMPLE,
                          objective=objective)
        packed = sm.packed
    finally:
        sm.free()
    idx_cols = res["idx_cols"]
    sel = idx_cols - 1
    if np.isnan(res["stat"][sel]).all() and np.isnan(A).any():
        raise ErrorException("cannot convert a value of type Missing to Float64")
    fit = Fit.new(A.shape[0], int(idx_cols.size))  # gwas.jl:133-140
    fit.model = "GWAS_REML"  # :574
    fit.trait = phenomes.traits[idx_trait - 1]
    fit.b_hat_labels = [genomes.loci_alleles[j] for j in sel]
    fit.entries = list(genomes.entries)
    fit.populations = list(genomes.populations)
    fit.metrics = {"": 0.0}
    fit.b_hat = np.ascontiguousarray(res["stat"][sel])
    tm = res["timing"]
    fit.extras = {"beta": res["beta"][sel], "se": res["se"][sel], "neglog10p": res["neglog10p"][sel],
                  "log_delta": res["log_delta"][sel], "null_log_delta": res["null_log_delta"], "idx_cols": idx_cols,
                  "eig_ms": tm["eig_ms"], "gemm_tflops": tm["rotation_tflops"], "search_ms": tm["search_ms"],
                  "ploidy": tm["ploidy"] if GRM_type == "ploidy-aware" else None, "objective": objective, "timing": tm,
                  "n_gpus": group.world, "storage": "u8 dosage codes" if packed else "float64"}
    if not fit.checkdims():  # :609-611
        raise ErrorException("Error performing GWAS via REML using the " + GRM_type + " GRM.")
    return fit


def gwasreml(*, genomes: Genomes, phenomes: Phenomes, idx_entries=None, idx_loci_alleles=None, idx_trait: int = 1,
             GRM_type: str = "simple", verbose: bool = False, objective: str = "reml") -> Fit:
    """gwasreml (/root/reference/src/gwas.jl:549-613): per-marker LMM with the GRM as the
    covariance of the random genotype effect, variance components re-estimated for every
    marker, fit.b_hat[j] = b[end]/sqrt(inv(X'V^-1 X)[end]) with X = [1, g_j] (:586, :596-599).

    Engine: eigen-rotation (cuSOLVER + FP64 DMMA GEMM) and a per-marker search on the device.
    ``objective`` (an extension; the reference has no such keyword):

    * ``"reml"`` (default): the standard REML log-likelihood on the symmetric un-standardised GRM, z with the
      profiled sigma^2 -- a proper LMM test statistic.
    * ``"reference"``: the reference's OWN objective, box and statistic (`0.5 log det V + y'Py + log det X'V^-1X`
      over [eps, 1]^2, no sigma^2 factor; :478, :588, :596-599) on the symmetric part of the column-standardised K
      that gwasprep hands to loglikreml (:130, :564-573) -- as close as a rotation-based engine can get; the
      non-symmetric part of that K and the L-BFGS path are what remains (oracle/lmm_oracle.py, DESIGN.md section 2).
    PARITY UNPINNED either way.

    With ``GBM_NUM_GPUS`` > 1 and no entries or loci subset, the markers are sharded over that many GPUs: one
    eigendecomposition on the first GPU, broadcast, every GPU rotates and searches its own markers."""
    if objective not in ("reml", "reference"):
        raise ArgumentError("objective must be \"reml\" or \"reference\"")
    ref = objective == "reference"
    from .multigpu import default_group

    group = default_group()  # GBM_NUM_GPUS > 1
    if group is not None:
        rows1, cols1, y = _validate_and_select(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)
        if GRM_type not in GRM_TYPES:
            raise ArgumentError("Unrecognised `GRM_type`. Please select from:\n\t‣ " + "\n\t‣ ".join(GRM_TYPES))
        if np.var(y, ddof=1) < _EPS:
            raise ArgumentError("No variance in the trait: " + phenomes.traits[idx_trait - 1] + ".")
        if rows1 is None and cols1 is None and np.shape(genomes.allele_frequencies)[1] >= group.world:
            return _gwasreml_multigpu(group, genomes, phenomes, idx_trait, GRM_type, y, objective)
    pr = _prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, ref, need_kstd=ref,
                  need_pc1=False)  # gwas.jl:564-573 (reml: K stays symmetric, standardise=False)
    try:
        if len(pr.entries) != pr.K.shape[0]:
            raise ArgumentError(
                "The GRM is computed on all entries of `genomes` (gwas.jl:120,:124) but some entries were dropped: "
                "y and the GRM have different sizes.")
        fit = _new_fit(pr)
        fit.model = "GWAS_REML"  # :574
        y = (pr.y - pr.y.mean()) / np.std(pr.y, ddof=1)  # :128 (the REML z is invariant to it; the reference box is not)
        K = 0.5 * (pr.K + pr.K.T) if ref else pr.K
        plan = LmmPlan(K, y)
        try:
            res = plan.run(pr.scan_dm, flags=_lib.LMM_REFERENCE_OBJECTIVE if ref else 0)
        finally:
            plan.free()
        sel = pr.idx_cols - 1
        fit.b_hat = np.ascontiguousarray(res["stat"][sel])
        fit.extras = {"beta": res["beta"][sel], "se": res["se"][sel], "neglog10p": res["neglog10p"][sel],
                      "log_delta": res["log_delta"][sel], "null_log_delta": plan.null_log_delta,
                      "idx_cols": pr.idx_cols, "eig_ms": plan.eig_ms, "gemm_tflops": res["gemm_tflops"],
                      "search_ms": res["search_ms"], "ploidy": pr.ploidy, "objective": objective}
        if not fit.checkdims():  # :609-611
            raise ErrorException("Error performing GWAS via REML using the " + GRM_type + " GRM.")
        return fit
    finally:
        pr.free()
