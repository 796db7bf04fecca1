/* gbm_b200.h -- C ABI of libgbm_b200.so: the B200 (sm_100a) implementation of the
 * GWAS-scan / GRM hot path of GenomicBreedingModels.jl v0.3.0.
 *
 * The reference has no FFI layer of its own (pure Julia).  Its boundary for this path is
 * the exported keyword API
 *     gwasprep  /root/reference/src/gwas.jl:77-142
 *     gwasols   /root/reference/src/gwas.jl:206-259
 *     gwaslmm   /root/reference/src/gwas.jl:329-399
 * plus GenomicBreedingCore's grmsimple / grmploidyaware (call sites gwas.jl:120, :124).
 * The entry points below are what a Julia `ccall` shim binds so that those functions keep
 * their signatures (INTEGRATION.md shows the shim); each one cites the reference lines it
 * replaces.
 *
 * Conventions
 *  - every function returns 0 (GBM_OK) or an error code; gbm_last_error() has the text.
 *    GBM_ERR_ARGUMENT maps to Julia ArgumentError, GBM_ERR_RUNTIME to ErrorException.
 *  - matrices are column-major Float64 (Julia layout).  Indices returned are 1-based Int64.
 *  - every `double*`, `int64_t*`, `uint8_t*` data argument may be a HOST pointer (pageable or
 *    pinned) or a DEVICE pointer of the selected GPU; the library tells them apart
 *    (unified virtual addressing).  Host pointers are never retained after return.
 *  - device memory is library-owned behind the opaque gbm_matrix handle.
 *  - gbm_init(device) selects one GPU for the single-GPU entry points.  Multi-GPU runs go through a
 *    gbm_group (section "multi-GPU" below): markers sharded by column block over the GPUs of one box,
 *    either all driven by this process (gbm_group_create_local: one host thread per GPU inside the
 *    library, what a Julia session uses) or one process per GPU (gbm_group_create_rank: torchrun / MPI).
 *    NCCL lives inside the library; the caller never issues a collective.
 *  - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef GBM_B200_H
#define GBM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GBM_ABI_VERSION 3

#define GBM_OK 0
#define GBM_ERR_ARGUMENT 1 /* Julia ArgumentError */
#define GBM_ERR_RUNTIME 2  /* Julia ErrorException */
#define GBM_ERR_CUDA 3     /* CUDA / cuSOLVER failure */
#define GBM_ERR_NOT_INITIALISED 4

/* GRM_type string enum of gwasprep (gwas.jl:101-107) */
#define GBM_GRM_SIMPLE 0
#define GBM_GRM_PLOIDY_AWARE 1
/* gbm_grm flags */
#define GBM_GRM_NO_CENTRE 1 /* simple GRM as A*A'/p (recalled upstream variant), default is centred */

/* scan models */
#define GBM_MODEL_OLS 0 /* gwasols statistic, p-values from TDist(n-1)   (gwas.jl:245, :252) */
#define GBM_MODEL_LMM 1 /* gwaslmm z statistic, p-values from Normal()   (gwas.jl:385, :392) */
/* scan flags */
#define GBM_PVALUE_TWO_SIDED 1 /* default is the one-sided upper tail of |stat| */
#define GBM_SCAN_HOST_NO_PACK 4 /* gbm_scan_host: never pack blocks to 1-byte codes, every block crosses PCIe and is
                                   scanned as Float64 (default: blocks that are all dosage codes are packed) */

/* synthetic generator kinds (oracle/synth.py defines the arithmetic) */
#define GBM_KIND_DIPLOID 0
#define GBM_KIND_TETRAPLOID 1
#define GBM_KIND_CONTINUOUS 2

typedef struct gbm_matrix gbm_matrix; /* n x p column-major Float64 slab resident in HBM */

/* timings of the last call, CUDA events on the library stream (milliseconds) */
typedef struct gbm_timing {
  double h2d_ms;    /* host -> device copies                        */
  double kernel_ms; /* all kernels of the call                      */
  double main_ms;   /* the dominant kernel alone (scan sums / DMMA) */
  double d2h_ms;    /* device -> host copies                        */
  int64_t launches; /* kernels launched by the call                 */
  int64_t packed_blocks; /* gbm_scan_host: column blocks scanned as 1-byte codes (all elements are codes) */
  int64_t host_packed_blocks; /* ... of which packed by the host cores, i.e. crossed PCIe as 1 byte per genotype;
                                 the others crossed as Float64 and were packed on the device */
  int64_t h2d_bytes; /* gbm_scan_host: genotype bytes that crossed PCIe */
} gbm_timing;

/* ---- life cycle ------------------------------------------------------------------- */
int gbm_abi_version(void);
const char* gbm_last_error(void);
int gbm_init(int device);            /* selects the GPU, creates stream + cuSOLVER handle   */
int gbm_shutdown(void);
int gbm_set_stream(void* cuda_stream); /* run on the caller's cudaStream_t (NULL: own stream) */
int gbm_synchronize(void);
int gbm_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes, char* name, int name_len);
int gbm_last_timing(gbm_timing* t);

/* ---- genotype matrix handles: replaces the n x p copy `G::Matrix{Float64} =
 *      genomes.allele_frequencies[rows, cols]` of extractxyetc
 *      (/root/reference/src/prediction.jl:129) -------------------------------------- */
/* A: n x p column-major with leading dimension lda (host or device). The device copy is
 * re-pitched to a 128-byte multiple.  Page-locked and device sources go through the copy engine
 * directly; a PAGEABLE source (a Julia Array) is copied by the calling process' cores into a ring of
 * pinned staging blocks that the copy engine drains. */
int gbm_matrix_upload(const double* A, int64_t n, int64_t p, int64_t lda, gbm_matrix** out);
/* Same, but the host cores first try to pack the matrix to 1-byte dosage codes (exactness-checked,
 * see "Compact storage" below): when EVERY element is a code the handle holds the codes (*packed = 1;
 * 1/8 of the bytes cross PCIe and live in HBM, results equal the Float64 path's), otherwise the
 * Float64 slab as gbm_matrix_upload (*packed = 0; the attempt stops at the first non-code element). */
int gbm_matrix_upload_compact(const double* A, int64_t n, int64_t p, int64_t lda, gbm_matrix** out, int* packed);
/* gather upload: rows[i] / cols[j] are 1-based indices into the n0 x p0 source (either may
 * be NULL = all); this is allele_frequencies[idx_entries[idx], idx_loci_alleles]. */
int gbm_matrix_upload_indexed(const double* A, int64_t n0, int64_t p0, int64_t lda, const int64_t* rows,
                              int64_t n, const int64_t* cols, int64_t p, gbm_matrix** out);
/* wrap an existing device buffer (not owned, not freed). lda must be even. */
int gbm_matrix_wrap(double* dA, int64_t n, int64_t p, int64_t lda, gbm_matrix** out);
/* synthetic columns col0 .. col0+p-1 of the counter-based generator, made on the device */
int gbm_matrix_generate(uint64_t seed, int64_t n, int64_t p, int64_t col0, int kind, gbm_matrix** out);
/* Compact storage (SURVEY.md 8f rank 3): one byte per genotype, code c in [0,240], a = c/240.
 * gbm_matrix_pack converts a resident Float64 matrix; *out is set only when EVERY element is
 * exactly a code (fl(c/240) == a), otherwise *out = NULL and *n_inexact > 0 (use the Float64
 * matrix).  Packed handles work with gbm_colstats, gbm_scan*, gbm_grm*, gbm_lmm_plan_run and
 * gbm_matrix_download (which returns Float64); results equal the Float64 path's.
 * gbm_matrix_upload_packed takes codes that are already compact on the host (n x p, pitch ld). */
int gbm_matrix_pack(const gbm_matrix* m, gbm_matrix** out, int64_t* n_inexact);
int gbm_matrix_upload_packed(const uint8_t* codes, int64_t n, int64_t p, int64_t ld, gbm_matrix** out);
/* multi-threaded host packer (all cores of the calling process' affinity mask) */
int gbm_pack_host(const double* A, int64_t n, int64_t p, int64_t lda, uint8_t* out, int64_t ldo, int64_t* n_inexact);
/* testing hook: col_ok[j] = 1 when the packer body of ISA level `isa` (0 scalar, 1 AVX2+FMA, 2 AVX-512)
 * accepts column j as all-codes; the vector bodies use a division-free test that must agree with
 * fl(c/240) == a element for element */
int gbm_pack_host_check(const double* A, int64_t n, int64_t p, int64_t lda, int isa, uint8_t* col_ok);
/* testing hook (host only, no GPU needed): the fixed-point form of the side vectors that the tensor-core code scan
 * multiplies (csrc/scan_u8_tc.cu).  Q: n x M (ldq), M <= 2.  digits: 16 x ld int8 with ld = n rounded up to 128 --
 * row 0 ones, rows 1..7 / 8..14 the seven balanced base-256 digits of q_1 / q_2 (least significant first), zero padded;
 * scale[m] = 2^(E_m - 55): q_i = scale * sum_k 256^k digit_k(i) up to one ulp of max |q|. */
int gbm_side_vector_digits(const double* Q, int64_t n, int M, int64_t ldq, int8_t* digits, int64_t ld, double* scale);
/* testing hook (host only, no GPU needed): the host half of the Lanczos PC1 solver (csrc/lanczos.cu) -- largest
 * eigenvalue theta (Sturm bisection) and unit eigenvector s (inverse iteration) of the m x m symmetric tridiagonal with
 * diagonal alpha[0..m) and off-diagonal beta[0..m-1); the solver's stopping test is |beta_m s_m| <= tol theta. */
int gbm_tridiag_top(const double* alpha, const double* beta, int64_t m, double* theta, double* s);
int gbm_matrix_download(const gbm_matrix* m, int64_t j0, int64_t ncols, double* dst, int64_t ldd);
/* G = G[:, idx_cols] and, with standardise != 0, G = (G .- mean(G, dims=1)) ./ std(G, dims=1)'
 * (/root/reference/src/gwas.jl:114, :129) on the device; dst (host or device) is n x ncols.
 * idx_cols: 1-based, NULL = all columns. */
int gbm_matrix_download_cols(const gbm_matrix* m, const int64_t* idx_cols, int64_t ncols, int standardise,
                             double* dst, int64_t ldd);
int gbm_matrix_info(const gbm_matrix* m, int64_t* n, int64_t* p, int64_t* lda, double** device_ptr);
int gbm_matrix_free(gbm_matrix* m);

/* ---- gwasprep: fixed-locus filter and ploidy inference ------------------------------
 * v = std(G, dims=1); idx_cols = findall(v > eps && finite)   (gwas.jl:112-113)
 * minimum(G[G .!= 0.0]) over kept columns                     (gwas.jl:119)
 * All outputs nullable. mean/sd/min_nonzero/keep have length p; idx_cols has room for p
 * entries, *n_keep receives l. ploidy = Int(round(1/min_nonzero_kept)). */
int gbm_colstats(const gbm_matrix* m, double* mean, double* sd, double* min_nonzero, uint8_t* keep,
                 int64_t* idx_cols, int64_t* n_keep, double* min_nonzero_kept);

/* ---- GRM: grmsimple(genomes) / grmploidyaware(genomes; ploidy)  (gwas.jl:120, :124) ---
 * K (n x n, column-major, host or device) receives the full symmetric matrix.
 *   simple       : (A - 1 mu')(A - 1 mu')' / p          (GBM_GRM_NO_CENTRE: A A' / p)
 *   ploidy-aware : ploidy (A - 1 q')(A - 1 q')' / sum_j q_j (1 - q_j)
 * tflops (nullable) receives n(n+1)p / time of the DMMA kernel. */
int gbm_grm(const gbm_matrix* m, int grm_type, int ploidy, int flags, double* K, double* tflops);
/* marker-sharded form: dK (DEVICE, n x n, zeroed by the caller or holding earlier partials)
 * += lower triangle of sum_j (a_j - mu_j)(a_j - mu_j)' over this shard's columns;
 * *sum_q1mq += sum_j q_j (1 - q_j).  After an all-reduce of dK (and the two scalars) over
 * the ranks, gbm_grm_finalize scales and mirrors. */
int gbm_grm_accumulate(const gbm_matrix* m, int centre, double* dK, double* sum_q1mq, double* tflops);
int gbm_grm_finalize(double* dK, int64_t n, double scale);

/* ---- K standardisation + PC1 ---------------------------------------------------------
 * Kstd = (K .- mean(K, dims=1)) ./ std(K, dims=1)               (gwas.jl:130)
 * pc1  = MultivariateStats.fit(PCA, Kstd; maxoutdim=1).proj[:,1] (gwas.jl:234, :357):
 *        rows centred, top left singular vector (unit norm, sign arbitrary).  Only this one vector is
 *        needed, so n >= 1024 uses Lanczos with full reorthogonalisation on the operator Z Z' (Z = the
 *        row-centred Kstd; never formed: one fused pass over Z per step, the whole reorthogonalisation in one
 *        cooperative kernel (GBM_PC1_NO_COOP=1: five launches), csrc/lanczos.cu; residual
 *        ||Z Z'x - theta x|| <= 5e-13 theta), smaller or non-converging problems and GBM_PC1_SOLVER=cusolver use
 *        cusolverDnDsyevdx.  K host or device; Kstd nullable; eig_ms (nullable) = time of the eigen step alone.
 *        Multi-GPU form: gbm_sharded_kstd_pc1 (columns of K sharded over the group). */
int gbm_kstd_pc1(const double* K, int64_t n, double* Kstd, double* pc1, double* eig_ms);

/* ---- the marker scan: the loops of gwasols (gwas.jl:239-249) and gwaslmm (:363-389) ---
 * Y : n x T phenotypes (ldy), used as given (the caller standardises, gwas.jl:128)
 * C : n x k covariates WITHOUT the intercept (ldc), k >= 0; the reference uses k = 1 (PC1)
 * Per marker j and trait t, with M the projector off [1, C] and g_j the standardised
 * column (gwas.jl:129):
 *   beta  = coefficient of g_j               se = its standard error
 *   stat  = GBM_MODEL_OLS: b[end]/sqrt(Vinv[end,end])           (gwas.jl:245)
 *           GBM_MODEL_LMM: z of `x` in y ~ 1 + PC1 + x + (1|entries), REML (gwas.jl:358-385)
 *   neglog10p = -log10 P(D > |stat|), D = TDist(n-1) resp. Normal()   (gwas.jl:252, :392)
 * Outputs (all nullable): beta, se, stat, neglog10p are p x T column-major (ld p);
 * mean, sd (length p) and keep (length p, the fixed-locus filter). Entries of filtered
 * or degenerate markers are NaN. */
int gbm_scan(const gbm_matrix* m, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k,
             int64_t ldc, int model, int flags, double* beta, double* se, double* stat, double* neglog10p,
             double* mean, double* sd, uint8_t* keep);

/* Reusable scan: side vectors (covariates orthonormalised, traits residualised) and
 * scratch are prepared once; every gbm_scan_plan_run is then the two kernel launches of one
 * pass over the resident matrix (streaming sums + finalisation).  Device output pointers are
 * written by the kernels in place, host ones are copied out.  The matrix handle must outlive
 * the plan.  gbm_scan == create + run + free. */
typedef struct gbm_scan_plan gbm_scan_plan;
int gbm_scan_plan_create(const gbm_matrix* m, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k,
                         int64_t ldc, int model, int flags, gbm_scan_plan** plan);
int gbm_scan_plan_run(gbm_scan_plan* plan, double* beta, double* se, double* stat, double* neglog10p, double* mean,
                      double* sd, uint8_t* keep);
int gbm_scan_plan_free(gbm_scan_plan* plan);

/* One call from host memory to results (the end-to-end path).  A is cut into ~128 MB column blocks
 * handed out dynamically to two lanes that run concurrently with the scan kernels:
 *  - host lane: the host cores pack a block to 1-byte dosage codes (exactness-checked) into pinned
 *    staging, so 1/8 of the bytes cross PCIe; it stops at the first block that is not all codes;
 *  - copy-engine lane (A page-locked, or the host lane unavailable): the block crosses PCIe as
 *    Float64 and is packed on the device.
 * A block that is all codes is scanned by the u8 kernel, any other block by the Float64 kernel,
 * whichever lane carried it, so the outputs do not depend on the scheduling.  Same outputs as
 * gbm_scan.  GBM_SCAN_HOST_NO_PACK: plain Float64 copies and the Float64 kernel only. */
int gbm_scan_host(const double* A, int64_t n, int64_t p, int64_t lda, const double* Y, int64_t T, int64_t ldy,
                  const double* C, int64_t k, int64_t ldc, int model, int flags, double* beta, double* se,
                  double* stat, double* neglog10p, double* mean, double* sd, uint8_t* keep);

/* ---- GRM-covariance LMM scan: the model of gwasreml / loglikreml ----------------------
 * (/root/reference/src/gwas.jl:450-483, :549-613: V = s2u*GRM + s2e*I, variance components
 * re-estimated for every marker, statistic b[end]/sqrt(inv(X'V^-1 X)[end]); restated as the
 * standard REML on the SYMMETRIC GRM -- oracle/lmm_oracle.py lists the differences.)
 * create: K = U S U' (cuSOLVER syevd, eig_ms), rotation of [1, C, y] by the DMMA GEMM,
 *         null-model log(delta) (returned in *null_log_delta).  K: n x n, host or device,
 *         lower triangle used; y: n; C: n x k, k <= 2 extra covariates (intercept implied).
 * run   : for the resident matrix m (n rows): U'A in column blocks by the FP64 DMMA GEMM,
 *         then one warp per marker searches delta = s2e/s2g (bracket marched from the null
 *         estimate, safeguarded Newton on dLL/dlog(delta)), and emits beta, se (of the
 *         standardised column), z, -log10 P(N(0,1) > |z|) and log(delta).  Outputs length p,
 *         host or device, nullable.  gemm_tflops: 2 n^2 p / DMMA GEMM time. */
/* gbm_lmm_plan_run flag: minimise the REFERENCE's own objective over its own box instead of the standard REML --
 * 0.5 log det V + y'Py + log det(X'V^-1X) (gwas.jl:478) over [s2e, s2u] in [eps, 1]^2 from [0.5, 0.5] (:578, :588),
 * statistic b[end] / sqrt(inv(X'V^-1X)[end]) with no sigma^2 factor (:596-599).  y must be standardised (the box is
 * absolute).  K must be symmetric to be rotated: pass the symmetric part of the column-standardised GRM to stay as
 * close as a rotation can to what the reference feeds loglikreml (csrc/lmm.cu has the algebra).  log_delta then
 * receives log(s2e / s2u), se = sqrt(s2u [ (X'WX)^-1 ]_xx). */
#define GBM_LMM_REFERENCE_OBJECTIVE 8
typedef struct gbm_lmm_plan gbm_lmm_plan;
int gbm_lmm_plan_create(const double* K, int64_t n, const double* y, const double* C, int64_t k, int64_t ldc,
                        gbm_lmm_plan** plan, double* eig_ms, double* null_log_delta);
int gbm_lmm_plan_run(gbm_lmm_plan* plan, const gbm_matrix* m, int flags, double* beta, double* se, double* stat,
                     double* neglog10p, double* log_delta, double* gemm_tflops, double* search_ms);
int gbm_lmm_plan_free(gbm_lmm_plan* plan);
/* C (M x N, ldc) = A' B, A: K x M (lda), B: K x N (ldb); column-major DEVICE buffers, lda and
 * ldb even, 16-byte aligned.  The rotation GEMM on its own. */
int gbm_gemm_tn(const double* dA, int64_t lda, const double* dB, int64_t ldb, double* dC, int64_t ldc, int64_t M,
                int64_t N, int64_t K, double* tflops);

/* ---- transformation screens (SURVEY.md 8f rank 4): the regressions of transform1 / transform2 /
 *      epistasisfeatures (/root/reference/src/transformation.jl:130-239, :319-466, :540-651) ----------
 * The reference calls `ols(genomes = g, phenomes = p)` ([1 f(x)] \ y, linear.jl:85) once per locus
 * (transform1) or once per ordered pair of loci (transform2: l^2 fits) and keeps b_hat[2].  `f` is one
 * of the package's named endofunctions (transformation.jl:1-55); an arbitrary Julia closure cannot
 * cross a C ABI, the shims raise ArgumentError for anything else. */
#define GBM_F1_SQUARE 0     /* square(x) = x^2                                            :9  */
#define GBM_F1_INVONEPLUS 1 /* invoneplus(x) = 1 / (1 + x)                                :18 */
#define GBM_F1_LOG10EPS 2   /* log10epsdivlog10eps(x) = log10(x + eps) / log10(eps)       :27 */
#define GBM_F2_MULT 0       /* mult(x, y) = x * y                                         :36 */
#define GBM_F2_ADDNORM 1    /* addnorm(x, y) = (x + y) / 2                                :45 */
#define GBM_F2_RAISE 2      /* raise(x, y) = x^y                                          :54 */
/* transform1 (:157-221): X .+= eps; use_abs -> abs.(X); beta[j] = slope of y ~ 1 + f(x_j), 0 when
 * var(x_j) < var_threshold; idx = sortperm(abs.(beta), rev = true)[1:n_new] filtered by abs(beta) > eps, in
 * that order (1-based).  y: n (host or device).  beta: p values, host or device, nullable.  idx: n_new slots. */
int gbm_transform1_screen(const gbm_matrix* m, const double* y, int f, double eps, int use_abs, double var_threshold,
                          int64_t n_new, double* beta, int64_t* idx, int64_t* count);
/* transform2 (:346-430): beta[(i-1) p + (j-1)] for every ordered pair (commutative: j >= i only), 0 for skipped
 * pairs; counters = the selected one-based positions in beta, ASCENDING (sort!(idx), :430); beta_sel their values.
 * beta: p*p values (host or device) or NULL -- the p^2 array then never leaves the device. */
int gbm_transform2_screen(const gbm_matrix* m, const double* y, int f, double eps, int use_abs, double var_threshold,
                          int commutative, int64_t n_new, double* beta, int64_t* counters, double* beta_sel,
                          int64_t* count);
/* Rows [row0, row1) (0-based i) of the same pair matrix: the unit of a multi-GPU screen (every rank holds the
 * n x p matrix and takes a block of rows; no data-path collective).  beta_slab: (row1 - row0) * p values or NULL.
 * counters / beta_sel: the slab's top min(n_new, slab size) effects with abs(beta) > eps in SELECTION order
 * (descending abs(beta), ties by ascending position), counters being global one-based positions -- merging the
 * ranks' lists in that order and cutting at n_new reproduces gbm_transform2_screen (gbm_b200/sharded.py). */
int gbm_transform2_screen_rows(const gbm_matrix* m, const double* y, int f, double eps, int use_abs,
                               double var_threshold, int commutative, int64_t row0, int64_t row1, int64_t n_new,
                               double* beta_slab, int64_t* counters, double* beta_sel, int64_t* count);
/* T = f.(X[:, idx]) resp. f.(X[:, i], X[:, j]) for the selected features, then abs(T) < eps -> 0 and
 * abs(T - 1) < eps -> 1 (:223-227, :440-461).  T: n x count, pitch ldt, host or device. */
int gbm_transform1_apply(const gbm_matrix* m, int f, double eps, int use_abs, const int64_t* idx, int64_t count,
                         double* T, int64_t ldt);
int gbm_transform2_apply(const gbm_matrix* m, int f, double eps, int use_abs, const int64_t* counters, int64_t count,
                         double* T, int64_t ldt);

/* ---- multi-GPU: marker shards over the GPUs of one box (SURVEY.md 8e) --------------------------------
 * The reference's only parallel axis is the marker loop (`Threads.@threads for j = 1:l`,
 * /root/reference/src/gwas.jl:239, :363); its B200 equivalent is one contiguous column block
 * [p r / W, p (r + 1) / W) per GPU r of W.  gwasprep's pieces then need exactly these exchanges, all done inside
 * the library over NCCL / NVLink:
 *   - GRM (gwas.jl:120, :124): every GPU contracts its own markers, ONE all-reduce sums the n x n partials;
 *   - K standardisation + PC1 (gwas.jl:130, :234, :357): the columns of K are sharded, one all-reduce of the
 *     row sums, then one all-reduce of an n-vector per Lanczos step;
 *   - fixed-locus filter (gwas.jl:113): local; idx_cols is the shard-order concatenation, offsets from the
 *     prefix of the per-shard counts;
 *   - marker loop (gwas.jl:239-249, :363-389): no exchange, results gathered in locus order.
 * Two ways to form a group, same entry points afterwards:
 *   gbm_group_create_local : this process drives n_gpus GPUs (devices[] or 0 .. n_gpus-1), one library-owned
 *                            host thread and State per GPU, ncclCommInitAll.  No gbm_init needed.
 *   gbm_group_create_rank  : one process per GPU; the GPU is the one of gbm_init.  Rank 0 makes the 128-byte id
 *                            with gbm_group_unique_id and hands it to the others (torch.distributed, MPI, a file);
 *                            every rank then calls gbm_group_create_rank (collective).
 * Every gbm_sharded_* call is collective over the group: all processes call it with the same arguments.  Host
 * outputs are full-length (all p markers, locus order) and are filled on EVERY process. */
typedef struct gbm_group gbm_group;
typedef struct gbm_sharded gbm_sharded; /* an n x p genotype matrix, column blocks resident on the group's GPUs */
#define GBM_GROUP_ID_BYTES 128
int gbm_group_create_local(int n_gpus, const int* devices, gbm_group** out);
int gbm_group_unique_id(void* id);
int gbm_group_create_rank(const void* id, int world, int rank, gbm_group** out);
int gbm_group_info(const gbm_group* g, int* world, int* n_local, int* first_rank);
int gbm_group_free(gbm_group* g);

/* A: the WHOLE n x p host matrix (every process passes the same matrix; each uploads the blocks of its own GPUs).
 * compact != 0: host cores pack to 1-byte dosage codes on the way when every element of every block is a code
 * (*packed = 1), otherwise Float64 slabs everywhere (*packed = 0).  This is extractxyetc's
 * `G = allele_frequencies[...]` copy (/root/reference/src/prediction.jl:129) landing sharded in HBM. */
int gbm_sharded_upload(gbm_group* g, const double* A, int64_t n, int64_t p, int64_t lda, int compact,
                       gbm_sharded** out, int* packed);
/* synthetic columns 0 .. p-1 of the counter-based generator, each block made on its GPU; pack != 0 converts
 * to dosage codes when every block packs */
int gbm_sharded_generate(gbm_group* g, uint64_t seed, int64_t n, int64_t p, int kind, int pack, gbm_sharded** out,
                         int* packed);
/* wrap blocks that are already resident: local[i] is the block of this process' i-th GPU (same n everywhere, any
 * column counts; blocks are ordered by rank).  The handles stay owned by the caller and must outlive *out. */
int gbm_sharded_adopt(gbm_group* g, gbm_matrix* const* local, gbm_sharded** out);
/* first_col / ncols: n_local entries, the column ranges of this process' blocks */
int gbm_sharded_info(const gbm_sharded* m, int64_t* n, int64_t* p, int64_t* first_col, int64_t* ncols, int* packed);
int gbm_sharded_free(gbm_sharded* m);

/* gbm_colstats over the shards; mean / sd / min_nonzero / keep have length p (all markers), idx_cols has room for
 * p entries: 1-based, ascending, global (gwas.jl:112-113, :119) */
int gbm_sharded_colstats(gbm_sharded* m, double* mean, double* sd, double* min_nonzero, uint8_t* keep,
                         int64_t* idx_cols, int64_t* n_keep, double* min_nonzero_kept);
/* gbm_grm over the shards: per-GPU partials, one all-reduce, scale + mirror.  K (host, n x n) nullable: the GRM then
 * only stays resident on the GPUs for gbm_sharded_kstd_pc1.  tflops: n(n+1)p / (slowest GPU's contraction + the
 * all-reduce), i.e. the aggregate rate of the group. */
int gbm_sharded_grm(gbm_sharded* m, int grm_type, int ploidy, int flags, double* K, double* tflops);
/* gbm_kstd_pc1 on the GRM left resident by gbm_sharded_grm (K = NULL) or on K (host, n x n, every process the same):
 * columns of K sharded (n >= 4096), Lanczos with one n-vector all-reduce per step.  That all-reduce is ONE kernel fused
 * with the reduction of the step's partial sums: every GPU stores its vector, stamped with the step number, into a
 * mailbox on every other GPU over NVLink (peer access inside a process, CUDA IPC mappings between processes) and adds
 * the W contributions in rank order -- identical bits on every GPU.  GPUs without a peer path, more than 8 ranks or
 * GBM_PC1_PEER=0: ncclAllReduce.  pc1: host, n. */
int gbm_sharded_kstd_pc1(gbm_sharded* m, const double* K, double* pc1, double* eig_ms);
/* gbm_scan over the shards: outputs p x T column-major (ld p) / length p, host, on every process */
int gbm_sharded_scan(gbm_sharded* m, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k, int64_t ldc,
                     int model, int flags, double* beta, double* se, double* stat, double* neglog10p, double* mean,
                     double* sd, uint8_t* keep);

/* The whole of gwasols (gwas.jl:206-259) / gwaslmm (:329-399) after extractxyetc, in one collective call:
 * filter + ploidy probe, GRM (+ all-reduce), K standardisation, PC1, marker scan with [1, PC1], gather.
 * y: n, used as given (the caller standardises, gwas.jl:128).  grm_type GBM_GRM_PLOIDY_AWARE infers the ploidy as
 * gwas.jl:119 does.  Outputs (host, nullable): stat / beta / se / neglog10p / mean / sd / keep of length p in locus
 * order (NaN for filtered or degenerate markers), idx_cols (room for p), pc1 (n). */
typedef struct gbm_gwas_timing {
  double colstats_ms, grm_ms, allreduce_ms, kstd_pc1_ms, eig_ms, scan_ms, gather_ms, total_ms; /* host wall clock */
  double grm_tflops;      /* n(n+1)p / (grm_ms + allreduce_ms): aggregate of the group */
  double scan_kernel_ms;  /* slowest GPU's streaming kernel (CUDA events) */
  int64_t launches;       /* kernels launched by this process */
  int32_t ploidy, lanczos_steps;
} gbm_gwas_timing;
int gbm_sharded_gwas(gbm_sharded* m, const double* y, int model, int grm_type, int flags, double* stat, double* beta,
                     double* se, double* neglog10p, double* mean, double* sd, uint8_t* keep, int64_t* idx_cols,
                     int64_t* n_keep, double* pc1, gbm_gwas_timing* timing);

/* The GRM-covariance LMM (gbm_lmm_plan_*, the model of gwasreml) over the shards.  K is factored ONCE: rank 0 runs
 * the syevd of gbm_lmm_plan_create, rotates [1, C, y] and fits the null model, then broadcasts U, S, U'y, U'[1, C],
 * the null log(delta) and the smallest eigenvalue to every GPU -- U is the same bits everywhere.  Every GPU then
 * rotates and searches its own column block exactly as gbm_lmm_plan_run does (no exchange); results are gathered in
 * locus order, so per-marker outputs equal the single-GPU engine's for the same K. */
typedef struct gbm_sharded_lmm_plan gbm_sharded_lmm_plan;
/* host wall clock (ms) of each step of one collective call; steps a call does not run stay 0.  kprep: K into rank 0's
 * factor buffer (standardised and symmetrised for the reference objective); eig: the plans' allocation, rank 0's
 * syevd, rotation of [1, C, y] and null model; broadcast: U, S and the rest to every GPU; scan: rotation + search on
 * every GPU; gather: the outputs in locus order */
typedef struct gbm_reml_timing {
  double colstats_ms, grm_ms, allreduce_ms, kprep_ms, eig_ms, broadcast_ms, scan_ms, gather_ms, total_ms;
  double rotation_ms;     /* slowest GPU's rotation GEMMs U'A (CUDA events) */
  double search_ms;       /* slowest GPU's per-marker delta search (CUDA events) */
  double rotation_tflops; /* 2 n^2 p / rotation_ms: aggregate of the group */
  double grm_tflops;      /* n(n+1)p / (grm_ms + allreduce_ms): aggregate of the group */
  int64_t launches;       /* kernels launched by this process */
  int32_t ploidy, n_gpus; /* ploidy the GRM used; GPUs of the group (all ranks) */
} gbm_reml_timing;
/* collective.  K: host n x n, the same on every process (only rank 0 reads it, lower triangle); y: n; C: n x k
 * (ldc), k = 0..2 covariates besides the intercept -- as gbm_lmm_plan_create.  eig_ms: rank 0's syevd. */
int gbm_sharded_lmm_plan_create(gbm_sharded* m, const double* K, const double* y, const double* C, int64_t k,
                                int64_t ldc, gbm_sharded_lmm_plan** plan, double* eig_ms, double* null_log_delta);
/* collective.  Outputs host, length p, locus order, on every process, nullable; flags as gbm_lmm_plan_run
 * (GBM_PVALUE_TWO_SIDED, GBM_LMM_REFERENCE_OBJECTIVE).  timing (nullable): the marker steps only. */
int gbm_sharded_lmm_plan_run(gbm_sharded_lmm_plan* plan, gbm_sharded* m, int flags, double* beta, double* se,
                             double* stat, double* neglog10p, double* log_delta, gbm_reml_timing* timing);
int gbm_sharded_lmm_plan_free(gbm_sharded_lmm_plan* plan);
/* The whole of gwasreml (gwas.jl:549-613) after extractxyetc in one collective call: filter + ploidy probe, GRM
 * (+ all-reduce; centred, never GBM_GRM_NO_CENTRE), with GBM_LMM_REFERENCE_OBJECTIVE the column standardisation of K
 * (gwas.jl:130) and its symmetric part (K + K') / 2 on the device, then the plan above.  y: n, used as given.  flags:
 * GBM_PVALUE_TWO_SIDED and GBM_LMM_REFERENCE_OBJECTIVE only, any other bit is an argument error.  Outputs (host,
 * nullable): stat / beta / se / neglog10p / log_delta of length p in locus order (NaN for filtered markers),
 * idx_cols (room for p), the null model's log(delta). */
int gbm_sharded_gwasreml(gbm_sharded* m, const double* y, int grm_type, int flags, double* stat, double* beta,
                         double* se, double* neglog10p, double* log_delta, int64_t* idx_cols, int64_t* n_keep,
                         double* null_log_delta, gbm_reml_timing* timing);

/* -log10 upper-tail probabilities on the device (log-space; finite where 1 - cdf saturates) */
int gbm_neglog10_sf(const double* stat, int64_t len, int dist /*0: TDist(df), 1: Normal*/, double df, double* out);

/* measured device-to-device copy bandwidth (GB/s, read+write bytes) -- for rooflines */
int gbm_measure_copy_bandwidth(int64_t bytes, int reps, double* gbps);

#ifdef __cplusplus
}
#endif
#endif /* GBM_B200_H */
