// Internal launch interfaces between the C-ABI translation unit and the kernel units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gbm {

// generate.cu
void launch_generate(double* A, int64_t n, int64_t p, int64_t lda, int64_t col0, uint64_t seed, int kind,
                     cudaStream_t stream);

// scan.cu ------------------------------------------------------------------------------
// Per-marker record written by the streaming kernel: [mean, SS, dot_1 .. dot_M (, minnz)]
// where SS = sum (a - mean)^2 and dot_m = sum a * q_m (q_m orthogonal to 1).
int scan_record_stride(int M, bool minnz);
// Largest M (number of side vectors) one pass supports.
int scan_max_side_vectors();
// Streams the n x p matrix once (TMA -> smem ring -> FP64 accumulators).  Q is n x M
// column-major with leading dimension ldq (device, ldq even, every column orthogonal to 1).
void launch_scan_sums(const double* A, int64_t n, int64_t p, int64_t lda, const double* Q, int M, int64_t ldq,
                      bool minnz, double* rec, int sm_count, cudaStream_t stream);

// scan_mt.cu: the same sums for up to 31 side vectors in one pass on the FP64 tensor pipe (DMMA).  Qx is
// n x (M + 1) with the vector of ones in column 0; records are [mean, SS, dot_1 .. dot_M] with pitch rec_stride.
int scan_mt_max_side_vectors();
void launch_scan_sums_mt(const double* A, int64_t n, int64_t p, int64_t lda, const double* Qx, int M, int64_t ldq,
                         double* rec, int rec_stride, int sm_count, cudaStream_t stream);

void launch_scan_sums_mt_u8(const uint8_t* A8, int64_t n, int64_t p, int64_t ld8, const double* Qx, int M, int64_t ldq,
                            double* rec, int rec_stride, int sm_count, cudaStream_t stream);

struct FinalizeParams {
  int64_t n, p;
  int64_t ld_out;      // leading dimension of the p x T outputs
  int k, T;            // covariates (orthonormal, first k dots) and traits (next T dots)
  int rec_stride;
  int model, flags;
  const double* rec;   // [p][rec_stride]
  const double* yMy;   // [T] device
  const double* wy;    // [T][k] device: w_a' (y_t - mean) for the orthonormal covariates (degenerate markers)
  double* beta;        // p x T (nullable)
  double* se;
  double* stat;
  double* nlp;
  double* mean;        // p (nullable)
  double* sd;
  uint8_t* keep;
};
void launch_scan_finalize(const FinalizeParams& prm, cudaStream_t stream);

// colstats finalisation: mean / sd / min_nonzero / keep from records with M = 0, minnz
void launch_colstats_finalize(const double* rec, int rec_stride, int64_t n, int64_t p, double* mean, double* sd,
                              double* minnz, uint8_t* keep, cudaStream_t stream);
// idx_cols (1-based ascending) + count + min over kept columns of minnz; single pass on device
void launch_compact_keep(const uint8_t* keep, const double* minnz, int64_t p, int64_t* idx_cols, int64_t* n_keep,
                         double* min_kept, cudaStream_t stream);

void launch_neglog10_sf(const double* stat, int64_t len, int dist, double df, double* out, cudaStream_t stream);

// scan_u8.cu --------------------------------------------------------------------------
// Compact dosage codes (1 byte per genotype, a = code/240).  Mp = padded side-vector count as in scan.cu;
// records have the same meaning and stride as the Float64 kernel's (Mp = 0 tracks min-nonzero).
void launch_scan_sums_u8(const uint8_t* A8, int64_t n, int64_t p, int64_t ld8, const double* Q, int Mp, int64_t ldq,
                         double* rec, int sm_count, cudaStream_t stream);
// scan_u8_tc.cu: the same sums with the dots on the tcgen05 INT8 tensor cores (side vectors as seven base-256
// fixed-point digits, exact integer contractions).  digits: 16 x ldd int8 (device), built by scan_u8_tc_build_digits
// on the host from the n x M side vectors (M <= 2); scale[m] = 2^(E_m - 55).
int scan_u8_tc_digit_rows(int64_t n);
void scan_u8_tc_build_digits(const double* Q, int64_t n, int M, int64_t ldq, int8_t* digits, int64_t ld, double* scale);
void launch_scan_sums_u8_tc(const uint8_t* A8, int64_t n, int64_t p, int64_t ld8, const int8_t* digits, int64_t ldd,
                            const double* scale, int M, int rec_stride, double* rec, int sm_count, cudaStream_t stream);
void launch_pack_u8(const double* A, int64_t n, int64_t p, int64_t lda, uint8_t* out, int64_t ld8,
                    unsigned long long* inexact, cudaStream_t stream);
void launch_decode_u8(const uint8_t* A8, int64_t n, int64_t p, int64_t ld8, double* out, int64_t ldo,
                      cudaStream_t stream);

// grm.cu -------------------------------------------------------------------------------
// dK (n x n col-major, ld n) += lower-triangle tiles of sum_j (a_j - mu_j)(a_j - mu_j)'.
// mu: device, length >= round_up(p, 16), zero padded (all zeros = uncentred).
// centred = false: mu must be all zeros and no correction pass is run.
void launch_grm_accumulate(const double* A, int64_t n, int64_t p, int64_t lda, const double* mu, double* dK,
                           int sm_count, cudaStream_t stream, bool centred);
// scale the lower triangle and mirror it into the upper one
void launch_grm_finalize(double* dK, int64_t n, double scale, cudaStream_t stream);
// out[0] += sum_j mu_j (1 - mu_j)
void launch_sum_q1mq(const double* mu, int64_t p, double* out, cudaStream_t stream);

// pc1.cu -------------------------------------------------------------------------------
// In place: K <- (K - colmean) / colsd ; then Z = Kstd - rowmean (written to Z). n x n, pitch ld.
void launch_k_standardise(double* K, int64_t n, int64_t ncols, int64_t ld, const double* colmean, const double* colsd,
                          cudaStream_t stream);
// Z[i, j] -= rowsum[i] * inv_cols over an n x ncols column block
void launch_row_shift(double* Z, int64_t n, int64_t ncols, int64_t ld, const double* rowsum, double inv_cols,
                      cudaStream_t stream);
void launch_row_centre(const double* Ks, double* Z, int64_t n, int64_t ld, cudaStream_t stream);
// K <- (K + K') / 2 in place (n x n, pitch ld)
void launch_symmetrise(double* K, int64_t n, int64_t ld, cudaStream_t stream);
// gather rows/cols (1-based indices, nullable) from a device source into a padded device matrix
void launch_gather(const double* src, int64_t lds, const int64_t* rows, int64_t n, const int64_t* cols, int64_t p,
                   double* dst, int64_t ldd, cudaStream_t stream);

void launch_gather_standardise(const double* src, int64_t lds, int64_t n, const int64_t* cols, int64_t ncols,
                               const double* mean, const double* sd, double* dst, int64_t ldd, cudaStream_t stream);

void launch_gather_standardise_u8(const uint8_t* src, int64_t lds, int64_t n, const int64_t* cols, int64_t ncols,
                                  const double* mean, const double* sd, double* dst, int64_t ldd, cudaStream_t stream);

// grm_i8.cu ---------------------------------------------------------------------------
// dG (n x n, zeroed by the caller) += lower-triangle tiles of C C' for the code matrix C (exact integers)
void launch_grm_i8_accumulate(const uint8_t* A8, int64_t n, int64_t p, int64_t ld8, double* dG, int sm_count,
                              cudaStream_t stream);
void launch_rowdot_u8(const uint8_t* A8, int64_t n, int64_t p, int64_t ld8, const double* S, double* U,
                      cudaStream_t stream);
void launch_code_sums(const double* mean, int64_t p, int64_t n, double* S, double* M2, cudaStream_t stream);
void launch_grm_i8_combine(const double* G, int64_t n, const double* U, const double* M2, int centre, double* dK,
                           cudaStream_t stream);

// gemm_tn.cu --------------------------------------------------------------------------
// C (M x N, ldc) = A' B with A: K x M (lda), B: K x N (ldb), all column-major, device; lda, ldb even.
void launch_gemm_tn(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int64_t M,
                    int64_t N, int64_t K, int sm_count, cudaStream_t stream);

// lmm.cu ------------------------------------------------------------------------------
// Per-marker REML delta search on a rotated block (one warp per marker). Q0 = fixed covariates incl. intercept.
void launch_lmm_delta(int Q0, const double* Ar, int64_t n, int64_t pb, int64_t ld, const double* S, const double* Yr,
                      const double* Cr, int64_t ldcr, double lam0, const double* col_sd, const uint8_t* keep,
                      double* beta, double* se, double* stat, double* nlp, double* log_delta, int flags,
                      int sm_count, cudaStream_t stream, int objective = 0, double s_min = 0.0);
// null-model log(delta) on the host from rotated vectors
double lmm_null_lam0(int Q0, const double* S, const double* Cr, int64_t ldcr, const double* Yr, int64_t n);

// lanczos.cu --------------------------------------------------------------------------
// Largest eigenpair of the symmetric PSD matrix B (n x n, pitch ldb even, 16-byte aligned, device) by Lanczos with
// full reorthogonalisation; x_dev (device, n) gets the unit eigenvector.  Returns false when the explicit residual
// ||B x - theta x|| <= max(5 tol, 2e-13) theta was not reached within max_iter steps (the caller then uses cuSOLVER).
// gram = true: the operator is B B' for a general (non-symmetric) n x n matrix B, applied as two matrix-vector
// products per step (B B' is never formed); x is then the top left singular vector of B.
bool lanczos_top_eigenpair(const double* B, int64_t n, int64_t ldb, bool gram, double tol, int max_iter, double* x_dev,
                           double* theta, int* iters, int sm_count, cudaStream_t stream);
// The same when the columns of Z (n x n) are sharded over the ranks of a group: Zg is this rank's n x nc column
// block (pitch ld).  Z Z' = sum over ranks of Zg Zg', so a step is u = Zg' v, w = Zg u (two passes over the block)
// and ONE all-reduce of the n-vector w; everything else runs replicated (NCCL hands every rank the same bits, so
// the replicas stay identical).  allreduce_sum(buf, count) must sum `count` doubles at `buf` (device) over the
// ranks, ordered on `stream`.  rowsum_out (nullable, n): Zg 1, the block's row sums, before any all-reduce.
struct ShardedAllReduce {
  virtual void sum(double* buf, int64_t count) = 0;
  // out = sum over the ranks of (sum_c partial[c][:]), c < chunks: the CTA partials of the fused Lanczos pass.  The
  // default reduces the partials and all-reduces the result; a group with peer access overrides it with ONE kernel
  // that does both over NVLink (peer_sum_kernel, lanczos.cu).
  virtual void sum_partials(const double* partial, int chunks, int64_t n, double* out, cudaStream_t stream);
  virtual ~ShardedAllReduce() {}
};
// host part of the Lanczos solver: largest eigenvalue (Sturm bisection) and its unit eigenvector (inverse iteration
// with a pivoted tridiagonal solve) of the m x m symmetric tridiagonal with diagonal a[0..m) and off-diagonal b[0..m-1)
void lanczos_tridiag_top(const double* a, const double* b, int m, double* theta, double* s);
// the fused one-pass Lanczos step holds a column of Z twice in shared memory: n <= kLanczosFusedMaxN
constexpr int64_t kLanczosFusedMaxN = 512 * 24;
// Mailboxes of a one-shot all-reduce over peer memory.  Every rank owns 2 (step parity) x W (source rank) x npad
// entries of 16 bytes; slots[q] is rank q's mailbox as seen from THIS device (peer access or a CUDA IPC mapping).  An
// entry carries one double as two 8-byte words {step << 32 | low half, step << 32 | high half}: the step number travels
// in the same (atomic) 8-byte store as the data, so a reader that sees the stamp has the data -- no fence, no separate
// flag, one NVLink crossing per exchange (the idea of NCCL's LL protocol, for FP64 payloads).
struct PeerMailbox {
  static constexpr int kMaxRanks = 8;
  double* slots[kMaxRanks];  // 2 doubles of storage per entry
  double* mine = nullptr;    // = slots[me]
  int world = 0, me = 0;
  int64_t npad = 0;
  int* error = nullptr;  // this device: set when a peer did not show up in time
};
// partial-sum reduction + all-reduce in one kernel: this rank's reduced vector is stored, stamped with `step`, into slot
// `me` of every rank's mailbox over NVLink; the kernel then polls the W slots of its own mailbox for the stamp and adds
// them in rank order (the same order, hence the same bits, on every rank).  `step` starts at 1 and grows by one per
// call on every rank; a slot is reused two steps later, when every reader is provably past it.
void launch_peer_sum(const PeerMailbox& mb, const double* partial, int chunks, int64_t n, unsigned long long step,
                     double* out, cudaStream_t stream);
void block_row_sums(const double* Zg, int64_t n, int64_t nc, int64_t ld, double* rowsum, cudaStream_t stream);
bool lanczos_top_singular_sharded(const double* Zg, int64_t n, int64_t nc, int64_t ld, ShardedAllReduce* ar, double tol,
                                  int max_iter, double* x_dev, double* theta, int* iters, int sm_count,
                                  cudaStream_t stream);

// transform.cu -------------------------------------------------------------------------
// Per-locus OLS screen of f(x): beta[j] (0 when var(x) < var_thr) and colvar[j] = var(x) (nullable).
// f = -1: variance pass only.  yc = y - ybar (device, n).
void launch_transform1_scan(int f, const double* A, int64_t n, int64_t p, int64_t lda, const double* yc, double ybar,
                            double eps, int use_abs, double var_thr, double* beta, double* colvar, int sm_count,
                            cudaStream_t stream);
// Pairwise screen over rows [row0, row1) of the l x l pair matrix (0-based i; the whole screen is [0, l)):
// beta[(i - row0) l + j] for every evaluated pair; beta ((row1 - row0) x l) must be zeroed by the caller.
void launch_transform2_scan(int f, const double* A, int64_t n, int64_t l, int64_t lda, const double* yc, double ybar,
                            const double* colvar, double eps, int use_abs, double var_thr, int commutative,
                            int64_t row0, int64_t row1, double* beta, cudaStream_t stream);
void launch_transform1_apply(int f, const double* A, int64_t n, int64_t lda, const int64_t* idx, int64_t count,
                             double eps, int use_abs, double* T, int64_t ldt, cudaStream_t stream);
void launch_transform2_apply(int f, const double* A, int64_t n, int64_t l, int64_t lda, const int64_t* counters,
                             int64_t count, double eps, int use_abs, double* T, int64_t ldt, cudaStream_t stream);
// top n_new of abs(beta) in Julia's stable sortperm order, filtered by abs(beta) > eps; returns the count,
// idx_host (1-based) and optionally the selected values.  A NaN among the top entries is reported by *has_nan.
int64_t transform_select(const double* beta_dev, int64_t len, int64_t n_new, double eps, int64_t* idx_host,
                         double* beta_host, bool* has_nan, int sm_count, cudaStream_t stream);
void launch_gather_values(const double* src, const long long* idx1, int64_t count, double* dst, cudaStream_t stream);

}  // namespace gbm

// gbm_api.cu: the LMM plan (gbm_lmm_plan_*) in steps, shared by the single-GPU entry points and the group engine
// (group.cu: rank 0 loads and factors K, the other GPUs receive U, S, U'y, U'[1, C], lam0 and s_min)
struct gbm_lmm_plan {
  int64_t n = 0, ldu = 0;
  int Q0 = 1;
  double* dU = nullptr;   // eigenvectors, n x n (ldu)
  double* dS = nullptr;   // eigenvalues ascending
  double* dYr = nullptr;  // U'y
  double* dCr = nullptr;  // U'[1, C], n x Q0 (ld n)
  double lam0 = 0.0;
  double s_min = 0.0;     // smallest eigenvalue (negative for an indefinite K)
};
namespace gbm {
// device buffers on the calling thread's GPU (ldu = n rounded up to 16); throws, leaving nothing allocated, on failure
gbm_lmm_plan* lmm_plan_alloc(int64_t n, int Q0);
void lmm_plan_destroy(gbm_lmm_plan* pl);
// K (n x n, pitch ldk, host or device) into dU, padding rows zeroed
void lmm_plan_load_k(gbm_lmm_plan* pl, const double* K, int64_t ldk);
// dU holds K: K = U S U' (cuSOLVER syevd, eig_ms = its time), rotation of [1, C, y], null-model lam0 and s_min
void lmm_plan_factor(gbm_lmm_plan* pl, const double* y, const double* C, int64_t k, int64_t ldc, double* eig_ms);
}  // namespace gbm
