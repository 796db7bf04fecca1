// C ABI of libgbm_b200.so (declared in include/gbm_b200.h).  Host-side orchestration only:
// argument checks that mirror the reference's error behaviour, device buffers, the small
// host-side linear algebra on the n x (k + T) side vectors, kernel launches, timing.
#include "../../include/gbm_b200.h"

#include <cusolverDn.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#ifdef __linux__
#include <sched.h>
#endif
#include <vector>

#include "common.cuh"
#include "kernels.h"

struct gbm_matrix {
  double* d = nullptr;      // Float64 slab (dtype 0)
  int64_t n = 0, p = 0, lda = 0;
  bool owned = false;
  int dtype = 0;            // 0: Float64, 1: one-byte dosage codes (a = code / 240)
  uint8_t* d8 = nullptr;    // code slab (dtype 1), column pitch ld8 bytes
  int64_t ld8 = 0;
  bool pooled = false;      // slab from the stream-ordered pool (small matrices: no driver call per upload / free)
};

namespace gbm {

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }
// entry points are serialised per State (SURVEY.md 8b "Threading"): State::api_mutex
static thread_local State* t_state = nullptr;
State& state() {
  static State s;
  return t_state ? *t_state : s;
}
void bind_state(State* s) { t_state = s; }
void require_ready() {
  State& st = state();
  if (!st.ready) throw Error{GBM_ERR_NOT_INITIALISED, "gbm_init has not been called (no CUDA device selected)"};
  // the current device is per host thread: a caller that comes in on another thread (Julia tasks migrate)
  // must still land on this State's GPU
  GBM_CUDA(cudaSetDevice(st.device));
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    GBM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (!p || qres != cudaDriverEntryPointSuccess) GBM_THROW(GBM_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

void make_tensor_map_2d_f64(CUtensorMap* map, const double* base, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                            uint32_t box_rows, uint32_t box_cols) {
  if ((reinterpret_cast<uintptr_t>(base) & 15u) != 0 || (ld_elems & 1u) != 0)
    GBM_THROW(GBM_ERR_ARGUMENT, "device matrix must be 16-byte aligned with an even leading dimension");
  cuuint64_t gdim[2] = {rows, cols};
  cuuint64_t gstride[1] = {ld_elems * sizeof(double)};
  cuuint32_t box[2] = {box_rows, box_cols};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
}

void make_tensor_map_2d_u64(CUtensorMap* map, const void* base, uint64_t rows64, uint64_t cols, uint64_t ld_bytes,
                            uint32_t box_rows64, uint32_t box_cols) {
  if ((reinterpret_cast<uintptr_t>(base) & 15u) != 0 || (ld_bytes & 15u) != 0)
    GBM_THROW(GBM_ERR_ARGUMENT, "packed matrix must be 16-byte aligned with a pitch that is a multiple of 16");
  cuuint64_t gdim[2] = {rows64, cols};
  cuuint64_t gstride[1] = {ld_bytes};
  cuuint32_t box[2] = {box_rows64, box_cols};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled()(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cuTensorMapEncodeTiled (u64) failed with code " + std::to_string((int)r));
}

void make_tensor_map_2d_u8(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld_bytes,
                           uint32_t box_rows, uint32_t box_cols) {
  if ((reinterpret_cast<uintptr_t>(base) & 15u) != 0 || (ld_bytes & 15u) != 0 || (box_rows & 15u) != 0)
    GBM_THROW(GBM_ERR_ARGUMENT, "packed matrix must be 16-byte aligned with a pitch that is a multiple of 16");
  cuuint64_t gdim[2] = {rows, cols};
  cuuint64_t gstride[1] = {ld_bytes};
  cuuint32_t box[2] = {box_rows, box_cols};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled()(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cuTensorMapEncodeTiled (u8) failed with code " + std::to_string((int)r));
}

void make_tensor_map_2d_u8_sw128(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld_bytes,
                                 uint32_t box_rows, uint32_t box_cols) {
  if ((reinterpret_cast<uintptr_t>(base) & 15u) != 0 || (ld_bytes & 15u) != 0)
    GBM_THROW(GBM_ERR_ARGUMENT, "packed matrix must be 16-byte aligned with a pitch that is a multiple of 16");
  cuuint64_t gdim[2] = {rows, cols};
  cuuint64_t gstride[1] = {ld_bytes};
  cuuint32_t box[2] = {box_rows, box_cols};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled()(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cuTensorMapEncodeTiled (u8, swizzle 128B) failed with code " + std::to_string((int)r));
}

// host_pack.cpp: worker queue of the calling process' cores (packing to dosage codes, staging copies)
struct PackJob;
PackJob* pack_submit(const double* A, int64_t n, int64_t lda, int64_t pc, uint8_t* out, int64_t ldo);
bool pack_wait(PackJob* job, const std::function<void()>* idle);
bool pack_block_host(const double* A, int64_t n, int64_t lda, int64_t pc, uint8_t* out, int64_t ldo,
                     const std::function<void()>* idle);
int64_t count_inexact_host(const double* A, int64_t n, int64_t lda, int64_t pc);
bool pack_check_columns(const double* A, int64_t n, int64_t lda, int64_t pc, int isa, uint8_t* col_ok);
int host_threads();
PackJob* copy_submit(const double* A, int64_t n, int64_t lda, int64_t pc, double* out, int64_t ldo);

static int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

static bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// page-locked host memory (cudaMallocHost / cudaHostRegister): async copies from it do not block
static bool is_pinned_host_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost;
}

// stream-ordered scratch buffer
template <typename T>
struct DevBuf {
  T* p = nullptr;
  cudaStream_t s;
  DevBuf(size_t count, cudaStream_t stream) : s(stream) {
    if (count) GBM_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p), count * sizeof(T), stream));
  }
  ~DevBuf() {
    if (p) cudaFreeAsync(p, s);
  }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
};

// streaming sums over a resident matrix of either storage type.  mt: Q is [1 | side vectors] (M + 1 columns)
// and the FP64 tensor-pipe kernel of scan_mt.cu runs (records of `stride` doubles); otherwise the streaming
// kernels of scan.cu / scan_u8.cu with their own record stride.
struct SideDigits {  // fixed-point digits of the side vectors for the tensor-core code kernel (scan_u8_tc.cu)
  const int8_t* d = nullptr;
  int64_t ld = 0;
  double scale[2] = {0.0, 0.0};
};
static bool use_u8_tensor_cores() {  // GBM_U8_TC=0: the CUDA-core kernel of scan_u8.cu (read at every call: tests toggle it)
  const char* e = getenv("GBM_U8_TC");
  return e ? atoi(e) != 0 : true;
}

static void scan_sums_any(const gbm_matrix* m, int64_t j0, int64_t pb, const double* Q, int M, int64_t ldq,
                          double* rec, bool mt = false, int mt_stride = 0, const SideDigits* dg = nullptr) {
  State& st = state();
  if (m->dtype == 0) {
    if (mt)
      launch_scan_sums_mt(m->d + j0 * m->lda, m->n, pb, m->lda, Q, M, ldq, rec, mt_stride, st.sm_count, st.stream);
    else
      launch_scan_sums(m->d + j0 * m->lda, m->n, pb, m->lda, Q, M, ldq, M == 0, rec, st.sm_count, st.stream);
  } else {
    const int stride = mt ? mt_stride : scan_record_stride(M, false);
    const int Mp = stride - 2 - (M == 0 ? 1 : 0);
    if (!mt && M >= 1 && M <= 2 && dg && dg->d && use_u8_tensor_cores()) {
      launch_scan_sums_u8_tc(m->d8 + j0 * m->ld8, m->n, pb, m->ld8, dg->d, dg->ld, dg->scale, M, stride, rec, st.sm_count,
                             st.stream);
    } else if (!mt && Mp <= 2) {
      launch_scan_sums_u8(m->d8 + j0 * m->ld8, m->n, pb, m->ld8, Q, Mp, ldq, rec, st.sm_count, st.stream);
    } else if (mt) {
      launch_scan_sums_mt_u8(m->d8 + j0 * m->ld8, m->n, pb, m->ld8, Q, M, ldq, rec, stride, st.sm_count, st.stream);
    } else {
      // many side vectors (multi-trait) on packed codes: decode column blocks, Float64 kernel
      const int64_t ldt = round_up(m->n, 16);
      int64_t PB = std::max<int64_t>(16, ((int64_t(1) << 30) / (8 * ldt)) / 16 * 16);
      PB = std::min(PB, round_up(pb, 16));
      DevBuf<double> tmp(static_cast<size_t>(ldt) * PB, st.stream);
      for (int64_t b0 = 0; b0 < pb; b0 += PB) {
        const int64_t pc = std::min(PB, pb - b0);
        launch_decode_u8(m->d8 + (j0 + b0) * m->ld8, m->n, pc, m->ld8, tmp.p, ldt, st.stream);
        if (mt)
          launch_scan_sums_mt(tmp.p, m->n, pc, ldt, Q, M, ldq, rec + b0 * stride, stride, st.sm_count, st.stream);
        else
          launch_scan_sums(tmp.p, m->n, pc, ldt, Q, M, ldq, false, rec + b0 * stride, st.sm_count, st.stream);
      }
    }
  }
}

// event-pair timing on the library stream
struct Span {
  cudaEvent_t a, b;
  cudaStream_t s;
  bool open = false;
  Span(cudaStream_t stream) : s(stream) {
    cudaEventCreate(&a);
    cudaEventCreate(&b);
  }
  ~Span() {
    cudaEventDestroy(a);
    cudaEventDestroy(b);
  }
  void start() {
    cudaEventRecord(a, s);
    open = true;
  }
  void stop() { cudaEventRecord(b, s); }
  double ms() {
    if (!open) return 0.0;
    cudaEventSynchronize(b);
    float t = 0.f;
    cudaEventElapsedTime(&t, a, b);
    return t;
  }
};

static void reset_timing() {
  State& st = state();
  st.h2d_ms = st.kernel_ms = st.main_ms = st.d2h_ms = 0.0;
  st.launches = 0;
  st.packed_blocks = st.host_packed_blocks = st.h2d_bytes = 0;
}

// staging of gbm_scan_host (see State)
static void free_scan_host_staging(State& st) {
  for (int b = 0; b < State::kHostSlots; ++b) {
    if (st.host_codes[b]) cudaFreeHost(st.host_codes[b]);
    if (st.dev_codes[b]) cudaFree(st.dev_codes[b]);
    st.host_codes[b] = st.dev_codes[b] = nullptr;
    if (st.hl_copied[b]) cudaEventDestroy(st.hl_copied[b]);
    if (st.hl_consumed[b]) cudaEventDestroy(st.hl_consumed[b]);
    st.hl_copied[b] = st.hl_consumed[b] = nullptr;
  }
  for (int b = 0; b < State::kRawSlots; ++b) {
    if (st.raw_f64[b]) cudaFree(st.raw_f64[b]);
    if (st.raw_codes[b]) cudaFree(st.raw_codes[b]);
    st.raw_f64[b] = st.raw_codes[b] = nullptr;
    if (st.raw_copied[b]) cudaEventDestroy(st.raw_copied[b]);
    if (st.raw_packed[b]) cudaEventDestroy(st.raw_packed[b]);
    if (st.raw_consumed[b]) cudaEventDestroy(st.raw_consumed[b]);
    st.raw_copied[b] = st.raw_packed[b] = st.raw_consumed[b] = nullptr;
  }
  for (int b = 0; b < State::kHostSlots; ++b) {
    if (st.up_stage[b]) cudaFreeHost(st.up_stage[b]);
    st.up_stage[b] = nullptr;
    if (st.up_copied[b]) cudaEventDestroy(st.up_copied[b]);
    st.up_copied[b] = nullptr;
  }
  st.up_bytes = 0;
  if (st.raw_flag_dev) cudaFree(st.raw_flag_dev);
  if (st.raw_flag_host) cudaFreeHost(st.raw_flag_host);
  st.raw_flag_dev = st.raw_flag_host = nullptr;
  st.code_bytes = st.raw_bytes = st.raw_code_bytes = 0;
}

static void copy_out(void* user, const void* dev, size_t bytes, cudaStream_t s) {
  if (user && bytes) GBM_CUDA(cudaMemcpyAsync(user, dev, bytes, cudaMemcpyDefault, s));
}

// --------------------------------------------------------------------------------------
// side vectors: orthonormalise [1, C] and residualise Y on the host (n x (k+T), tiny)
// --------------------------------------------------------------------------------------
struct SideVectors {
  int k_eff = 0;              // covariates that survived orthogonalisation
  std::vector<double> W;      // n x k_eff, orthonormal, orthogonal to 1
  std::vector<double> R;      // n x T residualised traits  (I - 11'/n - WW') y
  std::vector<double> yMy;    // T
  std::vector<double> wy;     // T x k_eff: w_a' (y_t - mean), the covariates' own coefficients (degenerate markers)
};

static SideVectors prepare_side_vectors(const double* Y, int64_t n, int64_t T, int64_t ldy, const double* C,
                                        int64_t k, int64_t ldc) {
  SideVectors sv;
  std::vector<double> hY(static_cast<size_t>(n) * T), hC(static_cast<size_t>(n) * std::max<int64_t>(k, 0));
  if (T > 0)
    GBM_CUDA(cudaMemcpy2D(hY.data(), n * sizeof(double), Y, ldy * sizeof(double), n * sizeof(double), T,
                          cudaMemcpyDefault));
  if (k > 0)
    GBM_CUDA(cudaMemcpy2D(hC.data(), n * sizeof(double), C, ldc * sizeof(double), n * sizeof(double), k,
                          cudaMemcpyDefault));
  auto centre = [&](double* v) {
    long double s = 0;
    for (int64_t i = 0; i < n; ++i) s += v[i];
    const double m = static_cast<double>(s / n);
    for (int64_t i = 0; i < n; ++i) v[i] -= m;
  };
  auto dot = [&](const double* a, const double* b) {
    long double s = 0;
    for (int64_t i = 0; i < n; ++i) s += static_cast<long double>(a[i]) * b[i];
    return static_cast<double>(s);
  };
  // modified Gram-Schmidt, twice, against 1 and the accepted covariates
  for (int64_t c = 0; c < k; ++c) {
    double* v = hC.data() + c * n;
    const double norm0 = sqrt(dot(v, v));
    for (int pass = 0; pass < 2; ++pass) {
      centre(v);
      for (int a = 0; a < sv.k_eff; ++a) {
        const double* w = sv.W.data() + static_cast<size_t>(a) * n;
        const double h = dot(w, v);
        for (int64_t i = 0; i < n; ++i) v[i] -= h * w[i];
      }
    }
    const double norm = sqrt(dot(v, v));
    if (!(norm > 1e-10 * norm0) || !(norm > 0.0)) continue;  // collinear with 1 / earlier covariates
    sv.W.resize(static_cast<size_t>(sv.k_eff + 1) * n);
    double* w = sv.W.data() + static_cast<size_t>(sv.k_eff) * n;
    for (int64_t i = 0; i < n; ++i) w[i] = v[i] / norm;
    sv.k_eff++;
  }
  sv.R.resize(static_cast<size_t>(n) * T);
  sv.yMy.resize(T);
  sv.wy.assign(static_cast<size_t>(T) * std::max(sv.k_eff, 1), 0.0);
  for (int64_t t = 0; t < T; ++t) {
    double* r = sv.R.data() + t * n;
    memcpy(r, hY.data() + t * n, sizeof(double) * n);
    for (int pass = 0; pass < 2; ++pass) {
      centre(r);
      for (int a = 0; a < sv.k_eff; ++a) {
        const double* w = sv.W.data() + static_cast<size_t>(a) * n;
        const double h = dot(w, r);
        sv.wy[static_cast<size_t>(t) * sv.k_eff + a] += h;
        for (int64_t i = 0; i < n; ++i) r[i] -= h * w[i];
      }
    }
    sv.yMy[t] = dot(r, r);
  }
  return sv;
}

// Device copies of the side vectors, one per pass over the matrix.  Up to two side vectors (the reference case:
// PC1 + one trait) use the streaming FMA kernels with Q = [W | R]; more go through the FP64 tensor-pipe kernel
// (scan_mt.cu) with Q = [1 | W | R], the k covariate vectors plus up to 31 - k traits per pass.
struct Pass {
  int64_t t0;
  int tcount, M, stride;
  bool mt;
  DevBuf<double> dQ, dyMy, dWy;
  DevBuf<int8_t> dDigits;  // M <= 2 without the tensor-pipe kernel: digits for the code matrix' tcgen05 kernel
  SideDigits digits;
  Pass(int64_t t0_, int tcount_, int M_, int stride_, bool mt_, size_t qcount, int k, size_t digit_bytes, cudaStream_t s)
      : t0(t0_), tcount(tcount_), M(M_), stride(stride_), mt(mt_), dQ(qcount, s), dyMy(tcount_ > 0 ? tcount_ : 1, s),
        dWy(static_cast<size_t>(tcount_ > 0 ? tcount_ : 1) * (k > 0 ? k : 1), s), dDigits(digit_bytes, s) {}
};

static std::vector<std::unique_ptr<Pass>> build_passes(const SideVectors& sv, int64_t n, int64_t T) {
  State& st = state();
  const int k = sv.k_eff;
  const bool mt = k + T > 2 && getenv("GBM_SCAN_NO_DMMA") == nullptr;
  const int max_m = mt ? scan_mt_max_side_vectors() : scan_max_side_vectors();
  if (k >= max_m) GBM_THROW(GBM_ERR_ARGUMENT, "too many covariates (at most " + std::to_string(max_m - 1) + ")");
  const int t_per_pass = max_m - k;
  const int64_t ldq = round_up(n, 2);
  std::vector<std::unique_ptr<Pass>> passes;
  for (int64_t t0 = 0; t0 < T; t0 += t_per_pass) {
    const int tcount = static_cast<int>(std::min<int64_t>(t_per_pass, T - t0));
    const int M = k + tcount;
    const int stride = mt ? 2 + M : scan_record_stride(M, false);
    const int ncols = mt ? M + 1 : stride - 2;  // columns of the device Q (padded for the FMA kernels)
    const int first = mt ? 1 : 0;               // [1 | W | R] for the tensor-pipe kernel
    const bool want_digits = !mt && M >= 1 && M <= 2;
    const int64_t ldd = scan_u8_tc_digit_rows(n);
    std::unique_ptr<Pass> ps(new Pass(t0, tcount, M, stride, mt, static_cast<size_t>(ldq) * ncols, k,
                                      want_digits ? static_cast<size_t>(16) * ldd : 0, st.stream));
    std::vector<int8_t> hdig;
    if (want_digits) {
      std::vector<double> hq(static_cast<size_t>(n) * M);
      if (k > 0) memcpy(hq.data(), sv.W.data(), sizeof(double) * n * k);
      memcpy(hq.data() + static_cast<size_t>(n) * k, sv.R.data() + static_cast<size_t>(t0) * n, sizeof(double) * n * tcount);
      hdig.resize(static_cast<size_t>(16) * ldd);
      scan_u8_tc_build_digits(hq.data(), n, M, n, hdig.data(), ldd, ps->digits.scale);
      GBM_CUDA(cudaMemcpyAsync(ps->dDigits.p, hdig.data(), hdig.size(), cudaMemcpyHostToDevice, st.stream));
      ps->digits.d = ps->dDigits.p;
      ps->digits.ld = ldd;
    }
    GBM_CUDA(cudaMemsetAsync(ps->dQ.p, 0, sizeof(double) * ldq * ncols, st.stream));
    std::vector<double> ones;
    if (mt) {
      ones.assign(static_cast<size_t>(n), 1.0);
      GBM_CUDA(cudaMemcpyAsync(ps->dQ.p, ones.data(), sizeof(double) * n, cudaMemcpyHostToDevice, st.stream));
    }
    if (k > 0)
      GBM_CUDA(cudaMemcpy2DAsync(ps->dQ.p + static_cast<size_t>(first) * ldq, ldq * sizeof(double), sv.W.data(),
                                 n * sizeof(double), n * sizeof(double), k, cudaMemcpyHostToDevice, st.stream));
    GBM_CUDA(cudaMemcpy2DAsync(ps->dQ.p + static_cast<size_t>(first + k) * ldq, ldq * sizeof(double),
                               sv.R.data() + static_cast<size_t>(t0) * n, n * sizeof(double), n * sizeof(double),
                               tcount, cudaMemcpyHostToDevice, st.stream));
    GBM_CUDA(cudaMemcpyAsync(ps->dyMy.p, sv.yMy.data() + t0, sizeof(double) * tcount, cudaMemcpyHostToDevice,
                             st.stream));
    if (k > 0)
      GBM_CUDA(cudaMemcpyAsync(ps->dWy.p, sv.wy.data() + static_cast<size_t>(t0) * k, sizeof(double) * tcount * k,
                               cudaMemcpyHostToDevice, st.stream));
    // the host vectors are pageable: make sure the copies have drained before they go away
    GBM_CUDA(cudaStreamSynchronize(st.stream));
    passes.push_back(std::move(ps));
  }
  return passes;
}

// Streaming pass(es) + finalisation over a device-resident column block.  dev_out holds
// DEVICE arrays of the full problem (leading dimension ld_out); this block writes entries
// col0 .. col0 + p_blk - 1 of each trait column.
struct ScanOutputs {
  double *beta, *se, *stat, *nlp, *mean, *sd;
  uint8_t* keep;
};

static void scan_block(const gbm_matrix& mat, int64_t p_blk, const std::vector<std::unique_ptr<Pass>>& passes,
                       const std::vector<double*>& rec_bufs, int k_eff, int model, int flags,
                       const ScanOutputs& dev_out, int64_t ld_out, int64_t col0, Span* main_span) {
  const int64_t n = mat.n;
  State& st = state();
  const int64_t ldq = round_up(n, 2);
  for (size_t pi = 0; pi < passes.size(); ++pi) {
    const auto& ps = passes[pi];
    const bool own_rec = rec_bufs.empty();
    DevBuf<double> rec_tmp(own_rec ? static_cast<size_t>(p_blk) * ps->stride : 0, st.stream);
    struct { double* p; } rec{own_rec ? rec_tmp.p : rec_bufs[pi]};
    if (main_span) main_span->start();
    scan_sums_any(&mat, 0, p_blk, ps->dQ.p, ps->M, ldq, rec.p, ps->mt, ps->stride, &ps->digits);
    if (main_span) main_span->stop();
    FinalizeParams fp;
    fp.n = n;
    fp.p = p_blk;
    fp.ld_out = ld_out;
    fp.k = k_eff;
    fp.T = ps->tcount;
    fp.rec_stride = ps->stride;
    fp.model = model;
    fp.flags = flags;
    fp.rec = rec.p;
    fp.yMy = ps->dyMy.p;
    fp.wy = ps->dWy.p;
    auto off = [&](double* base) { return base ? base + ps->t0 * ld_out + col0 : nullptr; };
    fp.beta = off(dev_out.beta);
    fp.se = off(dev_out.se);
    fp.stat = off(dev_out.stat);
    fp.nlp = off(dev_out.nlp);
    const bool first = ps->t0 == 0;
    fp.mean = (first && dev_out.mean) ? dev_out.mean + col0 : nullptr;
    fp.sd = (first && dev_out.sd) ? dev_out.sd + col0 : nullptr;
    fp.keep = (first && dev_out.keep) ? dev_out.keep + col0 : nullptr;
    launch_scan_finalize(fp, st.stream);
    st.launches += 2;
  }
}

// ------------------------------------------------------------------------------------
// host -> device ingestion of a column-major Float64 matrix
// ------------------------------------------------------------------------------------
// Up to kHostSlots column blocks are queued with the host workers ahead of the one being waited for.
// submit(slot, j0, pc) queues the block's job, consume(slot, j0, pc, ok) runs in block order; consume
// returning false stops the pipeline (queued jobs are drained first).  Returns true when every block
// was consumed.
template <typename Submit, typename Consume>
static bool run_block_pipeline(int64_t p, int64_t blk, Submit submit, Consume consume) {
  constexpr int K = State::kHostSlots;
  struct Ring {
    PackJob* job[K] = {};
    int64_t j0[K] = {};
    int head = 0, fill = 0, count = 0;
    ~Ring() {
      for (PackJob*& j : job)
        if (j) pack_wait(j, nullptr), j = nullptr;
    }
  } ring;
  int64_t next = 0;
  for (;;) {
    while (ring.count < K && next < p) {
      const int s = ring.fill;
      const int64_t pc = std::min(blk, p - next);
      ring.job[s] = submit(s, next, pc);
      ring.j0[s] = next;
      ring.fill = (s + 1) % K;
      ++ring.count;
      next += pc;
    }
    if (ring.count == 0) return true;
    const int s = ring.head;
    PackJob* job = ring.job[s];
    ring.job[s] = nullptr;
    ring.head = (s + 1) % K;
    --ring.count;
    const bool ok = pack_wait(job, nullptr);
    if (!consume(s, ring.j0[s], std::min(blk, p - ring.j0[s]), ok)) return false;
  }
}

// A (host or device, pitch lda) -> dst (device, pitch ldd >= n, pad rows zeroed).  Page-locked and device
// sources go through the copy engine directly.  Pageable sources are copied (and re-pitched) by the host
// workers into a ring of pinned staging blocks that the copy engine drains, instead of the driver's
// single-threaded bounce buffer.
static void upload_f64(const double* A, int64_t n, int64_t p, int64_t lda, double* dst, int64_t ldd) {
  State& st = state();
  if (is_device_ptr(A) || is_pinned_host_ptr(A) || host_threads() < 2) {
    if (ldd != n) GBM_CUDA(cudaMemsetAsync(dst, 0, sizeof(double) * ldd * p, st.stream));
    GBM_CUDA(cudaMemcpy2DAsync(dst, ldd * sizeof(double), A, lda * sizeof(double), n * sizeof(double), p,
                               cudaMemcpyDefault, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
    return;
  }
  constexpr int K = State::kHostSlots;
  const int64_t blk = std::max<int64_t>(16, ((int64_t(64) << 20) / (8 * ldd)) / 16 * 16);
  const size_t need = sizeof(double) * ldd * std::min(blk, p);
  if (st.up_bytes < need) {
    for (int b = 0; b < K; ++b) {
      if (st.up_stage[b]) cudaFreeHost(st.up_stage[b]);
      st.up_stage[b] = nullptr;
      GBM_CUDA(cudaMallocHost(&st.up_stage[b], need));
    }
    st.up_bytes = need;
  }
  for (int b = 0; b < K; ++b)
    if (!st.up_copied[b]) GBM_CUDA(cudaEventCreateWithFlags(&st.up_copied[b], cudaEventDisableTiming));
  run_block_pipeline(
      p, blk,
      [&](int s, int64_t j0, int64_t pc) {
        GBM_CUDA(cudaEventSynchronize(st.up_copied[s]));  // the staging block's previous H2D has drained
        return copy_submit(A + j0 * lda, n, lda, pc, static_cast<double*>(st.up_stage[s]), ldd);
      },
      [&](int s, int64_t j0, int64_t pc, bool) {
        GBM_CUDA(cudaMemcpyAsync(dst + j0 * ldd, st.up_stage[s], sizeof(double) * ldd * pc, cudaMemcpyHostToDevice,
                                 st.copy_stream));
        GBM_CUDA(cudaEventRecord(st.up_copied[s], st.copy_stream));
        return true;
      });
  GBM_CUDA(cudaStreamSynchronize(st.copy_stream));
}

// A (host, pitch lda) -> one-byte codes at d8 (device, pitch ld8), packed by the host workers.  Returns false
// (d8 incomplete) as soon as a block holds an element that is not exactly a code.
static bool upload_codes(const double* A, int64_t n, int64_t p, int64_t lda, uint8_t* d8, int64_t ld8) {
  State& st = state();
  constexpr int K = State::kHostSlots;
  const int64_t blk = std::max<int64_t>(16, ((int64_t(128) << 20) / (8 * n)) / 16 * 16);
  const size_t need8 = static_cast<size_t>(ld8) * std::min(blk, round_up(p, 16));
  if (st.code_bytes < need8) {
    for (int b = 0; b < K; ++b) {
      if (st.host_codes[b]) cudaFreeHost(st.host_codes[b]);
      if (st.dev_codes[b]) cudaFree(st.dev_codes[b]);
      st.host_codes[b] = st.dev_codes[b] = nullptr;
      GBM_CUDA(cudaMallocHost(&st.host_codes[b], need8));
      GBM_CUDA(cudaMalloc(&st.dev_codes[b], need8));
    }
    st.code_bytes = need8;
  }
  for (int b = 0; b < K; ++b)
    if (!st.hl_copied[b]) GBM_CUDA(cudaEventCreateWithFlags(&st.hl_copied[b], cudaEventDisableTiming));
  const bool all = run_block_pipeline(
      p, blk,
      [&](int s, int64_t j0, int64_t pc) {
        GBM_CUDA(cudaEventSynchronize(st.hl_copied[s]));
        return pack_submit(A + j0 * lda, n, lda, pc, static_cast<uint8_t*>(st.host_codes[s]), ld8);
      },
      [&](int s, int64_t j0, int64_t pc, bool ok) {
        if (!ok) return false;
        GBM_CUDA(cudaMemcpyAsync(d8 + j0 * ld8, st.host_codes[s], static_cast<size_t>(ld8) * pc, cudaMemcpyHostToDevice,
                                 st.copy_stream));
        GBM_CUDA(cudaEventRecord(st.hl_copied[s], st.copy_stream));
        return true;
      });
  GBM_CUDA(cudaStreamSynchronize(st.copy_stream));
  return all;
}

void init_state(State& st, int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    GBM_THROW(GBM_ERR_CUDA, "no CUDA device: libgbm_b200 has no CPU fallback");
  if (device < 0 || device >= count) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_init: device index out of range");
  GBM_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  GBM_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    GBM_THROW(GBM_ERR_CUDA, std::string("libgbm_b200 is built for sm_100a (B200) only; found ") + prop.name);
  if (st.ready && st.device == device) return;
  if (st.ready) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_init: already initialised on another device; call gbm_shutdown first");
  st.device = device;
  st.sm_count = prop.multiProcessorCount;
  if (!st.own_stream) GBM_CUDA(cudaStreamCreateWithFlags(&st.own_stream, cudaStreamNonBlocking));
  if (!st.copy_stream) GBM_CUDA(cudaStreamCreateWithFlags(&st.copy_stream, cudaStreamNonBlocking));
  st.stream = st.own_stream;
  {  // keep stream-ordered scratch allocations cached instead of returning them at every sync
    cudaMemPool_t pool;
    GBM_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t thr = UINT64_MAX;
    GBM_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
  }
  st.ready = true;
}

void shutdown_state(State& st) {
  if (!st.ready) return;
  cudaSetDevice(st.device);
  cudaStreamSynchronize(st.stream);
  if (st.cusolver) {
    cusolverDnDestroy(reinterpret_cast<cusolverDnHandle_t>(st.cusolver));
    st.cusolver = nullptr;
  }
  free_scan_host_staging(st);
  if (st.own_stream) cudaStreamDestroy(st.own_stream);
  if (st.copy_stream) cudaStreamDestroy(st.copy_stream);
  if (st.raw_stream) cudaStreamDestroy(st.raw_stream);
  st.own_stream = st.copy_stream = st.raw_stream = st.stream = nullptr;
  st.ready = false;
}

}  // namespace gbm

using namespace gbm;

// Error exit of an entry point: nothing of the call may still be reading the caller's host buffers or writing
// its outputs after the return ("host pointers are never retained"), so wait for every stream of this State.
static void drain_streams() {
  State& st = state();
  if (!st.ready) return;
  if (st.stream) cudaStreamSynchronize(st.stream);
  if (st.copy_stream) cudaStreamSynchronize(st.copy_stream);
  if (st.raw_stream) cudaStreamSynchronize(st.raw_stream);
  cudaGetLastError();
}

#define GBM_API_BEGIN                            \
  std::lock_guard<std::mutex> lock__(gbm::state().api_mutex); \
  try {
#define GBM_API_END                              \
  }                                              \
  catch (const gbm::Error& e) {                  \
    drain_streams();                             \
    set_error(e.msg);                            \
    return e.code;                               \
  }                                              \
  catch (const std::exception& e) {              \
    drain_streams();                             \
    set_error(std::string("internal: ") + e.what()); \
    return GBM_ERR_RUNTIME;                      \
  }                                              \
  return GBM_OK;

extern "C" {

int gbm_abi_version(void) { return GBM_ABI_VERSION; }
const char* gbm_last_error(void) { return g_error.c_str(); }

int gbm_init(int device) {
  GBM_API_BEGIN
  init_state(state(), device);
  GBM_API_END
}

int gbm_shutdown(void) {
  GBM_API_BEGIN
  shutdown_state(state());
  GBM_API_END
}

int gbm_set_stream(void* cuda_stream) {
  GBM_API_BEGIN
  require_ready();
  State& st = state();
  st.stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : st.own_stream;
  GBM_API_END
}

int gbm_synchronize(void) {
  GBM_API_BEGIN
  require_ready();
  GBM_CUDA(cudaStreamSynchronize(state().stream));
  GBM_API_END
}

int gbm_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes, char* name, int name_len) {
  GBM_API_BEGIN
  require_ready();
  cudaDeviceProp prop;
  GBM_CUDA(cudaGetDeviceProperties(&prop, state().device));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (hbm_bytes) *hbm_bytes = static_cast<int64_t>(prop.totalGlobalMem);
  if (name && name_len > 0) {
    strncpy(name, prop.name, name_len - 1);
    name[name_len - 1] = 0;
  }
  GBM_API_END
}

int gbm_last_timing(gbm_timing* t) {
  GBM_API_BEGIN
  if (!t) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_last_timing: null output");
  State& st = state();
  t->h2d_ms = st.h2d_ms;
  t->kernel_ms = st.kernel_ms;
  t->main_ms = st.main_ms;
  t->d2h_ms = st.d2h_ms;
  t->launches = st.launches;
  t->packed_blocks = st.packed_blocks;
  t->host_packed_blocks = st.host_packed_blocks;
  t->h2d_bytes = st.h2d_bytes;
  GBM_API_END
}

// ------------------------------------------------------------------------------------
// matrices
// ------------------------------------------------------------------------------------
// Slabs below 1 GB come from the device's stream-ordered pool (release threshold: never), so a steady stream of
// small problems (BASELINE configs[0]: 24 MB per call) makes no cudaMalloc / cudaFree driver calls -- those cost ~1.3 ms
// each and were the source of sporadic 0.03-0.8 s stalls; large slabs stay plain allocations that go back to the
// driver when freed (an 80 GB matrix must not stay parked in a pool).
static cudaError_t slab_malloc(gbm_matrix* m, void** ptr, size_t bytes) {
  if (bytes <= (size_t(1) << 30)) {
    m->pooled = true;
    cudaError_t e = cudaMallocAsync(ptr, bytes, state().stream);
    // the slab is filled from other streams too (copy engine lanes): make the allocation point visible to all of them
    if (e == cudaSuccess) e = cudaStreamSynchronize(state().stream);
    return e;
  }
  m->pooled = false;
  return cudaMalloc(ptr, bytes);
}
static void slab_free(gbm_matrix* m) {
  if (m->pooled && state().ready) {
    if (m->d) cudaFreeAsync(m->d, state().stream);
    if (m->d8) cudaFreeAsync(m->d8, state().stream);
  } else {
    if (m->d) cudaFree(m->d);
    if (m->d8) cudaFree(m->d8);
  }
  m->d = nullptr;
  m->d8 = nullptr;
}

// owns a half-built matrix until it is handed to the caller (an exception in between frees the slab and the handle)
struct MatGuard {
  gbm_matrix* m;
  explicit MatGuard(gbm_matrix* mm) : m(mm) {}
  ~MatGuard() {
    if (m) {
      slab_free(m);
      delete m;
    }
  }
  gbm_matrix* release() {
    gbm_matrix* r = m;
    m = nullptr;
    return r;
  }
};

static void check_dims(int64_t n, int64_t p, int64_t lda) {
  if (n < 2) GBM_THROW(GBM_ERR_ARGUMENT, "matrix needs at least 2 rows (entries)");
  if (p < 1) GBM_THROW(GBM_ERR_ARGUMENT, "matrix needs at least 1 column (locus-allele)");
  if (lda < n) GBM_THROW(GBM_ERR_ARGUMENT, "leading dimension smaller than the row count");
  if (n > (int64_t(1) << 31) - 512 || p > (int64_t(1) << 31) - 512)
    GBM_THROW(GBM_ERR_ARGUMENT, "dimension exceeds the 2^31 tensor-map coordinate range");
}

int gbm_matrix_upload(const double* A, int64_t n, int64_t p, int64_t lda, gbm_matrix** out) {
  GBM_API_BEGIN
  require_ready();
  if (!A || !out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_upload: null pointer");
  check_dims(n, p, lda);
  State& st = state();
  reset_timing();
  gbm_matrix* m = new gbm_matrix;
  m->n = n;
  m->p = p;
  m->lda = round_up(n, 16);
  m->owned = true;
  cudaError_t e = slab_malloc(m, reinterpret_cast<void**>(&m->d), sizeof(double) * m->lda * p);
  if (e != cudaSuccess) {
    delete m;
    GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the genotype slab failed: ") + cudaGetErrorString(e));
  }
  const auto t0 = std::chrono::steady_clock::now();
  try {
    upload_f64(A, n, p, lda, m->d, m->lda);
  } catch (...) {
    slab_free(m);
    delete m;
    throw;
  }
  st.h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  *out = m;
  GBM_API_END
}

int gbm_matrix_upload_compact(const double* A, int64_t n, int64_t p, int64_t lda, gbm_matrix** out, int* packed) {
  GBM_API_BEGIN
  require_ready();
  if (!A || !out || !packed) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_upload_compact: null pointer");
  check_dims(n, p, lda);
  State& st = state();
  reset_timing();
  *packed = 0;
  const auto t0 = std::chrono::steady_clock::now();
  if (!is_device_ptr(A) && host_threads() >= 2) {
    std::unique_ptr<gbm_matrix> q(new gbm_matrix);
    q->n = n;
    q->p = p;
    q->dtype = 1;
    q->owned = true;
    q->ld8 = round_up(n, 128);
    cudaError_t e = slab_malloc(q.get(), reinterpret_cast<void**>(&q->d8), static_cast<size_t>(q->ld8) * p);
    if (e != cudaSuccess) GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the code slab failed: ") + cudaGetErrorString(e));
    bool all = false;
    try {
      all = upload_codes(A, n, p, lda, q->d8, q->ld8);
    } catch (...) {
      slab_free(q.get());
      throw;
    }
    if (all) {
      st.h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      st.h2d_bytes = q->ld8 * p;
      *packed = 1;
      *out = q.release();
      return GBM_OK;
    }
    slab_free(q.get());  // not dosage data: Float64 slab below
  }
  gbm_matrix* m = new gbm_matrix;
  m->n = n;
  m->p = p;
  m->lda = round_up(n, 16);
  m->owned = true;
  cudaError_t e = slab_malloc(m, reinterpret_cast<void**>(&m->d), sizeof(double) * m->lda * p);
  if (e != cudaSuccess) {
    delete m;
    GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the genotype slab failed: ") + cudaGetErrorString(e));
  }
  try {
    upload_f64(A, n, p, lda, m->d, m->lda);
  } catch (...) {
    slab_free(m);
    delete m;
    throw;
  }
  st.h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  st.h2d_bytes = static_cast<int64_t>(sizeof(double)) * n * p;
  *out = m;
  GBM_API_END
}

int gbm_matrix_upload_indexed(const double* A, int64_t n0, int64_t p0, int64_t lda, const int64_t* rows, int64_t n,
                              const int64_t* cols, int64_t p, gbm_matrix** out) {
  GBM_API_BEGIN
  require_ready();
  if (!A || !out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_upload_indexed: null pointer");
  check_dims(n0, p0, lda);
  if (!rows) n = n0;
  if (!cols) p = p0;
  check_dims(n, p, n);
  State& st = state();
  reset_timing();
  // index validation mirrors extractxyetc (/root/reference/src/prediction.jl:82-111)
  std::vector<int64_t> hr, hc;
  if (rows) {
    hr.resize(n);
    GBM_CUDA(cudaMemcpy(hr.data(), rows, sizeof(int64_t) * n, cudaMemcpyDefault));
    for (int64_t v : hr)
      if (v < 1 || v > n0) GBM_THROW(GBM_ERR_ARGUMENT, "The indexes of the entries, `idx_entries` are out of bounds.");
  }
  if (cols) {
    hc.resize(p);
    GBM_CUDA(cudaMemcpy(hc.data(), cols, sizeof(int64_t) * p, cudaMemcpyDefault));
    for (int64_t v : hc)
      if (v < 1 || v > p0)
        GBM_THROW(GBM_ERR_ARGUMENT, "The indexes of the loci_alleles, `idx_loci_alleles` are out of bounds.");
  }
  gbm_matrix* m = new gbm_matrix;
  m->n = n;
  m->p = p;
  m->lda = round_up(n, 16);
  m->owned = true;
  cudaError_t e = slab_malloc(m, reinterpret_cast<void**>(&m->d), sizeof(double) * m->lda * p);
  if (e != cudaSuccess) {
    delete m;
    GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the genotype slab failed: ") + cudaGetErrorString(e));
  }
  MatGuard guard(m);
  GBM_CUDA(cudaMemsetAsync(m->d, 0, sizeof(double) * m->lda * p, st.stream));
  DevBuf<int64_t> dr(rows ? n : 0, st.stream), dc(cols ? p : 0, st.stream);
  if (rows) GBM_CUDA(cudaMemcpyAsync(dr.p, hr.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, st.stream));
  if (cols) GBM_CUDA(cudaMemcpyAsync(dc.p, hc.data(), sizeof(int64_t) * p, cudaMemcpyHostToDevice, st.stream));
  // stage source columns through the device in blocks, gather on the device
  const bool src_dev = is_device_ptr(A);
  const int64_t blk = std::max<int64_t>(1, std::min<int64_t>(p, (int64_t(256) << 20) / (8 * n0)));
  DevBuf<double> stage(src_dev ? 0 : static_cast<size_t>(n0) * blk, st.stream);
  Span sp(st.stream);
  sp.start();
  for (int64_t j0 = 0; j0 < p; j0 += blk) {
    const int64_t pc = std::min(blk, p - j0);
    if (src_dev) {
      launch_gather(A, lda, rows ? dr.p : nullptr, n, cols ? dc.p + j0 : nullptr, pc, m->d + j0 * m->lda, m->lda,
                    st.stream);
      if (!cols) A += pc * lda;
    } else {
      // copy the needed source columns contiguously into the stage (cols gathers on the host side of the copy)
      if (!cols) {
        GBM_CUDA(cudaMemcpy2DAsync(stage.p, n0 * sizeof(double), A + j0 * lda, lda * sizeof(double),
                                   n0 * sizeof(double), pc, cudaMemcpyDefault, st.stream));
      } else {
        for (int64_t j = 0; j < pc; ++j)
          GBM_CUDA(cudaMemcpyAsync(stage.p + j * n0, A + (hc[j0 + j] - 1) * lda, sizeof(double) * n0,
                                   cudaMemcpyDefault, st.stream));
      }
      launch_gather(stage.p, n0, rows ? dr.p : nullptr, n, nullptr, pc, m->d + j0 * m->lda, m->lda, st.stream);
    }
    st.launches++;
  }
  sp.stop();
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  st.h2d_ms = sp.ms();
  *out = guard.release();
  GBM_API_END
}

int gbm_matrix_wrap(double* dA, int64_t n, int64_t p, int64_t lda, gbm_matrix** out) {
  GBM_API_BEGIN
  require_ready();
  if (!dA || !out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_wrap: null pointer");
  check_dims(n, p, lda);
  if (!is_device_ptr(dA)) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_wrap: not a device pointer");
  if ((lda & 1) || (reinterpret_cast<uintptr_t>(dA) & 15u))
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_wrap: needs a 16-byte aligned buffer with an even leading dimension");
  gbm_matrix* m = new gbm_matrix;
  m->d = dA;
  m->n = n;
  m->p = p;
  m->lda = lda;
  m->owned = false;
  *out = m;
  GBM_API_END
}

int gbm_matrix_generate(uint64_t seed, int64_t n, int64_t p, int64_t col0, int kind, gbm_matrix** out) {
  GBM_API_BEGIN
  require_ready();
  if (!out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_generate: null pointer");
  check_dims(n, p, n);
  if (kind < 0 || kind > 2) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_generate: unknown kind");
  State& st = state();
  gbm_matrix* m = new gbm_matrix;
  m->n = n;
  m->p = p;
  m->lda = round_up(n, 16);
  m->owned = true;
  cudaError_t e = slab_malloc(m, reinterpret_cast<void**>(&m->d), sizeof(double) * m->lda * p);
  if (e != cudaSuccess) {
    delete m;
    GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the genotype slab failed: ") + cudaGetErrorString(e));
  }
  MatGuard guard(m);
  if (m->lda != n) GBM_CUDA(cudaMemsetAsync(m->d, 0, sizeof(double) * m->lda * p, st.stream));
  launch_generate(m->d, n, p, m->lda, col0, seed, kind, st.stream);
  GBM_CUDA(cudaGetLastError());
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  *out = guard.release();
  GBM_API_END
}

int gbm_matrix_pack(const gbm_matrix* m, gbm_matrix** out, int64_t* n_inexact) {
  GBM_API_BEGIN
  require_ready();
  if (!m || !out || !n_inexact) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_pack: null pointer");
  if (m->dtype != 0) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_pack: the matrix is already packed");
  State& st = state();
  *out = nullptr;
  std::unique_ptr<gbm_matrix> q(new gbm_matrix);
  q->n = m->n;
  q->p = m->p;
  q->dtype = 1;
  q->owned = true;
  q->ld8 = round_up(m->n, 128);
  cudaError_t e = slab_malloc(q.get(), reinterpret_cast<void**>(&q->d8), static_cast<size_t>(q->ld8) * m->p);
  if (e != cudaSuccess) GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the code slab failed: ") + cudaGetErrorString(e));
  DevBuf<unsigned long long> bad(1, st.stream);
  GBM_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(unsigned long long), st.stream));
  launch_pack_u8(m->d, m->n, m->p, m->lda, q->d8, q->ld8, bad.p, st.stream);
  unsigned long long h = 0;
  GBM_CUDA(cudaMemcpyAsync(&h, bad.p, sizeof(h), cudaMemcpyDeviceToHost, st.stream));
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  *n_inexact = static_cast<int64_t>(h);
  if (h != 0) {
    slab_free(q.get());  // not every element is a dosage code: the Float64 path must be used
    return GBM_OK;
  }
  *out = q.release();
  GBM_API_END
}

int gbm_matrix_upload_packed(const uint8_t* codes, int64_t n, int64_t p, int64_t ld, gbm_matrix** out) {
  GBM_API_BEGIN
  require_ready();
  if (!codes || !out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_upload_packed: null pointer");
  check_dims(n, p, ld);
  State& st = state();
  std::unique_ptr<gbm_matrix> q(new gbm_matrix);
  q->n = n;
  q->p = p;
  q->dtype = 1;
  q->owned = true;
  q->ld8 = round_up(n, 128);
  cudaError_t e = slab_malloc(q.get(), reinterpret_cast<void**>(&q->d8), static_cast<size_t>(q->ld8) * p);
  if (e != cudaSuccess) GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the code slab failed: ") + cudaGetErrorString(e));
  GBM_CUDA(cudaMemsetAsync(q->d8, 0, static_cast<size_t>(q->ld8) * p, st.stream));
  GBM_CUDA(cudaMemcpy2DAsync(q->d8, q->ld8, codes, ld, n, p, cudaMemcpyDefault, st.stream));
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  *out = q.release();
  GBM_API_END
}

int gbm_matrix_download(const gbm_matrix* m, int64_t j0, int64_t ncols, double* dst, int64_t ldd) {
  GBM_API_BEGIN
  require_ready();
  if (!m || !dst) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_download: null pointer");
  if (j0 < 0 || ncols < 0 || j0 + ncols > m->p || ldd < m->n)
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_download: range out of bounds");
  State& st = state();
  if (m->dtype == 1) {
    const int64_t ldt = round_up(m->n, 16);
    DevBuf<double> tmp(static_cast<size_t>(ldt) * std::max<int64_t>(ncols, 1), st.stream);
    launch_decode_u8(m->d8 + j0 * m->ld8, m->n, ncols, m->ld8, tmp.p, ldt, st.stream);
    GBM_CUDA(cudaMemcpy2DAsync(dst, ldd * sizeof(double), tmp.p, ldt * sizeof(double), m->n * sizeof(double), ncols,
                               cudaMemcpyDefault, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
    return GBM_OK;
  }
  GBM_CUDA(cudaMemcpy2DAsync(dst, ldd * sizeof(double), m->d + j0 * m->lda, m->lda * sizeof(double),
                             m->n * sizeof(double), ncols, cudaMemcpyDefault, st.stream));
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  GBM_API_END
}

int gbm_matrix_download_cols(const gbm_matrix* m, const int64_t* idx_cols, int64_t ncols, int standardise,
                             double* dst, int64_t ldd) {
  GBM_API_BEGIN
  require_ready();
  if (!m || !dst || ncols < 0 || ldd < m->n) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_download_cols: bad arguments");
  if (!idx_cols && ncols != m->p) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_download_cols: ncols must be p without an index");
  if (ncols == 0) return GBM_OK;
  State& st = state();
  const int64_t n = m->n;
  DevBuf<int64_t> dcols(idx_cols ? ncols : 0, st.stream);
  if (idx_cols) {
    std::vector<int64_t> hc(ncols);
    GBM_CUDA(cudaMemcpy(hc.data(), idx_cols, sizeof(int64_t) * ncols, cudaMemcpyDefault));
    for (int64_t v : hc)
      if (v < 1 || v > m->p) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_download_cols: column index out of bounds");
    GBM_CUDA(cudaMemcpyAsync(dcols.p, hc.data(), sizeof(int64_t) * ncols, cudaMemcpyHostToDevice, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
  }
  DevBuf<double> dmean(standardise ? m->p : 0, st.stream), dsd(standardise ? m->p : 0, st.stream);
  if (standardise) {  // column mean / sd by the streaming kernel (gwas.jl:112, :129)
    const int stride = scan_record_stride(0, true);
    DevBuf<double> rec(static_cast<size_t>(m->p) * stride, st.stream);
    scan_sums_any(m, 0, m->p, nullptr, 0, 0, rec.p);
    launch_colstats_finalize(rec.p, stride, n, m->p, dmean.p, dsd.p, nullptr, nullptr, st.stream);
  }
  // gather (+ standardise) column blocks on the device, copy each block out
  const int64_t ldt = round_up(n, 16);
  const int64_t PB = std::max<int64_t>(1, std::min<int64_t>(ncols, (int64_t(256) << 20) / (8 * ldt)));
  DevBuf<double> tmp(static_cast<size_t>(ldt) * PB, st.stream);
  for (int64_t c0 = 0; c0 < ncols; c0 += PB) {
    const int64_t pc = std::min(PB, ncols - c0);
    const double* mu = standardise ? (idx_cols ? dmean.p : dmean.p + c0) : nullptr;
    const double* sdv = standardise ? (idx_cols ? dsd.p : dsd.p + c0) : nullptr;
    if (m->dtype == 1)
      launch_gather_standardise_u8(idx_cols ? m->d8 : m->d8 + c0 * m->ld8, m->ld8, n, idx_cols ? dcols.p + c0 : nullptr,
                                   pc, mu, sdv, tmp.p, ldt, st.stream);
    else
      launch_gather_standardise(idx_cols ? m->d : m->d + c0 * m->lda, m->lda, n, idx_cols ? dcols.p + c0 : nullptr, pc,
                                mu, sdv, tmp.p, ldt, st.stream);
    GBM_CUDA(cudaMemcpy2DAsync(dst + c0 * ldd, ldd * sizeof(double), tmp.p, ldt * sizeof(double), n * sizeof(double),
                               pc, cudaMemcpyDefault, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
  }
  GBM_API_END
}

int gbm_matrix_info(const gbm_matrix* m, int64_t* n, int64_t* p, int64_t* lda, double** device_ptr) {
  GBM_API_BEGIN
  if (!m) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_matrix_info: null handle");
  if (n) *n = m->n;
  if (p) *p = m->p;
  if (lda) *lda = m->lda;
  if (lda && m->dtype == 1) *lda = m->ld8;
  if (device_ptr) *device_ptr = m->dtype == 1 ? reinterpret_cast<double*>(m->d8) : m->d;
  GBM_API_END
}

int gbm_matrix_free(gbm_matrix* m) {
  GBM_API_BEGIN
  if (m) {
    if (m->owned && (m->d || m->d8)) {
      if (state().ready) cudaStreamSynchronize(state().stream);
      slab_free(m);
    }
    delete m;
  }
  GBM_API_END
}

// ------------------------------------------------------------------------------------
// gwasprep pieces
// ------------------------------------------------------------------------------------
int gbm_colstats(const gbm_matrix* m, double* mean, double* sd, double* min_nonzero, uint8_t* keep,
                 int64_t* idx_cols, int64_t* n_keep, double* min_nonzero_kept) {
  GBM_API_BEGIN
  require_ready();
  if (!m) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_colstats: null handle");
  State& st = state();
  reset_timing();
  const int64_t p = m->p;
  const int stride = scan_record_stride(0, true);
  DevBuf<double> rec(static_cast<size_t>(p) * stride, st.stream);
  DevBuf<double> dmean(p, st.stream), dsd(p, st.stream), dmin(p, st.stream), dminkept(1, st.stream);
  DevBuf<uint8_t> dkeep(p, st.stream);
  DevBuf<int64_t> didx(p, st.stream), dcount(1, st.stream);
  Span all(st.stream), mainsp(st.stream);
  all.start();
  mainsp.start();
  scan_sums_any(m, 0, p, nullptr, 0, 0, rec.p);
  mainsp.stop();
  launch_colstats_finalize(rec.p, stride, m->n, p, dmean.p, dsd.p, dmin.p, dkeep.p, st.stream);
  launch_compact_keep(dkeep.p, dmin.p, p, didx.p, dcount.p, dminkept.p, st.stream);
  all.stop();
  st.launches = 3;
  Span d2h(st.stream);
  d2h.start();
  copy_out(mean, dmean.p, sizeof(double) * p, st.stream);
  copy_out(sd, dsd.p, sizeof(double) * p, st.stream);
  copy_out(min_nonzero, dmin.p, sizeof(double) * p, st.stream);
  copy_out(keep, dkeep.p, p, st.stream);
  int64_t count = 0;
  GBM_CUDA(cudaMemcpyAsync(&count, dcount.p, sizeof(int64_t), cudaMemcpyDeviceToHost, st.stream));
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  if (idx_cols && count > 0) copy_out(idx_cols, didx.p, sizeof(int64_t) * count, st.stream);
  copy_out(min_nonzero_kept, dminkept.p, sizeof(double), st.stream);
  if (n_keep) {
    if (is_device_ptr(n_keep))
      copy_out(n_keep, dcount.p, sizeof(int64_t), st.stream);
    else
      *n_keep = count;
  }
  d2h.stop();
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  st.kernel_ms = all.ms();
  st.main_ms = mainsp.ms();
  st.d2h_ms = d2h.ms();
  GBM_API_END
}

// ------------------------------------------------------------------------------------
// GRM
// ------------------------------------------------------------------------------------
static void column_means_padded(const gbm_matrix* m, double* dmu_pad /* round_up(p,16), zeroed */) {
  State& st = state();
  const int stride = scan_record_stride(0, true);
  DevBuf<double> rec(static_cast<size_t>(m->p) * stride, st.stream);
  scan_sums_any(m, 0, m->p, nullptr, 0, 0, rec.p);
  launch_colstats_finalize(rec.p, stride, m->n, m->p, dmu_pad, nullptr, nullptr, nullptr, st.stream);
  st.launches += 2;
}

static bool use_int8_grm() {
  static const bool v = [] { const char* e = getenv("GBM_GRM_INT8"); return e ? atoi(e) != 0 : true; }();
  return v;
}

static void grm_accumulate_impl(const gbm_matrix* m, int centre, double* dK, double* dsumq /*device, nullable*/,
                                double* tflops) {
  State& st = state();
  const int64_t ppad = round_up(m->p, 16);
  DevBuf<double> dmu(ppad, st.stream);
  GBM_CUDA(cudaMemsetAsync(dmu.p, 0, sizeof(double) * ppad, st.stream));
  Span all(st.stream), mainsp(st.stream);
  all.start();
  if (centre || dsumq) column_means_padded(m, dmu.p);
  if (dsumq) {
    launch_sum_q1mq(dmu.p, m->p, dsumq, st.stream);
    st.launches++;
  }
  if (!centre) GBM_CUDA(cudaMemsetAsync(dmu.p, 0, sizeof(double) * ppad, st.stream));
  mainsp.start();
  if (m->dtype == 0) {
    launch_grm_accumulate(m->d, m->n, m->p, m->lda, dmu.p, dK, st.sm_count, st.stream, centre != 0);
  } else if (use_int8_grm() && 57600.0 * static_cast<double>(m->n) * static_cast<double>(m->p) < 9007199254740992.0) {
    // (U_i = sum_j S_j c_ij <= 240 n * 240 * p must stay an exact FP64 integer)
    // packed codes: exact integer contraction on the tcgen05 INT8 tensor cores (grm_i8.cu)
    const int64_t n = m->n;
    DevBuf<double> dG(static_cast<size_t>(n) * n, st.stream), dS(m->p, st.stream), dU(n, st.stream), dM2(1, st.stream);
    GBM_CUDA(cudaMemsetAsync(dG.p, 0, sizeof(double) * n * n, st.stream));
    GBM_CUDA(cudaMemsetAsync(dU.p, 0, sizeof(double) * n, st.stream));
    GBM_CUDA(cudaMemsetAsync(dM2.p, 0, sizeof(double), st.stream));
    launch_grm_i8_accumulate(m->d8, n, m->p, m->ld8, dG.p, st.sm_count, st.stream);
    if (centre) {
      // dmu holds the column means (a scale): S_j = round(mu_j * n * 240) are the exact code sums
      launch_code_sums(dmu.p, m->p, n, dS.p, dM2.p, st.stream);
      launch_rowdot_u8(m->d8, n, m->p, m->ld8, dS.p, dU.p, st.stream);
    }
    launch_grm_i8_combine(dG.p, n, dU.p, dM2.p, centre, dK, st.stream);
    st.launches += 4;
  } else {
    // packed codes: decode column blocks (<= 1 GB of Float64) and accumulate block by block
    const int64_t ldt = round_up(m->n, 16);
    int64_t PB = std::max<int64_t>(16, ((int64_t(1) << 30) / (8 * ldt)) / 16 * 16);
    PB = std::min(PB, ppad);
    DevBuf<double> tmp(static_cast<size_t>(ldt) * PB, st.stream);
    for (int64_t j0 = 0; j0 < m->p; j0 += PB) {
      const int64_t pb = std::min(PB, m->p - j0);
      launch_decode_u8(m->d8 + j0 * m->ld8, m->n, pb, m->ld8, tmp.p, ldt, st.stream);
      launch_grm_accumulate(tmp.p, m->n, pb, ldt, dmu.p + j0, dK, st.sm_count, st.stream, centre != 0);
      st.launches += 2;
    }
  }
  mainsp.stop();
  all.stop();
  st.launches++;
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  st.kernel_ms += all.ms();
  const double ms = mainsp.ms();
  st.main_ms += ms;
  if (tflops) *tflops = static_cast<double>(m->n) * static_cast<double>(m->n + 1) * static_cast<double>(m->p) /
                        (ms * 1e-3) / 1e12;
}

int gbm_grm_accumulate(const gbm_matrix* m, int centre, double* dK, double* sum_q1mq, double* tflops) {
  GBM_API_BEGIN
  require_ready();
  if (!m || !dK) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_grm_accumulate: null pointer");
  if (!is_device_ptr(dK)) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_grm_accumulate: dK must be a device pointer");
  State& st = state();
  reset_timing();
  DevBuf<double> dsum(1, st.stream);
  GBM_CUDA(cudaMemsetAsync(dsum.p, 0, sizeof(double), st.stream));
  grm_accumulate_impl(m, centre, dK, sum_q1mq ? dsum.p : nullptr, tflops);
  if (sum_q1mq) {
    double h = 0.0;
    GBM_CUDA(cudaMemcpyAsync(&h, dsum.p, sizeof(double), cudaMemcpyDeviceToHost, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
    if (is_device_ptr(sum_q1mq)) {
      double prev = 0.0;
      GBM_CUDA(cudaMemcpy(&prev, sum_q1mq, sizeof(double), cudaMemcpyDeviceToHost));
      prev += h;
      GBM_CUDA(cudaMemcpy(sum_q1mq, &prev, sizeof(double), cudaMemcpyHostToDevice));
    } else {
      *sum_q1mq += h;
    }
  }
  GBM_API_END
}

int gbm_grm_finalize(double* dK, int64_t n, double scale) {
  GBM_API_BEGIN
  require_ready();
  if (!dK || n < 1) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_grm_finalize: bad arguments");
  if (!is_device_ptr(dK)) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_grm_finalize: dK must be a device pointer");
  State& st = state();
  launch_grm_finalize(dK, n, scale, st.stream);
  st.launches++;
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  GBM_API_END
}

int gbm_grm(const gbm_matrix* m, int grm_type, int ploidy, int flags, double* K, double* tflops) {
  GBM_API_BEGIN
  require_ready();
  if (!m || !K) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_grm: null pointer");
  if (grm_type != GBM_GRM_SIMPLE && grm_type != GBM_GRM_PLOIDY_AWARE)
    GBM_THROW(GBM_ERR_ARGUMENT, "Unrecognised `GRM_type`. Please select from:\n\t‣ simple\n\t‣ ploidy-aware");
  if (grm_type == GBM_GRM_PLOIDY_AWARE && ploidy < 1) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_grm: ploidy must be >= 1");
  State& st = state();
  reset_timing();
  const int64_t n = m->n;
  const bool dev_out = is_device_ptr(K);
  DevBuf<double> tmp(dev_out ? 0 : static_cast<size_t>(n) * n, st.stream);
  double* dK = dev_out ? K : tmp.p;
  GBM_CUDA(cudaMemsetAsync(dK, 0, sizeof(double) * n * n, st.stream));
  DevBuf<double> dsum(1, st.stream);
  GBM_CUDA(cudaMemsetAsync(dsum.p, 0, sizeof(double), st.stream));
  const int centre = (grm_type == GBM_GRM_PLOIDY_AWARE) ? 1 : ((flags & GBM_GRM_NO_CENTRE) ? 0 : 1);
  grm_accumulate_impl(m, centre, dK, grm_type == GBM_GRM_PLOIDY_AWARE ? dsum.p : nullptr, tflops);
  double scale = 1.0 / static_cast<double>(m->p);
  if (grm_type == GBM_GRM_PLOIDY_AWARE) {
    double h = 0.0;
    GBM_CUDA(cudaMemcpyAsync(&h, dsum.p, sizeof(double), cudaMemcpyDeviceToHost, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
    if (!(h > 0.0)) GBM_THROW(GBM_ERR_RUNTIME, "gbm_grm: sum q(1-q) is not positive (all loci fixed)");
    scale = static_cast<double>(ploidy) / h;
  }
  launch_grm_finalize(dK, n, scale, st.stream);
  st.launches++;
  if (!dev_out) {
    Span d2h(st.stream);
    d2h.start();
    GBM_CUDA(cudaMemcpyAsync(K, dK, sizeof(double) * n * n, cudaMemcpyDefault, st.stream));
    d2h.stop();
    st.d2h_ms = d2h.ms();
  }
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  GBM_API_END
}

// ------------------------------------------------------------------------------------
// K standardisation + PC1
// ------------------------------------------------------------------------------------
// Lanczos stops when the Ritz residual estimate is below kPc1Tol * theta; the explicit residual ||Bx - theta x|| is
// then required to be <= 2e-13 theta.  With the ~3e-3 relative gap of the standardised GRM's top eigenvalue that puts
// PC1 within ~1e-10 of the exact vector, two orders below the 1e-9 the statistics are held to.
static constexpr double kPc1Tol = 1e-13;

int gbm_kstd_pc1(const double* K, int64_t n, double* Kstd, double* pc1, double* eig_ms) {
  GBM_API_BEGIN
  require_ready();
  if (!K || n < 2) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_kstd_pc1: bad arguments");
  State& st = state();
  reset_timing();
  const int64_t ld = round_up(n, 16);
  DevBuf<double> dKs(static_cast<size_t>(ld) * n, st.stream);
  Span h2d(st.stream);
  h2d.start();
  if (ld != n) GBM_CUDA(cudaMemsetAsync(dKs.p, 0, sizeof(double) * ld * n, st.stream));
  GBM_CUDA(cudaMemcpy2DAsync(dKs.p, ld * sizeof(double), K, n * sizeof(double), n * sizeof(double), n,
                             cudaMemcpyDefault, st.stream));
  h2d.stop();
  Span all(st.stream);
  all.start();
  // column mean / sd of K through the streaming scan (two-pass-equivalent shifted sums)
  const int stride = scan_record_stride(0, true);
  DevBuf<double> rec(static_cast<size_t>(n) * stride, st.stream), dmean(n, st.stream), dsd(n, st.stream);
  launch_scan_sums(dKs.p, n, n, ld, nullptr, 0, 0, true, rec.p, st.sm_count, st.stream);
  launch_colstats_finalize(rec.p, stride, n, n, dmean.p, dsd.p, nullptr, nullptr, st.stream);
  launch_k_standardise(dKs.p, n, n, ld, dmean.p, dsd.p, st.stream);
  st.launches += 3;
  if (Kstd)
    GBM_CUDA(cudaMemcpy2DAsync(Kstd, n * sizeof(double), dKs.p, ld * sizeof(double), n * sizeof(double), n,
                               cudaMemcpyDefault, st.stream));
  if (pc1) {
    DevBuf<double> dZ(static_cast<size_t>(ld) * n, st.stream);
    if (ld != n) GBM_CUDA(cudaMemsetAsync(dZ.p, 0, sizeof(double) * ld * n, st.stream));
    launch_row_centre(dKs.p, dZ.p, n, ld, st.stream);
    // PC1 = the top left singular vector of Z = the eigenvector of the largest eigenvalue of B = Z Z'.  Only ONE
    // eigenvector is needed, not the decomposition: Lanczos with full reorthogonalisation (csrc/lanczos.cu) --
    //   n >= 12,000: on Z itself (two matrix-vector products per step; the n^3 SYRK for B costs more than it saves),
    //   n >= 1,024 : on B, formed by the DMMA SYRK (one matrix-vector product per step),
    // and cusolverDnDsyevdx on B below that, when Lanczos does not converge, or with GBM_PC1_SOLVER=cusolver.
    // Timed separately either way (eig_ms).
    const char* solver_env = getenv("GBM_PC1_SOLVER");
    const bool force_cusolver = solver_env && !strcmp(solver_env, "cusolver");
    const bool force_lanczos = solver_env && !strcmp(solver_env, "lanczos");
    const bool force_gram = solver_env && !strcmp(solver_env, "lanczos-gram");
    bool have_pc1 = false;
    auto run_lanczos = [&](const double* mat, int64_t ldm, bool gram) {
      DevBuf<double> dx(static_cast<size_t>(n), st.stream);
      Span eig(st.stream);
      eig.start();
      int iters = 0;
      double theta = 0.0;
      have_pc1 = lanczos_top_eigenpair(mat, n, ldm, gram, kPc1Tol, 3000, dx.p, &theta, &iters, st.sm_count, st.stream);
      eig.stop();
      if (have_pc1) {
        copy_out(pc1, dx.p, sizeof(double) * n, st.stream);
        GBM_CUDA(cudaStreamSynchronize(st.stream));
        if (eig_ms) *eig_ms = eig.ms();
        st.main_ms = eig.ms();
        st.launches += iters;
      }
    };
    // odd n: B = Z Z' has an odd pitch (128-bit loads of its columns would be misaligned), Z is padded: gram operator
    // n >= 1,024: Lanczos on Z itself (operator Z Z', never formed).  Even n up to 12,288 take the fused one-pass
    // step (a column in shared memory: its dot with v and its update of w from one read of Z), larger or odd n the
    // two-pass step; either way the n^3 SYRK for B = Z Z' is not paid.  GBM_PC1_SOLVER=lanczos keeps the older route
    // through B (one symmetric matrix-vector product per step).
    if (!force_cusolver && !force_lanczos && (n >= 1024 || force_gram)) run_lanczos(dZ.p, ld, true);
    if (have_pc1) {
      all.stop();
      GBM_CUDA(cudaStreamSynchronize(st.stream));
      st.h2d_ms = h2d.ms();
      st.kernel_ms = all.ms();
      return GBM_OK;
    }
    // B = Z Z' through the DMMA SYRK (no centring), full symmetric
    DevBuf<double> dB(static_cast<size_t>(n) * n, st.stream);
    GBM_CUDA(cudaMemsetAsync(dB.p, 0, sizeof(double) * n * n, st.stream));
    const int64_t npad = round_up(n, 16);
    DevBuf<double> dzero(npad, st.stream);
    GBM_CUDA(cudaMemsetAsync(dzero.p, 0, sizeof(double) * npad, st.stream));
    launch_grm_accumulate(dZ.p, n, n, ld, dzero.p, dB.p, st.sm_count, st.stream, false);
    launch_grm_finalize(dB.p, n, 1.0, st.stream);
    st.launches += 3;
    if (!force_cusolver && !force_gram && (n >= 1024 || force_lanczos) && (n & 1) == 0) run_lanczos(dB.p, n, false);
    if (!have_pc1) {
    // largest eigenpair of B through cuSOLVER
    if (!st.cusolver) {
      cusolverDnHandle_t h;
      if (cusolverDnCreate(&h) != CUSOLVER_STATUS_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cusolverDnCreate failed");
      st.cusolver = h;
    }
    cusolverDnHandle_t h = reinterpret_cast<cusolverDnHandle_t>(st.cusolver);
    if (cusolverDnSetStream(h, st.stream) != CUSOLVER_STATUS_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cusolverDnSetStream failed");
    if (n > 2147483647) GBM_THROW(GBM_ERR_ARGUMENT, "n too large for cuSOLVER");
    const int ni = static_cast<int>(n);
    int lwork = 0, meig = 0;
    DevBuf<double> dW(n, st.stream);
    DevBuf<int> dinfo(1, st.stream);
    if (cusolverDnDsyevdx_bufferSize(h, CUSOLVER_EIG_MODE_VECTOR, CUSOLVER_EIG_RANGE_I, CUBLAS_FILL_MODE_LOWER, ni,
                                     dB.p, ni, 0.0, 0.0, ni, ni, &meig, dW.p, &lwork) != CUSOLVER_STATUS_SUCCESS)
      GBM_THROW(GBM_ERR_CUDA, "cusolverDnDsyevdx_bufferSize failed");
    DevBuf<double> dwork(static_cast<size_t>(lwork), st.stream);
    Span eig(st.stream);
    eig.start();
    cusolverStatus_t cs = cusolverDnDsyevdx(h, CUSOLVER_EIG_MODE_VECTOR, CUSOLVER_EIG_RANGE_I, CUBLAS_FILL_MODE_LOWER,
                                            ni, dB.p, ni, 0.0, 0.0, ni, ni, &meig, dW.p, dwork.p, lwork, dinfo.p);
    eig.stop();
    if (cs != CUSOLVER_STATUS_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cusolverDnDsyevdx failed, status " + std::to_string((int)cs));
    int info = 0;
    GBM_CUDA(cudaMemcpyAsync(&info, dinfo.p, sizeof(int), cudaMemcpyDeviceToHost, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
    if (info != 0 || meig != 1) GBM_THROW(GBM_ERR_RUNTIME, "PCA of the GRM failed (syevdx info " + std::to_string(info) + ")");
    copy_out(pc1, dB.p, sizeof(double) * n, st.stream);  // first column = the eigenvector
    if (eig_ms) *eig_ms = eig.ms();
    }
  }
  all.stop();
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  st.h2d_ms = h2d.ms();
  st.kernel_ms = all.ms();
  GBM_API_END
}

// ------------------------------------------------------------------------------------
// scan
// ------------------------------------------------------------------------------------
static void check_scan_args(int64_t n, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k,
                            int64_t ldc, int model) {
  if (T < 1 || !Y) GBM_THROW(GBM_ERR_ARGUMENT, "scan: at least one trait is required");
  if (ldy < n) GBM_THROW(GBM_ERR_ARGUMENT, "scan: ldy smaller than the number of entries");
  if (k < 0 || (k > 0 && (!C || ldc < n))) GBM_THROW(GBM_ERR_ARGUMENT, "scan: bad covariate arguments");
  if (model != GBM_MODEL_OLS && model != GBM_MODEL_LMM) GBM_THROW(GBM_ERR_ARGUMENT, "scan: unknown model");
  if (n - k - 2 < 1) GBM_THROW(GBM_ERR_ARGUMENT, "scan: not enough entries for the number of covariates");
}

// Resolves the user's output pointers: device pointers are written by the kernels in place,
// host pointers get a device scratch array that is copied out afterwards.
struct OutTargets {
  struct Slot {
    void* user = nullptr;
    void* dev = nullptr;
    void* scratch = nullptr;
    size_t bytes = 0;
  };
  Slot slot[7];
  cudaStream_t s;
  explicit OutTargets(cudaStream_t stream) : s(stream) {}
  ~OutTargets() {
    for (auto& q : slot)
      if (q.scratch) cudaFreeAsync(q.scratch, s);
  }
  OutTargets(const OutTargets&) = delete;
  OutTargets& operator=(const OutTargets&) = delete;
  void bind(int i, void* user, size_t bytes) {
    Slot& q = slot[i];
    q.user = user;
    if (!user) {
      q.dev = nullptr;
      return;
    }
    if (is_device_ptr(user)) {
      q.dev = user;
      return;
    }
    if (!q.scratch || q.bytes < bytes) {
      if (q.scratch) cudaFreeAsync(q.scratch, s);
      GBM_CUDA(cudaMallocAsync(&q.scratch, bytes, s));
      q.bytes = bytes;
    }
    q.dev = q.scratch;
  }
  void bind_all(int64_t p, int64_t T, double* beta, double* se, double* stat, double* nlp, double* mean,
                double* sd, uint8_t* keep) {
    bind(0, beta, sizeof(double) * p * T);
    bind(1, se, sizeof(double) * p * T);
    bind(2, stat, sizeof(double) * p * T);
    bind(3, nlp, sizeof(double) * p * T);
    bind(4, mean, sizeof(double) * p);
    bind(5, sd, sizeof(double) * p);
    bind(6, keep, static_cast<size_t>(p));
  }
  ScanOutputs view() const {
    return ScanOutputs{static_cast<double*>(slot[0].dev), static_cast<double*>(slot[1].dev),
                       static_cast<double*>(slot[2].dev), static_cast<double*>(slot[3].dev),
                       static_cast<double*>(slot[4].dev), static_cast<double*>(slot[5].dev),
                       static_cast<uint8_t*>(slot[6].dev)};
  }
  void copy_back(int64_t p, int64_t T) {
    const size_t sz[7] = {sizeof(double) * p * T, sizeof(double) * p * T, sizeof(double) * p * T,
                          sizeof(double) * p * T, sizeof(double) * p,     sizeof(double) * p,
                          static_cast<size_t>(p)};
    for (int i = 0; i < 7; ++i)
      if (slot[i].user && slot[i].dev != slot[i].user) copy_out(slot[i].user, slot[i].dev, sz[i], s);
  }
};

}  // extern "C"  (plan type lives at global scope)

struct gbm_scan_plan {
  const gbm_matrix* m = nullptr;
  int64_t T = 0;
  int k_eff = 0, model = 0, flags = 0;
  std::vector<std::unique_ptr<gbm::Pass>> passes;
  std::vector<double*> rec;  // one record buffer per pass, kept for the plan's lifetime
  std::unique_ptr<OutTargets> out;
};

extern "C" {

int gbm_scan_plan_create(const gbm_matrix* m, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k,
                         int64_t ldc, int model, int flags, gbm_scan_plan** plan_out) {
  GBM_API_BEGIN
  require_ready();
  if (!m || !plan_out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_scan_plan_create: null pointer");
  check_scan_args(m->n, Y, T, ldy, C, k, ldc, model);
  State& st = state();
  SideVectors sv = prepare_side_vectors(Y, m->n, T, ldy, C, k, ldc);
  for (int64_t t = 0; t < T; ++t)
    if (!(sv.yMy[t] > 0.0)) GBM_THROW(GBM_ERR_ARGUMENT, "No variance in the trait after removing the covariates.");
  std::unique_ptr<gbm_scan_plan> pl(new gbm_scan_plan);
  pl->m = m;
  pl->T = T;
  pl->k_eff = sv.k_eff;
  pl->model = model;
  pl->flags = flags;
  pl->passes = build_passes(sv, m->n, T);
  for (const auto& ps : pl->passes) {
    // stream-ordered pool allocation: a plain cudaMalloc / cudaFree pair per gbm_scan call cost between
    // 20 ms and more than a second of host time at p = 1,000,000 (tools/diag_scan.py)
    double* r = nullptr;
    GBM_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&r), sizeof(double) * m->p * ps->stride, st.stream));
    pl->rec.push_back(r);
  }
  pl->out.reset(new OutTargets(st.stream));
  *plan_out = pl.release();
  GBM_API_END
}

int gbm_scan_plan_run(gbm_scan_plan* pl, double* beta, double* se, double* stat, double* neglog10p, double* mean,
                      double* sd, uint8_t* keep) {
  GBM_API_BEGIN
  require_ready();
  if (!pl) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_scan_plan_run: null plan");
  State& st = state();
  reset_timing();
  const gbm_matrix* m = pl->m;
  const int64_t p = m->p;
  pl->out->s = st.stream;
  pl->out->bind_all(p, pl->T, beta, se, stat, neglog10p, mean, sd, keep);
  Span all(st.stream), mainsp(st.stream);
  all.start();
  scan_block(*m, p, pl->passes, pl->rec, pl->k_eff, pl->model, pl->flags, pl->out->view(), p, 0, &mainsp);
  all.stop();
  Span d2h(st.stream);
  d2h.start();
  pl->out->copy_back(p, pl->T);
  d2h.stop();
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  st.kernel_ms = all.ms();
  st.main_ms = mainsp.ms();
  st.d2h_ms = d2h.ms();
  GBM_API_END
}

int gbm_scan_plan_free(gbm_scan_plan* pl) {
  GBM_API_BEGIN
  if (pl) {
    if (state().ready) {
      for (double* r : pl->rec) cudaFreeAsync(r, state().stream);
      cudaStreamSynchronize(state().stream);
    } else {
      for (double* r : pl->rec) cudaFree(r);
    }
    delete pl;
  }
  GBM_API_END
}

int gbm_scan(const gbm_matrix* m, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k, int64_t ldc,
             int model, int flags, double* beta, double* se, double* stat, double* neglog10p, double* mean,
             double* sd, uint8_t* keep) {
  gbm_scan_plan* pl = nullptr;
  int rc = gbm_scan_plan_create(m, Y, T, ldy, C, k, ldc, model, flags, &pl);
  if (rc != GBM_OK) return rc;
  rc = gbm_scan_plan_run(pl, beta, se, stat, neglog10p, mean, sd, keep);
  std::string keep_msg = rc != GBM_OK ? std::string(gbm_last_error()) : std::string();
  gbm_scan_plan_free(pl);
  if (rc != GBM_OK) set_error(keep_msg);
  return rc;
}

// ---- host-side packer entry points ----
int gbm_pack_host(const double* A, int64_t n, int64_t p, int64_t lda, uint8_t* out, int64_t ldo, int64_t* n_inexact) {
  GBM_API_BEGIN
  if (!A || !out || !n_inexact || n < 1 || p < 1 || lda < n || ldo < n)
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_pack_host: bad arguments");
  if (pack_block_host(A, n, lda, p, out, ldo, nullptr))
    *n_inexact = 0;
  else
    *n_inexact = count_inexact_host(A, n, lda, p);
  GBM_API_END
}

int gbm_pack_host_check(const double* A, int64_t n, int64_t p, int64_t lda, int isa, uint8_t* col_ok) {
  GBM_API_BEGIN
  if (!A || !col_ok || n < 1 || p < 1 || lda < n) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_pack_host_check: bad arguments");
  if (!pack_check_columns(A, n, lda, p, isa, col_ok))
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_pack_host_check: this CPU does not have the requested instruction set");
  GBM_API_END
}

int gbm_side_vector_digits(const double* Q, int64_t n, int M, int64_t ldq, int8_t* digits, int64_t ld, double* scale) {
  GBM_API_BEGIN
  if (!Q || !digits || !scale || n < 1 || M < 1 || M > 2 || ldq < n || ld != scan_u8_tc_digit_rows(n))
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_side_vector_digits: bad arguments");
  scan_u8_tc_build_digits(Q, n, M, ldq, digits, ld, scale);
  GBM_API_END
}

int gbm_tridiag_top(const double* alpha, const double* beta, int64_t m, double* theta, double* s) {
  GBM_API_BEGIN
  if (!alpha || (m > 1 && !beta) || !theta || !s || m < 1 || m > 100000)
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_tridiag_top: bad arguments");
  lanczos_tridiag_top(alpha, beta, static_cast<int>(m), theta, s);
  GBM_API_END
}

int gbm_scan_host(const double* A, int64_t n, int64_t p, int64_t lda, const double* Y, int64_t T, int64_t ldy,
                  const double* C, int64_t k, int64_t ldc, int model, int flags, double* beta, double* se,
                  double* stat, double* neglog10p, double* mean, double* sd, uint8_t* keep) {
  GBM_API_BEGIN
  require_ready();
  if (!A) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_scan_host: null matrix");
  check_dims(n, p, lda);
  check_scan_args(n, Y, T, ldy, C, k, ldc, model);
  State& st = state();
  reset_timing();
  SideVectors sv = prepare_side_vectors(Y, n, T, ldy, C, k, ldc);
  for (int64_t t = 0; t < T; ++t)
    if (!(sv.yMy[t] > 0.0)) GBM_THROW(GBM_ERR_ARGUMENT, "No variance in the trait after removing the covariates.");
  OutTargets out(st.stream);
  out.bind_all(p, T, beta, se, stat, neglog10p, mean, sd, keep);
  auto passes = build_passes(sv, n, T);
  const std::vector<double*> no_rec;
  const int kflags = flags & GBM_PVALUE_TWO_SIDED;
  const bool want_codes = (flags & GBM_SCAN_HOST_NO_PACK) == 0;  // scan blocks as 1-byte codes when they are codes
  const bool device_src = is_device_ptr(A);
  const bool pinned = device_src || is_pinned_host_ptr(A);
  // Two lanes feed the scan kernels, column blocks are handed out dynamically (results do not
  // depend on the lane: a block that is all dosage codes is scanned by the u8 kernel, any other
  // block by the Float64 kernel, wherever it was packed):
  //  * host lane: the host cores pack a block to codes (exactness-checked) into pinned staging, 1/8 of
  //    the bytes cross PCIe.  Needs >= 2 host threads; stops at the first block that is not all codes.
  //  * copy-engine lane: the block crosses PCIe as Float64 (cudaMemcpyAsync from the caller's pinned
  //    buffer) and is packed on the device.  Pageable memory would make those copies synchronous, so
  //    this lane then only takes what the host lane cannot.
  // Default: the host lane alone when this process has >= 12 host threads, else the copy-engine lane alone.
  // Measured on the pool's hosts (markers/s of the whole job, host lane / copy-engine lane): 1 GPU x 16 threads
  // 1.75 M / 0.69 M; 2 GPUs x 24 threads 1.91 M / 1.38 M; 4 GPUs x 8 threads 1.85 M / 2.67 M; 8 GPUs x 4 threads
  // 1.86 M / 2.33 M -- a packing core reads 4.6-8.8 GB/s of Float64, a GPU's link takes up to 55 GB/s.
  // Running both at once is a switch (GBM_SCAN_HOST_LANES=both): on the pool's hosts the copy engine's
  // reads slow the packing cores down by more than they add (1 GPU x 16 threads: 1.29 M markers/s together
  // against 1.71-1.76 M for the host lane alone; 8 GPUs x 4 threads: 2.28 M together, 2.33 M copy lane
  // alone), on a host with more memory bandwidth per core it pays.
  // Which lane wins depends on the host (cores and memory bandwidth per GPU, how many ranks share them), so the
  // choice is MEASURED: the first call with enough blocks runs two blocks through the host lane alone, two through
  // the copy-engine lane alone (every rank of a multi-GPU job does this at the same time, so the contention is the
  // real one) and keeps the faster for the rest of the call and for later calls of this State.  Until then, and
  // for short calls: the host lane with >= 12 host threads for this rank, else the copy-engine lane.
  const bool can_host = want_codes && !device_src && host_threads() >= 2;
  bool host_lane = want_codes && !device_src && host_threads() >= 12;
  bool raw_lane = !host_lane;
  bool forced = false;
  if (const char* e = getenv("GBM_SCAN_HOST_LANES")) {
    if (!strcmp(e, "host") && can_host) host_lane = true, raw_lane = false, forced = true;
    if (!strcmp(e, "copy")) host_lane = false, raw_lane = true, forced = true;
    if (!strcmp(e, "both") && can_host) host_lane = true, raw_lane = pinned, forced = true;
  }
  if (!forced && can_host && st.lane_choice_threads == host_threads() && st.lane_choice != 0) {
    host_lane = st.lane_choice == 1;
    raw_lane = !host_lane;
  }
  // column blocks of ~128 MB of Float64
  const int64_t ldd = round_up(n, 16);
  const int64_t ld8 = round_up(n, 128);
  int64_t blk = std::max<int64_t>(16, ((int64_t(128) << 20) / (8 * ldd)) / 16 * 16);
  blk = std::min(blk, round_up(p, 16));
  const int64_t nblk = (p + blk - 1) / blk;
  constexpr int kRaw = State::kRawSlots;
  // staging buffers and events are cached across calls
  const size_t need = sizeof(double) * ldd * blk;
  const size_t need8 = static_cast<size_t>(ld8) * blk;
  if (!st.raw_stream) GBM_CUDA(cudaStreamCreateWithFlags(&st.raw_stream, cudaStreamNonBlocking));
  auto make_event = [](cudaEvent_t* e) {
    if (!*e) GBM_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  };
  if (st.raw_bytes < need) {
    for (int b = 0; b < kRaw; ++b) {
      if (st.raw_f64[b]) cudaFree(st.raw_f64[b]);
      st.raw_f64[b] = nullptr;
      GBM_CUDA(cudaMalloc(&st.raw_f64[b], need));
    }
    st.raw_bytes = need;
  }
  if (want_codes && st.raw_code_bytes < need8) {
    for (int b = 0; b < kRaw; ++b) {
      if (st.raw_codes[b]) cudaFree(st.raw_codes[b]);
      st.raw_codes[b] = nullptr;
      GBM_CUDA(cudaMalloc(&st.raw_codes[b], need8));
    }
    st.raw_code_bytes = need8;
  }
  if (!st.raw_flag_dev) {
    GBM_CUDA(cudaMalloc(reinterpret_cast<void**>(&st.raw_flag_dev), sizeof(unsigned long long) * kRaw));
    GBM_CUDA(cudaMallocHost(reinterpret_cast<void**>(&st.raw_flag_host), sizeof(unsigned long long) * kRaw));
  }
  constexpr int kHost = State::kHostSlots;
  // the calibration below may switch the host lane on even when it does not start the call
  if ((host_lane || (can_host && !forced)) && st.code_bytes < need8) {
    for (int b = 0; b < kHost; ++b) {
      if (st.host_codes[b]) cudaFreeHost(st.host_codes[b]);
      if (st.dev_codes[b]) cudaFree(st.dev_codes[b]);
      st.host_codes[b] = st.dev_codes[b] = nullptr;
      GBM_CUDA(cudaMallocHost(&st.host_codes[b], need8));
      GBM_CUDA(cudaMalloc(&st.dev_codes[b], need8));
    }
    st.code_bytes = need8;
  }
  for (int b = 0; b < kHost; ++b) make_event(&st.hl_copied[b]), make_event(&st.hl_consumed[b]);
  for (int b = 0; b < kRaw; ++b) {
    make_event(&st.raw_copied[b]), make_event(&st.raw_packed[b]), make_event(&st.raw_consumed[b]);
    if (ldd != n) GBM_CUDA(cudaMemsetAsync(st.raw_f64[b], 0, need, st.raw_stream));  // pad rows stay zero
  }
  const bool contiguous = (lda == n && ldd == n);
  const bool stage_pageable = !pinned && host_threads() >= 2;
  const bool pinned_or_staged = pinned || stage_pageable;  // the copy-engine lane is asynchronous
  if (stage_pageable) {
    static_assert(State::kRawSlots <= State::kHostSlots, "one pinned staging block per copy-engine slot");
    if (st.up_bytes < need) {
      for (int b = 0; b < State::kHostSlots; ++b) {
        if (st.up_stage[b]) cudaFreeHost(st.up_stage[b]);
        st.up_stage[b] = nullptr;
        GBM_CUDA(cudaMallocHost(&st.up_stage[b], need));
      }
      st.up_bytes = need;
    }
    for (int b = 0; b < State::kHostSlots; ++b) make_event(&st.up_copied[b]);
  }

  int64_t next = 0;              // next unassigned block
  int64_t end_blk = nblk;        // blocks [next, end_blk) are handed out (the lane calibration runs in slices)
  std::deque<int64_t> handback;  // blocks the host lane could not pack
  int64_t code_blocks = 0, host_blocks = 0, h2d_bytes = 0;
  auto take_block = [&](bool for_raw) -> int64_t {
    if (for_raw && !handback.empty()) {
      const int64_t bi = handback.front();
      handback.pop_front();
      return bi;
    }
    return next < end_blk ? next++ : -1;
  };
  struct RawSlot {
    int state = 0;  // 0 free, 1 copy in flight, 2 device pack in flight
    int64_t bi = -1;
  } slot[kRaw];
  int raw_busy = 0;

  Span all(st.stream);
  all.start();
  for (int b = 0; b < kHost; ++b) GBM_CUDA(cudaEventRecord(st.hl_consumed[b], st.stream));
  for (int b = 0; b < kRaw; ++b) GBM_CUDA(cudaEventRecord(st.raw_consumed[b], st.stream));

  auto raw_issue = [&](int s) {
    const int64_t bi = take_block(true);
    if (bi < 0) return;
    const int64_t j0 = bi * blk, pc = std::min(blk, p - j0);
    double* dst = static_cast<double*>(st.raw_f64[s]);
    if (stage_pageable) {
      // pageable source: the host workers copy (and re-pitch) the block into pinned staging, the copy engine
      // takes it from there -- not the driver's single-threaded bounce buffer
      GBM_CUDA(cudaEventSynchronize(st.up_copied[s]));
      pack_wait(copy_submit(A + j0 * lda, n, lda, pc, static_cast<double*>(st.up_stage[s]), ldd), nullptr);
      GBM_CUDA(cudaStreamWaitEvent(st.raw_stream, st.raw_consumed[s], 0));
      GBM_CUDA(cudaMemcpyAsync(dst, st.up_stage[s], sizeof(double) * ldd * pc, cudaMemcpyHostToDevice, st.raw_stream));
      GBM_CUDA(cudaEventRecord(st.up_copied[s], st.raw_stream));
    } else if (contiguous) {
      GBM_CUDA(cudaStreamWaitEvent(st.raw_stream, st.raw_consumed[s], 0));
      GBM_CUDA(cudaMemcpyAsync(dst, A + j0 * lda, sizeof(double) * n * pc, cudaMemcpyDefault, st.raw_stream));
    } else {
      GBM_CUDA(cudaStreamWaitEvent(st.raw_stream, st.raw_consumed[s], 0));
      GBM_CUDA(cudaMemcpy2DAsync(dst, ldd * sizeof(double), A + j0 * lda, lda * sizeof(double), n * sizeof(double),
                                 pc, cudaMemcpyDefault, st.raw_stream));
    }
    GBM_CUDA(cudaEventRecord(st.raw_copied[s], st.raw_stream));
    h2d_bytes += static_cast<int64_t>(sizeof(double)) * n * pc;
    slot[s].state = 1;
    slot[s].bi = bi;
    ++raw_busy;
  };
  auto event_done = [&](cudaEvent_t e, bool wait) {
    if (wait) {
      GBM_CUDA(cudaEventSynchronize(e));
      return true;
    }
    const cudaError_t r = cudaEventQuery(e);
    if (r == cudaSuccess) return true;
    if (r != cudaErrorNotReady) GBM_CUDA(r);
    return false;
  };
  auto raw_scan = [&](int s, bool as_codes) {
    const int64_t j0 = slot[s].bi * blk, pc = std::min(blk, p - j0);
    gbm_matrix view;
    view.n = n;
    view.p = pc;
    if (as_codes) {
      view.dtype = 1;
      view.d8 = static_cast<uint8_t*>(st.raw_codes[s]);
      view.ld8 = ld8;
      ++code_blocks;
    } else {
      view.dtype = 0;
      view.d = static_cast<double*>(st.raw_f64[s]);
      view.lda = ldd;
    }
    scan_block(view, pc, passes, no_rec, sv.k_eff, model, kflags, out.view(), p, j0, nullptr);
    GBM_CUDA(cudaEventRecord(st.raw_consumed[s], st.stream));
    slot[s].state = 0;
    --raw_busy;
    raw_issue(s);
  };
  // advances the copy-engine lane; wait = block on the oldest pending event instead of polling
  auto raw_service = [&](bool wait) {
    if (!raw_lane) return;
    for (int s = 0; s < kRaw; ++s) {
      if (slot[s].state == 0) raw_issue(s);
      if (slot[s].state == 1 && event_done(st.raw_copied[s], wait)) {
        if (!want_codes) {
          raw_scan(s, false);
          continue;
        }
        const int64_t pc = std::min(blk, p - slot[s].bi * blk);
        GBM_CUDA(cudaMemsetAsync(st.raw_flag_dev + s, 0, sizeof(unsigned long long), st.stream));
        launch_pack_u8(static_cast<double*>(st.raw_f64[s]), n, pc, ldd, static_cast<uint8_t*>(st.raw_codes[s]), ld8,
                       st.raw_flag_dev + s, st.stream);
        GBM_CUDA(cudaMemcpyAsync(st.raw_flag_host + s, st.raw_flag_dev + s, sizeof(unsigned long long),
                                 cudaMemcpyDeviceToHost, st.stream));
        GBM_CUDA(cudaEventRecord(st.raw_packed[s], st.stream));
        slot[s].state = 2;
        st.launches += 1;
      }
      if (slot[s].state == 2 && event_done(st.raw_packed[s], wait)) raw_scan(s, st.raw_flag_host[s] == 0);
    }
  };
  const std::function<void()> idle = [&] { raw_service(false); };

  // host lane: up to kHost blocks are queued with the packer ahead of the one being waited for, so the
  // workers never join between blocks
  struct HostSlots {
    PackJob* job[State::kHostSlots] = {};
    int64_t bi[State::kHostSlots] = {};
    int head = 0, fill = 0, count = 0;
    ~HostSlots() {  // never leave workers writing into the staging buffers behind an exception
      for (PackJob*& j : job)
        if (j) pack_wait(j, nullptr), j = nullptr;
    }
  } hs;
  // hands out and finishes blocks [next, end) with the lanes currently switched on
  auto run_until = [&](int64_t end) {
  end_blk = end;
  raw_service(false);
  while (host_lane) {
    while (hs.count < kHost) {
      const int64_t bi = take_block(false);
      if (bi < 0) break;
      const int s = hs.fill;
      const int64_t j0 = bi * blk, pc = std::min(blk, p - j0);
      // the pinned buffer s went to the copy engine kHost host-lane blocks ago: wait for that copy
      GBM_CUDA(cudaEventSynchronize(st.hl_copied[s]));
      hs.job[s] = pack_submit(A + j0 * lda, n, lda, pc, static_cast<uint8_t*>(st.host_codes[s]), ld8);
      hs.bi[s] = bi;
      hs.fill = (s + 1) % kHost;
      ++hs.count;
    }
    if (hs.count == 0) break;
    const int s = hs.head;
    const int64_t bi = hs.bi[s];
    const int64_t j0 = bi * blk, pc = std::min(blk, p - j0);
    PackJob* job = hs.job[s];
    hs.job[s] = nullptr;
    hs.head = (s + 1) % kHost;
    --hs.count;
    if (!pack_wait(job, raw_lane ? &idle : nullptr)) {
      // not dosage data: this block, the queued ones and the rest travel as Float64
      handback.push_back(bi);
      for (; hs.count > 0; --hs.count, hs.head = (hs.head + 1) % kHost) {
        pack_wait(hs.job[hs.head], nullptr);
        hs.job[hs.head] = nullptr;
        handback.push_back(hs.bi[hs.head]);
      }
      host_lane = false;
      raw_lane = true;
      break;
    }
    GBM_CUDA(cudaStreamWaitEvent(st.copy_stream, st.hl_consumed[s], 0));
    GBM_CUDA(cudaMemcpyAsync(st.dev_codes[s], st.host_codes[s], static_cast<size_t>(ld8) * pc, cudaMemcpyHostToDevice,
                             st.copy_stream));
    GBM_CUDA(cudaEventRecord(st.hl_copied[s], st.copy_stream));
    GBM_CUDA(cudaStreamWaitEvent(st.stream, st.hl_copied[s], 0));
    gbm_matrix view;
    view.n = n;
    view.p = pc;
    view.dtype = 1;
    view.d8 = static_cast<uint8_t*>(st.dev_codes[s]);
    view.ld8 = ld8;
    scan_block(view, pc, passes, no_rec, sv.k_eff, model, kflags, out.view(), p, j0, nullptr);
    GBM_CUDA(cudaEventRecord(st.hl_consumed[s], st.stream));
    ++code_blocks;
    ++host_blocks;
    h2d_bytes += ld8 * pc;
    raw_service(false);
  }
  // drain: whatever is left goes through the copy-engine lane
  while (raw_busy > 0 || next < end_blk || !handback.empty()) {
    if (!raw_lane) GBM_THROW(GBM_ERR_RUNTIME, "gbm_scan_host: internal scheduling error");
    raw_service(true);
  }
  };
  const bool calibrate = !forced && can_host && pinned_or_staged && nblk >= 12 &&
                         !(st.lane_choice_threads == host_threads() && st.lane_choice != 0);
  if (calibrate) {
    auto drain_all = [&] {
      GBM_CUDA(cudaStreamSynchronize(st.stream));
      GBM_CUDA(cudaStreamSynchronize(st.copy_stream));
      GBM_CUDA(cudaStreamSynchronize(st.raw_stream));
    };
    host_lane = true, raw_lane = false;
    auto t0 = std::chrono::steady_clock::now();
    run_until(3);
    drain_all();
    const double t_host = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    const bool still_codes = host_lane;  // the host lane switches itself off at the first block that is not all codes
    host_lane = false, raw_lane = true;
    t0 = std::chrono::steady_clock::now();
    run_until(std::min<int64_t>(next + 3, nblk));
    drain_all();
    const double t_copy = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (still_codes) {  // dosage data: remember the faster lane; other data always travels as Float64
      st.lane_choice = t_host <= t_copy ? 1 : 2;
      st.lane_choice_threads = host_threads();
      host_lane = st.lane_choice == 1;
      raw_lane = !host_lane;
    }
    run_until(nblk);
  } else {
    run_until(nblk);
  }
  all.stop();
  out.copy_back(p, T);
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  GBM_CUDA(cudaStreamSynchronize(st.copy_stream));
  GBM_CUDA(cudaStreamSynchronize(st.raw_stream));
  st.kernel_ms = all.ms();  // copy + compute overlapped: wall time of the pipeline on the device
  st.packed_blocks = code_blocks;
  st.host_packed_blocks = host_blocks;
  st.h2d_bytes = device_src ? 0 : h2d_bytes;
  GBM_API_END
}

}  // extern "C"

// ------------------------------------------------------------------------------------
// GRM-covariance LMM scan (rotation + per-marker delta search)
// ------------------------------------------------------------------------------------
namespace gbm {

gbm_lmm_plan* lmm_plan_alloc(int64_t n, int Q0) {
  std::unique_ptr<gbm_lmm_plan> pl(new gbm_lmm_plan);
  pl->n = n;
  pl->ldu = round_up(n, 16);
  pl->Q0 = Q0;
  auto dalloc = [&](double** p, size_t count) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), sizeof(double) * count);
    if (e != cudaSuccess) {
      lmm_plan_destroy(pl.release());
      GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
    }
  };
  dalloc(&pl->dU, static_cast<size_t>(pl->ldu) * n);
  dalloc(&pl->dS, n);
  dalloc(&pl->dYr, n);
  dalloc(&pl->dCr, static_cast<size_t>(n) * Q0);
  return pl.release();
}

void lmm_plan_destroy(gbm_lmm_plan* pl) {
  if (!pl) return;
  cudaFree(pl->dU);
  cudaFree(pl->dS);
  cudaFree(pl->dYr);
  cudaFree(pl->dCr);
  delete pl;
}

void lmm_plan_load_k(gbm_lmm_plan* pl, const double* K, int64_t ldk) {
  State& st = state();
  const int64_t n = pl->n;
  if (pl->ldu != n) GBM_CUDA(cudaMemsetAsync(pl->dU, 0, sizeof(double) * pl->ldu * n, st.stream));
  GBM_CUDA(cudaMemcpy2DAsync(pl->dU, pl->ldu * sizeof(double), K, ldk * sizeof(double), n * sizeof(double), n,
                             cudaMemcpyDefault, st.stream));
}

void lmm_plan_factor(gbm_lmm_plan* pl, const double* y, const double* C, int64_t k, int64_t ldc, double* eig_ms) {
  State& st = state();
  const int64_t n = pl->n;
  const int Q0 = pl->Q0;
  // K = U S U' through cuSOLVER (lower triangle), timed separately
  if (!st.cusolver) {
    cusolverDnHandle_t h;
    if (cusolverDnCreate(&h) != CUSOLVER_STATUS_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cusolverDnCreate failed");
    st.cusolver = h;
  }
  cusolverDnHandle_t h = reinterpret_cast<cusolverDnHandle_t>(st.cusolver);
  if (cusolverDnSetStream(h, st.stream) != CUSOLVER_STATUS_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cusolverDnSetStream failed");
  const int ni = static_cast<int>(n), ldi = static_cast<int>(pl->ldu);
  int lwork = 0;
  if (cusolverDnDsyevd_bufferSize(h, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_LOWER, ni, pl->dU, ldi, pl->dS,
                                  &lwork) != CUSOLVER_STATUS_SUCCESS)
    GBM_THROW(GBM_ERR_CUDA, "cusolverDnDsyevd_bufferSize failed");
  {
    DevBuf<double> dwork(static_cast<size_t>(lwork), st.stream);
    DevBuf<int> dinfo(1, st.stream);
    Span eig(st.stream);
    eig.start();
    cusolverStatus_t cs = cusolverDnDsyevd(h, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_LOWER, ni, pl->dU, ldi,
                                           pl->dS, dwork.p, lwork, dinfo.p);
    eig.stop();
    if (cs != CUSOLVER_STATUS_SUCCESS) GBM_THROW(GBM_ERR_CUDA, "cusolverDnDsyevd failed, status " + std::to_string((int)cs));
    int info = 0;
    GBM_CUDA(cudaMemcpyAsync(&info, dinfo.p, sizeof(int), cudaMemcpyDeviceToHost, st.stream));
    GBM_CUDA(cudaStreamSynchronize(st.stream));
    if (info != 0) GBM_THROW(GBM_ERR_RUNTIME, "eigendecomposition of the GRM failed (syevd info " + std::to_string(info) + ")");
    if (eig_ms) *eig_ms = eig.ms();
  }
  // rotate [1, C, y] with the DMMA GEMM
  const int64_t ldb = round_up(n, 16);
  std::vector<double> hB(static_cast<size_t>(ldb) * (Q0 + 1), 0.0);
  for (int64_t i = 0; i < n; ++i) hB[i] = 1.0;
  if (k > 0)
    GBM_CUDA(cudaMemcpy2D(hB.data() + ldb, ldb * sizeof(double), C, ldc * sizeof(double), n * sizeof(double), k,
                          cudaMemcpyDefault));
  GBM_CUDA(cudaMemcpy(hB.data() + static_cast<size_t>(ldb) * Q0, y, n * sizeof(double), cudaMemcpyDefault));
  {
    DevBuf<double> dB(hB.size(), st.stream), dOut(static_cast<size_t>(n) * (Q0 + 1), st.stream);
    GBM_CUDA(cudaMemcpyAsync(dB.p, hB.data(), sizeof(double) * hB.size(), cudaMemcpyHostToDevice, st.stream));
    launch_gemm_tn(pl->dU, pl->ldu, dB.p, ldb, dOut.p, n, n, Q0 + 1, n, st.sm_count, st.stream);
    GBM_CUDA(cudaMemcpyAsync(pl->dCr, dOut.p, sizeof(double) * n * Q0, cudaMemcpyDeviceToDevice, st.stream));
    GBM_CUDA(cudaMemcpyAsync(pl->dYr, dOut.p + static_cast<size_t>(n) * Q0, sizeof(double) * n,
                             cudaMemcpyDeviceToDevice, st.stream));
    st.launches++;
    GBM_CUDA(cudaStreamSynchronize(st.stream));
  }
  // null model on the host (n-vector work)
  std::vector<double> hS(n), hY(n), hC(static_cast<size_t>(n) * Q0);
  GBM_CUDA(cudaMemcpy(hS.data(), pl->dS, sizeof(double) * n, cudaMemcpyDeviceToHost));
  GBM_CUDA(cudaMemcpy(hY.data(), pl->dYr, sizeof(double) * n, cudaMemcpyDeviceToHost));
  GBM_CUDA(cudaMemcpy(hC.data(), pl->dCr, sizeof(double) * n * Q0, cudaMemcpyDeviceToHost));
  pl->s_min = hS[0];
  pl->lam0 = lmm_null_lam0(Q0, hS.data(), hC.data(), n, hY.data(), n);
}

}  // namespace gbm

extern "C" {

int gbm_lmm_plan_create(const double* K, int64_t n, const double* y, const double* C, int64_t k, int64_t ldc,
                        gbm_lmm_plan** plan_out, double* eig_ms, double* null_log_delta) {
  GBM_API_BEGIN
  require_ready();
  if (!K || !y || !plan_out || n < 4) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_lmm_plan_create: bad arguments");
  if (k < 0 || k > 2 || (k > 0 && (!C || ldc < n)))
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_lmm_plan_create: 0..2 covariates besides the intercept are supported");
  if (n > 2147483647) GBM_THROW(GBM_ERR_ARGUMENT, "n too large for cuSOLVER");
  reset_timing();
  std::unique_ptr<gbm_lmm_plan, void (*)(gbm_lmm_plan*)> pl(lmm_plan_alloc(n, static_cast<int>(k) + 1), lmm_plan_destroy);
  lmm_plan_load_k(pl.get(), K, n);
  lmm_plan_factor(pl.get(), y, C, k, ldc, eig_ms);
  if (null_log_delta) *null_log_delta = pl->lam0;
  *plan_out = pl.release();
  GBM_API_END
}

int gbm_lmm_plan_run(gbm_lmm_plan* pl, const gbm_matrix* m, int flags, double* beta, double* se, double* stat,
                     double* neglog10p, double* log_delta, double* gemm_tflops, double* search_ms) {
  GBM_API_BEGIN
  require_ready();
  if (!pl || !m) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_lmm_plan_run: null pointer");
  if (m->n != pl->n) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_lmm_plan_run: the matrix and the GRM have different numbers of entries");
  State& st = state();
  reset_timing();
  const int64_t n = pl->n, p = m->p;
  const bool ref_obj = (flags & GBM_LMM_REFERENCE_OBJECTIVE) != 0;
  // fixed-locus filter + column sd (beta / se are reported for the standardised column)
  const int stride = scan_record_stride(0, true);
  DevBuf<double> rec(static_cast<size_t>(p) * stride, st.stream), dsd(p, st.stream);
  DevBuf<uint8_t> dkeep(p, st.stream);
  scan_sums_any(m, 0, p, nullptr, 0, 0, rec.p);
  launch_colstats_finalize(rec.p, stride, n, p, nullptr, dsd.p, nullptr, dkeep.p, st.stream);
  st.launches += 2;
  OutTargets out(st.stream);
  out.bind(0, beta, sizeof(double) * p);
  out.bind(1, se, sizeof(double) * p);
  out.bind(2, stat, sizeof(double) * p);
  out.bind(3, neglog10p, sizeof(double) * p);
  out.bind(4, log_delta, sizeof(double) * p);
  const int64_t ldr = round_up(n, 16);
  int64_t PB = std::max<int64_t>(128, ((int64_t(1) << 30) / (8 * ldr)) / 128 * 128);
  PB = std::min<int64_t>(PB, round_up(p, 128));
  DevBuf<double> dAr(static_cast<size_t>(ldr) * PB, st.stream);
  DevBuf<double> dDec(m->dtype == 1 ? static_cast<size_t>(ldr) * PB : 0, st.stream);
  double gemm_total = 0.0, search_total = 0.0;
  std::vector<std::unique_ptr<Span>> gs, ss;
  for (int64_t j0 = 0; j0 < p; j0 += PB) {
    const int64_t pb = std::min(PB, p - j0);
    gs.emplace_back(new Span(st.stream));
    gs.back()->start();
    if (m->dtype == 0) {
      launch_gemm_tn(pl->dU, pl->ldu, m->d + j0 * m->lda, m->lda, dAr.p, ldr, n, pb, n, st.sm_count, st.stream);
    } else {
      launch_decode_u8(m->d8 + j0 * m->ld8, n, pb, m->ld8, dDec.p, ldr, st.stream);
      launch_gemm_tn(pl->dU, pl->ldu, dDec.p, ldr, dAr.p, ldr, n, pb, n, st.sm_count, st.stream);
    }
    gs.back()->stop();
    ss.emplace_back(new Span(st.stream));
    ss.back()->start();
    auto off = [&](int i) { return out.slot[i].dev ? static_cast<double*>(out.slot[i].dev) + j0 : nullptr; };
    // reference objective: the search starts at s2e / s2u = 1, the reference's theta_init = [0.5, 0.5] (gwas.jl:578)
    launch_lmm_delta(pl->Q0, dAr.p, n, pb, ldr, pl->dS, pl->dYr, pl->dCr, n, ref_obj ? 0.0 : pl->lam0, dsd.p + j0,
                     dkeep.p + j0, off(0), off(1), off(2), off(3), off(4), flags & GBM_PVALUE_TWO_SIDED, st.sm_count,
                     st.stream, ref_obj ? 1 : 0, pl->s_min);
    ss.back()->stop();
    st.launches += 2;
  }
  const size_t sz = sizeof(double) * p;
  for (int i = 0; i < 5; ++i)
    if (out.slot[i].user && out.slot[i].dev != out.slot[i].user) copy_out(out.slot[i].user, out.slot[i].dev, sz, st.stream);
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  for (auto& s : gs) gemm_total += s->ms();
  for (auto& s : ss) search_total += s->ms();
  st.main_ms = gemm_total;
  st.kernel_ms = gemm_total + search_total;
  if (gemm_tflops) *gemm_tflops = 2.0 * n * n * static_cast<double>(p) / (gemm_total * 1e-3) / 1e12;
  if (search_ms) *search_ms = search_total;
  GBM_API_END
}

int gbm_lmm_plan_free(gbm_lmm_plan* pl) {
  GBM_API_BEGIN
  if (pl) {
    if (state().ready) cudaStreamSynchronize(state().stream);
    lmm_plan_destroy(pl);
  }
  GBM_API_END
}

/* plain C = A'B on the DMMA GEMM (device pointers), exposed for tests and for rotating extra vectors */
int gbm_gemm_tn(const double* dA, int64_t lda, const double* dB, int64_t ldb, double* dC, int64_t ldc, int64_t M,
                int64_t N, int64_t K, double* tflops) {
  GBM_API_BEGIN
  require_ready();
  if (!dA || !dB || !dC || M < 1 || N < 1 || K < 1 || lda < K || ldb < K || ldc < M)
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_gemm_tn: bad arguments");
  if (!is_device_ptr(dA) || !is_device_ptr(dB) || !is_device_ptr(dC))
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_gemm_tn: device pointers required");
  State& st = state();
  Span sp(st.stream);
  sp.start();
  launch_gemm_tn(dA, lda, dB, ldb, dC, ldc, M, N, K, st.sm_count, st.stream);
  sp.stop();
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  if (tflops) *tflops = 2.0 * M * static_cast<double>(N) * K / (sp.ms() * 1e-3) / 1e12;
  GBM_API_END
}

int gbm_neglog10_sf(const double* stat, int64_t len, int dist, double df, double* out) {
  GBM_API_BEGIN
  require_ready();
  if (!stat || !out || len < 0) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_neglog10_sf: bad arguments");
  if (dist != 0 && dist != 1) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_neglog10_sf: dist must be 0 (t) or 1 (normal)");
  if (dist == 0 && !(df > 0)) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_neglog10_sf: df must be positive");
  State& st = state();
  DevBuf<double> din(len, st.stream), dout(len, st.stream);
  GBM_CUDA(cudaMemcpyAsync(din.p, stat, sizeof(double) * len, cudaMemcpyDefault, st.stream));
  launch_neglog10_sf(din.p, len, dist, df, dout.p, st.stream);
  copy_out(out, dout.p, sizeof(double) * len, st.stream);
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  GBM_API_END
}

int gbm_measure_copy_bandwidth(int64_t bytes, int reps, double* gbps) {
  GBM_API_BEGIN
  require_ready();
  if (bytes < 1024 || reps < 1 || !gbps) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_measure_copy_bandwidth: bad arguments");
  State& st = state();
  DevBuf<uint8_t> a(bytes, st.stream), b(bytes, st.stream);
  GBM_CUDA(cudaMemsetAsync(a.p, 1, bytes, st.stream));
  GBM_CUDA(cudaMemcpyAsync(b.p, a.p, bytes, cudaMemcpyDeviceToDevice, st.stream));
  double best = 0.0;
  for (int r = 0; r < reps; ++r) {
    Span sp(st.stream);
    sp.start();
    GBM_CUDA(cudaMemcpyAsync(b.p, a.p, bytes, cudaMemcpyDeviceToDevice, st.stream));
    sp.stop();
    const double ms = sp.ms();
    best = std::max(best, 2.0 * static_cast<double>(bytes) / (ms * 1e-3) / 1e9);
  }
  *gbps = best;
  GBM_API_END
}

}  // extern "C"

// ------------------------------------------------------------------------------------
// transformation screens (transform1 / transform2 of transformation.jl)
// ------------------------------------------------------------------------------------
namespace {

// Float64 view of a handle: the slab itself, or a decoded copy of a packed one
struct F64View {
  const double* d = nullptr;
  int64_t lda = 0;
  std::unique_ptr<DevBuf<double>> tmp;
  F64View(const gbm_matrix* m, cudaStream_t s) {
    if (m->dtype == 0) {
      d = m->d;
      lda = m->lda;
    } else {
      lda = round_up(m->n, 16);
      tmp.reset(new DevBuf<double>(static_cast<size_t>(lda) * m->p, s));
      launch_decode_u8(m->d8, m->n, m->p, m->ld8, tmp->p, lda, s);
      d = tmp->p;
    }
    if ((lda & 1) != 0 || (reinterpret_cast<uintptr_t>(d) & 15u) != 0)
      GBM_THROW(GBM_ERR_ARGUMENT, "device matrix must be 16-byte aligned with an even leading dimension");
  }
};

// y -> (ybar, device copy of y - ybar)
struct CentredTrait {
  double ybar = 0.0;
  DevBuf<double> dyc;
  CentredTrait(const double* y, int64_t n, cudaStream_t s) : dyc(static_cast<size_t>(round_up(n, 2)), s) {
    std::vector<double> h(static_cast<size_t>(round_up(n, 2)), 0.0);
    GBM_CUDA(cudaMemcpy(h.data(), y, sizeof(double) * n, cudaMemcpyDefault));
    long double sum = 0;
    for (int64_t i = 0; i < n; ++i) sum += h[i];
    ybar = static_cast<double>(sum / n);
    for (int64_t i = 0; i < n; ++i) h[i] -= ybar;
    GBM_CUDA(cudaMemcpyAsync(dyc.p, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, s));
    GBM_CUDA(cudaStreamSynchronize(s));
  }
};

void check_transform_args(const gbm_matrix* m, const double* y, int64_t n_new, const void* idx, const int64_t* count) {
  if (!m || !y || !idx || !count) GBM_THROW(GBM_ERR_ARGUMENT, "transform screen: null pointer");
  if (m->n < 2) GBM_THROW(GBM_ERR_ARGUMENT, "transform screen: at least 2 entries are needed");
  if (n_new < 0) GBM_THROW(GBM_ERR_ARGUMENT, "transform screen: n_new_features_per_transformation must not be negative");
}

const char* kCannotTransform =
    "Cannot transform the allele frequencies using this function (NaN effects). Please consider adding a larger "
    "`\xcf\xb5` and/or using absolute values, i.e. use `use_abs=true`.";

}  // namespace

extern "C" {

int gbm_transform1_screen(const gbm_matrix* m, const double* y, int f, double eps, int use_abs, double var_threshold,
                          int64_t n_new, double* beta, int64_t* idx, int64_t* count) {
  GBM_API_BEGIN
  require_ready();
  check_transform_args(m, y, n_new, idx, count);
  if (f < GBM_F1_SQUARE || f > GBM_F1_LOG10EPS) GBM_THROW(GBM_ERR_ARGUMENT, "transform1: unknown transformation code");
  if (n_new > m->p)  // sortperm(...)[1:n_new] on a shorter vector (transformation.jl:212)
    GBM_THROW(GBM_ERR_ARGUMENT, "BoundsError: attempt to access " + std::to_string(m->p) + "-element Vector{Int64} at index [1:" +
                                    std::to_string(n_new) + "]");
  State& st = state();
  reset_timing();
  F64View A(m, st.stream);
  CentredTrait yt(y, m->n, st.stream);
  DevBuf<double> dbeta(static_cast<size_t>(m->p), st.stream);
  Span mainsp(st.stream);
  mainsp.start();
  launch_transform1_scan(f, A.d, m->n, m->p, A.lda, yt.dyc.p, yt.ybar, eps, use_abs, var_threshold, dbeta.p, nullptr,
                         st.sm_count, st.stream);
  mainsp.stop();
  bool has_nan = false;
  *count = transform_select(dbeta.p, m->p, n_new, eps, idx, nullptr, &has_nan, st.sm_count, st.stream);
  if (beta) copy_out(beta, dbeta.p, sizeof(double) * m->p, st.stream);
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  st.main_ms = st.kernel_ms = mainsp.ms();
  st.launches = 1;
  if (has_nan) GBM_THROW(GBM_ERR_ARGUMENT, kCannotTransform);
  GBM_API_END
}

// rows [row0, row1) of the pair matrix; sel / val in selection order (descending |beta|, ties by position), positions
// are global one-based counters
static int64_t transform2_rows(const gbm_matrix* m, const double* y, int f, double eps, int use_abs,
                               double var_threshold, int commutative, int64_t row0, int64_t row1, int64_t n_new,
                               double* beta, std::vector<int64_t>* sel, std::vector<double>* val, bool* has_nan) {
  State& st = state();
  reset_timing();
  const int64_t l = m->p, rows = row1 - row0;
  F64View A(m, st.stream);
  CentredTrait yt(y, m->n, st.stream);
  DevBuf<double> dvar(static_cast<size_t>(l), st.stream);
  // beta on the device: the caller's buffer when it is device memory, else scratch
  const bool user_dev = beta && is_device_ptr(beta);
  DevBuf<double> dscratch(user_dev ? 0 : static_cast<size_t>(rows) * l, st.stream);
  double* dbeta = user_dev ? beta : dscratch.p;
  GBM_CUDA(cudaMemsetAsync(dbeta, 0, sizeof(double) * rows * l, st.stream));
  launch_transform1_scan(-1, A.d, m->n, l, A.lda, yt.dyc.p, yt.ybar, eps, use_abs, var_threshold, nullptr, dvar.p,
                         st.sm_count, st.stream);
  Span mainsp(st.stream);
  mainsp.start();
  launch_transform2_scan(f, A.d, m->n, l, A.lda, yt.dyc.p, yt.ybar, dvar.p, eps, use_abs, var_threshold, commutative,
                         row0, row1, dbeta, st.stream);
  mainsp.stop();
  const int64_t take = std::min<int64_t>(n_new, rows * l);
  sel->assign(static_cast<size_t>(std::max<int64_t>(take, 1)), 0);
  val->assign(sel->size(), 0.0);
  const int64_t cnt = transform_select(dbeta, rows * l, take, eps, sel->data(), val->data(), has_nan, st.sm_count, st.stream);
  for (int64_t k = 0; k < cnt; ++k) (*sel)[k] += row0 * l;  // slab position -> global counter
  if (beta && !user_dev) copy_out(beta, dbeta, sizeof(double) * rows * l, st.stream);
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  st.main_ms = st.kernel_ms = mainsp.ms();
  st.launches = 2;
  return cnt;
}

int gbm_transform2_screen(const gbm_matrix* m, const double* y, int f, double eps, int use_abs, double var_threshold,
                          int commutative, int64_t n_new, double* beta, int64_t* counters, double* beta_sel,
                          int64_t* count) {
  GBM_API_BEGIN
  require_ready();
  check_transform_args(m, y, n_new, counters, count);
  if (f < GBM_F2_MULT || f > GBM_F2_RAISE) GBM_THROW(GBM_ERR_ARGUMENT, "transform2: unknown transformation code");
  const int64_t l = m->p;
  if (l > 3000000) GBM_THROW(GBM_ERR_ARGUMENT, "transform2: l^2 effects do not fit");
  if (n_new > l * l)
    GBM_THROW(GBM_ERR_ARGUMENT, "BoundsError: attempt to access " + std::to_string(l * l) + "-element Vector{Int64} at index [1:" +
                                    std::to_string(n_new) + "]");
  bool has_nan = false;
  std::vector<int64_t> sel;
  std::vector<double> val;
  const int64_t cnt = transform2_rows(m, y, f, eps, use_abs, var_threshold, commutative, 0, l, n_new, beta, &sel, &val, &has_nan);
  // sort!(idx) (transformation.jl:430): ascending positions, values follow
  std::vector<int64_t> order(static_cast<size_t>(cnt));
  for (int64_t k = 0; k < cnt; ++k) order[k] = k;
  std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return sel[a] < sel[b]; });
  for (int64_t k = 0; k < cnt; ++k) {
    counters[k] = sel[order[k]];
    if (beta_sel) beta_sel[k] = val[order[k]];
  }
  *count = cnt;
  if (has_nan) GBM_THROW(GBM_ERR_ARGUMENT, kCannotTransform);
  GBM_API_END
}

int gbm_transform2_screen_rows(const gbm_matrix* m, const double* y, int f, double eps, int use_abs,
                               double var_threshold, int commutative, int64_t row0, int64_t row1, int64_t n_new,
                               double* beta_slab, int64_t* counters, double* beta_sel, int64_t* count) {
  GBM_API_BEGIN
  require_ready();
  check_transform_args(m, y, n_new, counters, count);
  if (f < GBM_F2_MULT || f > GBM_F2_RAISE) GBM_THROW(GBM_ERR_ARGUMENT, "transform2: unknown transformation code");
  const int64_t l = m->p;
  if (l > 3000000) GBM_THROW(GBM_ERR_ARGUMENT, "transform2: l^2 effects do not fit");
  if (row0 < 0 || row1 > l || row0 >= row1) GBM_THROW(GBM_ERR_ARGUMENT, "transform2: row range out of bounds");
  bool has_nan = false;
  std::vector<int64_t> sel;
  std::vector<double> val;
  const int64_t cnt = transform2_rows(m, y, f, eps, use_abs, var_threshold, commutative, row0, row1, n_new, beta_slab, &sel,
                                      &val, &has_nan);
  for (int64_t k = 0; k < cnt; ++k) {  // selection order: descending |beta|, ties by ascending position
    counters[k] = sel[k];
    if (beta_sel) beta_sel[k] = val[k];
  }
  *count = cnt;
  if (has_nan) GBM_THROW(GBM_ERR_ARGUMENT, kCannotTransform);
  GBM_API_END
}

static void check_apply_args(const gbm_matrix* m, const int64_t* idx, int64_t count, const double* T, int64_t ldt) {
  if (!m || count < 0 || (count > 0 && (!idx || !T)) || ldt < (m ? m->n : 0))
    GBM_THROW(GBM_ERR_ARGUMENT, "transform apply: bad arguments");
}

// copies a 1-based index list to the device after range-checking it against [1, hi]
static void upload_indices(const int64_t* idx, int64_t count, int64_t hi, int64_t* dst, cudaStream_t s) {
  std::vector<int64_t> h(static_cast<size_t>(count));
  GBM_CUDA(cudaMemcpy(h.data(), idx, sizeof(int64_t) * count, cudaMemcpyDefault));
  for (int64_t v : h)
    if (v < 1 || v > hi) GBM_THROW(GBM_ERR_ARGUMENT, "transform apply: feature index out of bounds");
  GBM_CUDA(cudaMemcpyAsync(dst, h.data(), sizeof(int64_t) * count, cudaMemcpyHostToDevice, s));
  GBM_CUDA(cudaStreamSynchronize(s));
}

int gbm_transform1_apply(const gbm_matrix* m, int f, double eps, int use_abs, const int64_t* idx, int64_t count,
                         double* T, int64_t ldt) {
  GBM_API_BEGIN
  require_ready();
  check_apply_args(m, idx, count, T, ldt);
  if (f < GBM_F1_SQUARE || f > GBM_F1_LOG10EPS) GBM_THROW(GBM_ERR_ARGUMENT, "transform1: unknown transformation code");
  if (count == 0) return GBM_OK;
  State& st = state();
  F64View A(m, st.stream);
  DevBuf<int64_t> didx(static_cast<size_t>(count), st.stream);
  upload_indices(idx, count, m->p, didx.p, st.stream);
  const bool user_dev = is_device_ptr(T);
  DevBuf<double> dscratch(user_dev ? 0 : static_cast<size_t>(m->n) * count, st.stream);
  double* dT = user_dev ? T : dscratch.p;
  const int64_t ld = user_dev ? ldt : m->n;
  launch_transform1_apply(f, A.d, m->n, A.lda, didx.p, count, eps, use_abs, dT, ld, st.stream);
  if (!user_dev)
    GBM_CUDA(cudaMemcpy2DAsync(T, ldt * sizeof(double), dT, ld * sizeof(double), m->n * sizeof(double), count,
                               cudaMemcpyDeviceToHost, st.stream));
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  GBM_API_END
}

int gbm_transform2_apply(const gbm_matrix* m, int f, double eps, int use_abs, const int64_t* counters, int64_t count,
                         double* T, int64_t ldt) {
  GBM_API_BEGIN
  require_ready();
  check_apply_args(m, counters, count, T, ldt);
  if (f < GBM_F2_MULT || f > GBM_F2_RAISE) GBM_THROW(GBM_ERR_ARGUMENT, "transform2: unknown transformation code");
  if (count == 0) return GBM_OK;
  State& st = state();
  F64View A(m, st.stream);
  DevBuf<int64_t> didx(static_cast<size_t>(count), st.stream);
  upload_indices(counters, count, m->p * m->p, didx.p, st.stream);
  const bool user_dev = is_device_ptr(T);
  DevBuf<double> dscratch(user_dev ? 0 : static_cast<size_t>(m->n) * count, st.stream);
  double* dT = user_dev ? T : dscratch.p;
  const int64_t ld = user_dev ? ldt : m->n;
  launch_transform2_apply(f, A.d, m->n, m->p, A.lda, didx.p, count, eps, use_abs, dT, ld, st.stream);
  if (!user_dev)
    GBM_CUDA(cudaMemcpy2DAsync(T, ldt * sizeof(double), dT, ld * sizeof(double), m->n * sizeof(double), count,
                               cudaMemcpyDeviceToHost, st.stream));
  GBM_CUDA(cudaStreamSynchronize(st.stream));
  GBM_API_END
}

}  // extern "C"
