// Element-wise kernels around the PC1 step of gwasols / gwaslmm:
//   K = (K .- mean(K, dims=1)) ./ std(K, dims=1)                    /root/reference/src/gwas.jl:130
//   MultivariateStats.fit(PCA, K; maxoutdim=1): centre the rows     /root/reference/src/gwas.jl:234, :357
// the symmetric part of the standardised K (gwasreml's reference objective), and the gather behind `allele_frequencies[idx_entries[idx], idx_loci_alleles]`
// (/root/reference/src/prediction.jl:129).  HBM-bound streaming kernels, 128-bit accesses
// where the layout allows it.
#include "common.cuh"
#include "kernels.h"

namespace gbm {

// One CTA column-slab: grid.y = column, threads stride down the rows (coalesced).
__global__ void __launch_bounds__(256)
    k_standardise_kernel(double* __restrict__ K, int64_t n, int64_t ld, const double* __restrict__ colmean,
                         const double* __restrict__ colsd) {
  const int64_t j = blockIdx.y;
  const double mu = colmean[j], sd = colsd[j];
  double* col = K + j * ld;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    col[i] = (col[i] - mu) / sd;  // a true division, as the reference's ./
}

void launch_k_standardise(double* K, int64_t n, int64_t ncols, int64_t ld, const double* colmean, const double* colsd,
                          cudaStream_t stream) {
  if (n <= 0 || ncols <= 0) return;
  unsigned gx = static_cast<unsigned>((n + 255) / 256);
  if (gx > 8) gx = 8;
  for (int64_t j0 = 0; j0 < ncols; j0 += 65535) {
    const unsigned gy = static_cast<unsigned>(ncols - j0 < 65535 ? ncols - j0 : 65535);
    k_standardise_kernel<<<dim3(gx, gy), 256, 0, stream>>>(K + j0 * ld, n, ld, colmean + j0, colsd + j0);
  }
  GBM_CUDA(cudaGetLastError());
}

// Row means of an n x n column-major matrix, then Z = Ks - rowmean.  Thread i owns row i
// and walks the columns, so each warp reads 256 contiguous bytes per column; the sum over
// columns is sequential per row (deterministic).
__global__ void __launch_bounds__(128)
    row_centre_kernel(const double* __restrict__ Ks, double* __restrict__ Z, int64_t n, int64_t ld) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int64_t j = 0;
  for (; j + 3 < n; j += 4) {
    s0 += Ks[j * ld + i];
    s1 += Ks[(j + 1) * ld + i];
    s2 += Ks[(j + 2) * ld + i];
    s3 += Ks[(j + 3) * ld + i];
  }
  for (; j < n; ++j) s0 += Ks[j * ld + i];
  const double m = ((s0 + s1) + (s2 + s3)) / static_cast<double>(n);
  for (j = 0; j < n; ++j) Z[j * ld + i] = Ks[j * ld + i] - m;
}

void launch_row_centre(const double* Ks, double* Z, int64_t n, int64_t ld, cudaStream_t stream) {
  if (n <= 0) return;
  row_centre_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, stream>>>(Ks, Z, n, ld);
  GBM_CUDA(cudaGetLastError());
}

// K <- (K + K') / 2 in place: the symmetric part of the column-standardised GRM, the matrix the eigen-rotation of
// gwasreml's reference objective factors.  One CTA per 32 x 32 tile pair (I, J), I >= J, both tiles through shared
// memory before any store (the diagonal tile is its own partner); both entries get 0.5 * (a + b), the same bits in
// either order.
__global__ void __launch_bounds__(256) symmetrise_kernel(double* __restrict__ K, int64_t n, int64_t ld) {
  __shared__ double a[32][33], b[32][33];
  const int bi = blockIdx.x, bj = blockIdx.y;
  if (bj > bi) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const int64_t r0 = static_cast<int64_t>(bi) * 32, c0 = static_cast<int64_t>(bj) * 32;
  for (int r = ty; r < 32; r += 8) {
    a[r][tx] = (r0 + tx < n && c0 + r < n) ? K[(c0 + r) * ld + r0 + tx] : 0.0;  // tile (I, J): K[r0 + tx, c0 + r]
    b[r][tx] = (c0 + tx < n && r0 + r < n) ? K[(r0 + r) * ld + c0 + tx] : 0.0;  // tile (J, I): K[c0 + tx, r0 + r]
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    if (r0 + tx < n && c0 + r < n) K[(c0 + r) * ld + r0 + tx] = 0.5 * (a[r][tx] + b[tx][r]);
    if (c0 + tx < n && r0 + r < n) K[(r0 + r) * ld + c0 + tx] = 0.5 * (b[r][tx] + a[tx][r]);
  }
}

void launch_symmetrise(double* K, int64_t n, int64_t ld, cudaStream_t stream) {
  if (n <= 0) return;
  const unsigned nb = static_cast<unsigned>((n + 31) / 32);
  symmetrise_kernel<<<dim3(nb, nb), 256, 0, stream>>>(K, n, ld);
  GBM_CUDA(cudaGetLastError());
}

// Z[i, j] -= rowmean[i] on an n x ncols column block (the row-centring step when the columns of Kstd are
// sharded over GPUs: the row sums are all-reduced first)
__global__ void __launch_bounds__(256)
    row_shift_kernel(double* __restrict__ Z, int64_t n, int64_t ld, const double* __restrict__ rowsum, double inv_cols) {
  const int64_t j = blockIdx.y;
  double* col = Z + j * ld;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    col[i] -= rowsum[i] * inv_cols;
}

void launch_row_shift(double* Z, int64_t n, int64_t ncols, int64_t ld, const double* rowsum, double inv_cols,
                      cudaStream_t stream) {
  if (n <= 0 || ncols <= 0) return;
  unsigned gx = static_cast<unsigned>((n + 255) / 256);
  if (gx > 8) gx = 8;
  for (int64_t j0 = 0; j0 < ncols; j0 += 65535) {
    const unsigned gy = static_cast<unsigned>(ncols - j0 < 65535 ? ncols - j0 : 65535);
    row_shift_kernel<<<dim3(gx, gy), 256, 0, stream>>>(Z + j0 * ld, n, ld, rowsum, inv_cols);
  }
  GBM_CUDA(cudaGetLastError());
}

// dst[i, j] = src[rows[i]-1, cols[j]-1]; rows / cols nullable (identity).
__global__ void __launch_bounds__(256)
    gather_kernel(const double* __restrict__ src, int64_t lds, const int64_t* __restrict__ rows, int64_t n,
                  const int64_t* __restrict__ cols, double* __restrict__ dst, int64_t ldd) {
  const int64_t j = blockIdx.y;
  const int64_t sj = cols ? cols[j] - 1 : j;
  const double* s = src + sj * lds;
  double* d = dst + j * ldd;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    d[i] = s[rows ? rows[i] - 1 : i];
}

void launch_gather(const double* src, int64_t lds, const int64_t* rows, int64_t n, const int64_t* cols, int64_t p,
                   double* dst, int64_t ldd, cudaStream_t stream) {
  if (n <= 0 || p <= 0) return;
  unsigned gx = static_cast<unsigned>((n + 255) / 256);
  if (gx > 16) gx = 16;
  for (int64_t j0 = 0; j0 < p; j0 += 65535) {
    const unsigned gy = static_cast<unsigned>(p - j0 < 65535 ? p - j0 : 65535);
    gather_kernel<<<dim3(gx, gy), 256, 0, stream>>>(src, lds, rows, n, cols ? cols + j0 : nullptr, dst + j0 * ldd,
                                                    ldd);
    if (!cols) src += 65535 * lds;
  }
  GBM_CUDA(cudaGetLastError());
}

// dst[i, c] = (src[i, cols[c]-1] - mean[cols[c]-1]) / sd[cols[c]-1]   (mean/sd nullable: plain gather)
// G = (G .- mean(G, dims=1)) ./ v[idx_cols]'  (/root/reference/src/gwas.jl:114, :129) on the device.
__global__ void __launch_bounds__(256)
    gather_standardise_kernel(const double* __restrict__ src, int64_t lds, int64_t n, const int64_t* __restrict__ cols,
                              const double* __restrict__ mean, const double* __restrict__ sd,
                              double* __restrict__ dst, int64_t ldd) {
  const int64_t c = blockIdx.y;
  const int64_t sj = cols ? cols[c] - 1 : c;
  const double mu = mean ? mean[sj] : 0.0, v = sd ? sd[sj] : 1.0;
  const double* s = src + sj * lds;
  double* d = dst + c * ldd;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    d[i] = (mean || sd) ? (s[i] - mu) / v : s[i];
}

// the same from one-byte dosage codes (a = code / 240, correctly rounded: exactly the packed matrix' values)
__global__ void __launch_bounds__(256)
    gather_standardise_u8_kernel(const uint8_t* __restrict__ src, int64_t lds, int64_t n,
                                 const int64_t* __restrict__ cols, const double* __restrict__ mean,
                                 const double* __restrict__ sd, double* __restrict__ dst, int64_t ldd) {
  const int64_t c = blockIdx.y;
  const int64_t sj = cols ? cols[c] - 1 : c;
  const double mu = mean ? mean[sj] : 0.0, v = sd ? sd[sj] : 1.0;
  const uint8_t* s = src + sj * lds;
  double* d = dst + c * ldd;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const double a = static_cast<double>(s[i]) / 240.0;
    d[i] = (mean || sd) ? (a - mu) / v : a;
  }
}

void launch_gather_standardise_u8(const uint8_t* src, int64_t lds, int64_t n, const int64_t* cols, int64_t ncols,
                                  const double* mean, const double* sd, double* dst, int64_t ldd,
                                  cudaStream_t stream) {
  if (n <= 0 || ncols <= 0) return;
  unsigned gx = static_cast<unsigned>((n + 255) / 256);
  if (gx > 16) gx = 16;
  for (int64_t c0 = 0; c0 < ncols; c0 += 65535) {
    const unsigned gy = static_cast<unsigned>(ncols - c0 < 65535 ? ncols - c0 : 65535);
    gather_standardise_u8_kernel<<<dim3(gx, gy), 256, 0, stream>>>(src, lds, n, cols ? cols + c0 : nullptr, mean, sd,
                                                                    dst + c0 * ldd, ldd);
    if (!cols) src += 65535 * lds;
  }
  GBM_CUDA(cudaGetLastError());
}

void launch_gather_standardise(const double* src, int64_t lds, int64_t n, const int64_t* cols, int64_t ncols,
                               const double* mean, const double* sd, double* dst, int64_t ldd, cudaStream_t stream) {
  if (n <= 0 || ncols <= 0) return;
  unsigned gx = static_cast<unsigned>((n + 255) / 256);
  if (gx > 16) gx = 16;
  for (int64_t c0 = 0; c0 < ncols; c0 += 65535) {
    const unsigned gy = static_cast<unsigned>(ncols - c0 < 65535 ? ncols - c0 : 65535);
    gather_standardise_kernel<<<dim3(gx, gy), 256, 0, stream>>>(src, lds, n, cols ? cols + c0 : nullptr, mean, sd,
                                                                 dst + c0 * ldd, ldd);
    if (!cols) src += 65535 * lds;
  }
  GBM_CUDA(cudaGetLastError());
}

}  // namespace gbm
