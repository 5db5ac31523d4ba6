// Scene preprocessing on device (SURVEY 8-f1): the reference's featureNormalize / PCANorm
// (tools/hyper_tools.py:8-32, called at :289-292) split into
//   fit   : column means and the centred Gram matrix sum (x-mu)(x-mu)^T in float64 (the reference
//           computes np.cov and the per-band std in float64); the B x B SVD stays on the host;
//   apply : per pixel  spectra = (x - mu_b) / sigma_b            (featureNormalize(X, 1), :292)
//                       cube    = ((x - mu_b) . U[:, :60] - m) / s  (PCANorm + featureNormalize, :289)
//           i.e. both inputs of the scene path derive from the raw cube, so the end-to-end entry
//           point only has to move the raw uint16 cube over PCIe (42.7 MB instead of 135 MB for PaviaU).
#include "common.cuh"

namespace cmlpl {

template <typename T> __device__ __forceinline__ double to_f64(T v) { return double(v); }

// ---- column sums (float64), one warp-column group per 32 columns
template <typename T>
__global__ void colsum_f64_kernel(const T* __restrict__ x, int64_t n, int B, double* __restrict__ sum) {
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rgrp = threadIdx.x >> 5, ngrp = blockDim.x >> 5;
  double s = 0.0;
  if (col < B)
    for (int64_t r = blockIdx.y * ngrp + rgrp; r < n; r += int64_t(gridDim.y) * ngrp) s += to_f64(x[r * B + col]);
  __shared__ double part[8][33];
  part[rgrp][threadIdx.x & 31] = s;
  __syncthreads();
  if (rgrp == 0 && col < B) {
    double t = 0.0;
    for (int i = 0; i < ngrp; ++i) t += part[i][threadIdx.x];
    atomicAdd(sum + col, t);
  }
}

// ---- the same from a band-major cube (BIL / BSQ): a CTA sums one band over a group of rows, threads along the columns
template <typename T>
__global__ void __launch_bounds__(256)
colsum_f64_bm_kernel(const T* __restrict__ x, BandMajor bm, int rows, double* __restrict__ sum) {
  const int b = blockIdx.x;
  double s = 0.0;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const T* line = x + int64_t(r) * bm.rs + int64_t(b) * bm.bs;
    for (int c = threadIdx.x; c < bm.cols; c += blockDim.x) s += to_f64(line[c]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ double part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += part[i];
    atomicAdd(sum + b, t);
  }
}

// ---- centred Gram matrix, 32x32 tiles of G, row chunks over blockIdx.z, float64 accumulation.  kBM: a band-major cube
// (addressed through bm), staged with pixels as the fast index so that a warp's loads of one band are consecutive columns
template <typename T, bool kBM>
__device__ __forceinline__ void
gram_f64_body(const T* __restrict__ x, int64_t n, int B, const double* __restrict__ mean, double* __restrict__ gram,
              int64_t rows_per_cta, BandMajor bm) {
  __shared__ double sa[32][33], sb[32][33];
  const int ti = blockIdx.y * 32, tj = blockIdx.x * 32;
  if (tj < ti) return;                                     // symmetric: upper tiles only, mirrored by the host
  __builtin_assume(threadIdx.x < 256);                     // the kernels' launch bounds, as seen by the inlined body
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // thread owns G[ti + ty*4 .. +3][tj + tx]
  double acc[4] = {0, 0, 0, 0};
  const int64_t r0 = blockIdx.z * rows_per_cta, r1 = (r0 + rows_per_cta < n) ? r0 + rows_per_cta : n;
  const double mi = 0, mj = 0; (void)mi; (void)mj;
  for (int64_t r = r0; r < r1; r += 32) {
    // stage 32 rows x 32 columns of the two column blocks (centred)
    if constexpr (kBM) {
      const int rr = threadIdx.x & 31;
      const int64_t row = r + rr, pr = row / bm.cols;
      const T* xp = x + pr * bm.rs + (row - pr * bm.cols);
      for (int cc = threadIdx.x >> 5; cc < 32; cc += 8) {
        sa[rr][cc] = (row < r1 && ti + cc < B) ? to_f64(xp[(ti + cc) * bm.bs]) - mean[ti + cc] : 0.0;
        sb[rr][cc] = (row < r1 && tj + cc < B) ? to_f64(xp[(tj + cc) * bm.bs]) - mean[tj + cc] : 0.0;
      }
    } else {
      for (int e = threadIdx.x; e < 32 * 32; e += 256) {
        const int rr = e >> 5, cc = e & 31;
        const int64_t row = r + rr;
        sa[rr][cc] = (row < r1 && ti + cc < B) ? to_f64(x[row * B + ti + cc]) - mean[ti + cc] : 0.0;
        sb[rr][cc] = (row < r1 && tj + cc < B) ? to_f64(x[row * B + tj + cc]) - mean[tj + cc] : 0.0;
      }
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < 32; ++rr) {
      const double b = sb[rr][tx];
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q] = fma(sa[rr][ty * 4 + q], b, acc[q]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int i = ti + ty * 4 + q, j = tj + tx;
    if (i < B && j < B) atomicAdd(gram + int64_t(i) * B + j, acc[q]);
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
gram_f64_kernel(const T* __restrict__ x, int64_t n, int B, const double* __restrict__ mean, double* __restrict__ gram,
                int64_t rows_per_cta) {
  gram_f64_body<T, false>(x, n, B, mean, gram, rows_per_cta, BandMajor{});
}

template <typename T>
__global__ void __launch_bounds__(256)
gram_f64_bm_kernel(const T* __restrict__ x, BandMajor bm, int64_t n, int B, const double* __restrict__ mean,
                   double* __restrict__ gram, int64_t rows_per_cta) {
  gram_f64_body<T, true>(x, n, B, mean, gram, rows_per_cta, bm);
}

// ---- apply: one warp per pixel; lanes stride over bands for the spectra, then over the 60 components
template <typename T>
__global__ void __launch_bounds__(256)
preprocess_apply_kernel(const T* __restrict__ x, int64_t n, int B, int npc, const float* __restrict__ mu,
                        const float* __restrict__ inv_sigma, const float* __restrict__ Us /* [B][npc], U/s */,
                        const float* __restrict__ shift /* [npc], m/s */, float* __restrict__ cube,
                        float* __restrict__ spectra) {
  extern __shared__ float sm[];                            // per warp: centred spectrum [B]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* xc = sm + wid * B;
  for (int64_t p = blockIdx.x * int64_t(blockDim.x >> 5) + wid; p < n; p += int64_t(gridDim.x) * (blockDim.x >> 5)) {
    for (int b = lane; b < B; b += 32) {
      const float c = float(x[p * B + b]) - mu[b];
      xc[b] = c;
      if (spectra) spectra[p * B + b] = c * inv_sigma[b];
    }
    __syncwarp();
    for (int k = lane; k < npc; k += 32) {
      float acc = 0.f;
      for (int b = 0; b < B; ++b) acc = fmaf(xc[b], __ldg(Us + b * npc + k), acc);
      cube[p * npc + k] = acc - shift[k];
    }
    __syncwarp();
  }
}

__global__ void scale_f64_kernel(double* v, int n, double f) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] *= f;
}

// mean and centred Gram of a rows x cols cube, pixel-major (bm == nullptr) or band-major
template <typename T>
static int fit_impl(const T* x, const BandMajor* bm, int64_t rows, int B, double* mean, double* gram, cudaStream_t s) {
  const int64_t n = rows * (bm ? bm->cols : 1);
  CMLPL_CUDA(cudaMemsetAsync(mean, 0, sizeof(double) * B, s));
  CMLPL_CUDA(cudaMemsetAsync(gram, 0, sizeof(double) * B * B, s));
  if (bm) {
    colsum_f64_bm_kernel<T><<<dim3(B, unsigned(rows < 256 ? rows : 256)), 256, 0, s>>>(x, *bm, int(rows), mean);
  } else {
    const int gy = int(n / 256 < 1 ? 1 : (n / 256 > 512 ? 512 : n / 256));
    colsum_f64_kernel<T><<<dim3((B + 31) / 32, gy), 256, 0, s>>>(x, n, B, mean);
  }
  CMLPL_CHECK_LAUNCH("colsum_f64");
  scale_f64_kernel<<<(B + 255) / 256, 256, 0, s>>>(mean, B, 1.0 / double(n));
  CMLPL_CHECK_LAUNCH("mean_scale");
  const int tiles = (B + 31) / 32;
  int64_t rows_per_cta = (n + 63) / 64;
  rows_per_cta = (rows_per_cta + 31) / 32 * 32;
  const int gz = int((n + rows_per_cta - 1) / rows_per_cta);
  if (bm)
    gram_f64_bm_kernel<T><<<dim3(tiles, tiles, gz), 256, 0, s>>>(x, *bm, n, B, mean, gram, rows_per_cta);
  else
    gram_f64_kernel<T><<<dim3(tiles, tiles, gz), 256, 0, s>>>(x, n, B, mean, gram, rows_per_cta);
  CMLPL_CHECK_LAUNCH("gram_f64");
  return CMLPL_OK;
}

static int fit_cube(const char* fn, const void* x, int dtype, int64_t rows, int cols, int B, double* mean, double* gram,
                    cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && mean && gram, "%s: null pointer", fn);
  const int rc = check_raw_code(fn, "x", x, dtype);
  if (rc != CMLPL_OK) return rc;
  CMLPL_CHECK_ARG(rows > 0 && cols > 0 && rows * cols > 1 && B > 0, "%s: bad dims (rows=%lld cols=%d bands=%d)", fn,
                  static_cast<long long>(rows), cols, B);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int il = dtype & 0xf0, sample = dtype & 0x0f;
  const BandMajor bmv = band_major(dtype, B, rows, cols);
  const BandMajor* bm = il == CMLPL_RAW_BIP ? nullptr : &bmv;
  const int64_t r = bm ? rows : rows * cols;                 // pixel-major: one row of cols * B samples per pixel
  if (sample == CMLPL_RAW_U16) return fit_impl(static_cast<const uint16_t*>(x), bm, r, B, mean, gram, s);
  if (sample == CMLPL_RAW_I16) return fit_impl(static_cast<const int16_t*>(x), bm, r, B, mean, gram, s);
  return fit_impl(static_cast<const float*>(x), bm, r, B, mean, gram, s);
}

}  // namespace cmlpl

using namespace cmlpl;

// dtype: sample | interleave (include/cmlpl.h, CMLPL_RAW_*)
extern "C" int cmlpl_preprocess_fit_cube_f64(const void* x, int dtype, int rows, int cols, int B, double* mean,
                                             double* gram, cmlpl_stream_t stream) {
  return fit_cube("preprocess_fit_cube", x, dtype, rows, cols, B, mean, gram, stream);
}

// x [n, B] band-interleaved-by-pixel: the cube fit with rows = n, cols = 1
extern "C" int cmlpl_preprocess_fit_f64(const void* x, int dtype, int64_t n, int B, double* mean, double* gram,
                                        cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG((dtype & 0xf0) != CMLPL_RAW_BIL && (dtype & 0xf0) != CMLPL_RAW_BSQ,
                  "preprocess_fit: x is [n, B] band-interleaved-by-pixel (BIL / BSQ: cmlpl_preprocess_fit_cube_f64)");
  return fit_cube("preprocess_fit", x, dtype, n, 1, B, mean, gram, stream);
}

extern "C" int cmlpl_preprocess_apply(const void* x, int dtype, int64_t n, int B, int npc, const float* mu,
                                      const float* inv_sigma, const float* Us, const float* shift, float* cube,
                                      float* spectra, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && mu && inv_sigma && Us && shift && cube, "preprocess_apply: null pointer");
  CMLPL_CHECK_ARG(n >= 0 && B > 0 && B <= 1024 && npc > 0 && dtype >= CMLPL_RAW_U16 && dtype <= CMLPL_RAW_I16,
                  "preprocess_apply: bad args (dtype: BIP uint16, float32 or int16)");
  if (n == 0) return CMLPL_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int64_t grid = (n + 7) / 8; const int64_t cap = int64_t(sm_count()) * 8; if (grid > cap) grid = cap;
  const size_t smem = sizeof(float) * 8 * B;
  if (dtype == CMLPL_RAW_U16)
    preprocess_apply_kernel<uint16_t><<<int(grid), 256, smem, s>>>(static_cast<const uint16_t*>(x), n, B, npc, mu, inv_sigma, Us, shift, cube, spectra);
  else if (dtype == CMLPL_RAW_I16)
    preprocess_apply_kernel<int16_t><<<int(grid), 256, smem, s>>>(static_cast<const int16_t*>(x), n, B, npc, mu, inv_sigma, Us, shift, cube, spectra);
  else
    preprocess_apply_kernel<float><<<int(grid), 256, smem, s>>>(static_cast<const float*>(x), n, B, npc, mu, inv_sigma, Us, shift, cube, spectra);
  CMLPL_CHECK_LAUNCH("preprocess_apply");
  return CMLPL_OK;
}
