// Scene preprocessing on device (SURVEY 8-f1): the reference's featureNormalize / PCANorm
// (tools/hyper_tools.py:8-32, called at :289-292) split into
//   fit   : column means and the centred Gram matrix sum (x-mu)(x-mu)^T in float64 (the reference
//           computes np.cov and the per-band std in float64); the B x B SVD stays on the host;
//   apply : per pixel  spectra = (x - mu_b) / sigma_b            (featureNormalize(X, 1), :292)
//                       cube    = ((x - mu_b) . U[:, :60] - m) / s  (PCANorm + featureNormalize, :289)
//           i.e. both inputs of the scene path derive from the raw cube, so the end-to-end entry
//           point only has to move the raw uint16 cube over PCIe (42.7 MB instead of 135 MB for PaviaU).
// No-data pixels (fill values, NaN / Inf): valid_mask builds the u8 validity mask [rows, cols] in one read of the cube;
// with a mask, fit sums over the valid pixels only and apply writes the imputed values (x = mu) for the others.
#include <math.h>

#include "common.cuh"

namespace cmlpl {

template <typename T> __device__ __forceinline__ double to_f64(T v) { return double(v); }

// ---- column sums (float64), one warp-column group per 32 columns; valid (u8 [n] or nullptr): pixels with 0 are skipped.
// Feature col < B reads raw band raw_band(sel, col) of rows of ld samples (Sel: common.cuh)
template <typename T, class Sel>
__global__ void colsum_f64_kernel(const T* __restrict__ x, int64_t n, int B, int ld, Sel sel,
                                  const uint8_t* __restrict__ valid, double* __restrict__ sum) {
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rgrp = threadIdx.x >> 5, ngrp = blockDim.x >> 5;
  double s = 0.0;
  if (col < B) {
    const T* xc = x + raw_band(sel, col);
    for (int64_t r = blockIdx.y * ngrp + rgrp; r < n; r += int64_t(gridDim.y) * ngrp)
      if (!valid || valid[r]) s += to_f64(xc[r * ld]);
  }
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
template <typename T, class Sel>
__global__ void __launch_bounds__(256)
colsum_f64_bm_kernel(const T* __restrict__ x, BandMajor bm, int rows, Sel sel, const uint8_t* __restrict__ valid,
                     double* __restrict__ sum) {
  const int b = blockIdx.x;
  double s = 0.0;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const T* line = x + int64_t(r) * bm.rs + int64_t(raw_band(sel, b)) * bm.bs;
    const uint8_t* vline = valid ? valid + int64_t(r) * bm.cols : nullptr;
    for (int c = threadIdx.x; c < bm.cols; c += blockDim.x)
      if (!vline || vline[c]) s += to_f64(line[c]);
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
// (addressed through bm), staged with pixels as the fast index so that a warp's loads of one band are consecutive columns.
// valid (u8 [n] over the pixels in raster order, or nullptr): a pixel with 0 is staged as a zero row.  Feature i < B is
// raw band raw_band(sel, i); a pixel-major row holds ld samples
template <typename T, bool kBM, class Sel>
__device__ __forceinline__ void
gram_f64_body(const T* __restrict__ x, int64_t n, int B, int ld, const Sel& sel, const double* __restrict__ mean,
              double* __restrict__ gram, int64_t rows_per_cta, BandMajor bm, const uint8_t* __restrict__ valid) {
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
      const bool ok = row < r1 && (!valid || valid[row]);
      for (int cc = threadIdx.x >> 5; cc < 32; cc += 8) {
        sa[rr][cc] = (ok && ti + cc < B) ? to_f64(xp[int64_t(raw_band(sel, ti + cc)) * bm.bs]) - mean[ti + cc] : 0.0;
        sb[rr][cc] = (ok && tj + cc < B) ? to_f64(xp[int64_t(raw_band(sel, tj + cc)) * bm.bs]) - mean[tj + cc] : 0.0;
      }
    } else {
      const int cc = threadIdx.x & 31;                       // the same column for all of this thread's rows
      const int ba = ti + cc < B ? raw_band(sel, ti + cc) : 0, bb = tj + cc < B ? raw_band(sel, tj + cc) : 0;
      for (int e = threadIdx.x; e < 32 * 32; e += 256) {
        const int rr = e >> 5;
        const int64_t row = r + rr;
        const bool ok = row < r1 && (!valid || valid[row]);
        sa[rr][cc] = (ok && ti + cc < B) ? to_f64(x[row * ld + ba]) - mean[ti + cc] : 0.0;
        sb[rr][cc] = (ok && tj + cc < B) ? to_f64(x[row * ld + bb]) - mean[tj + cc] : 0.0;
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

template <typename T, class Sel>
__global__ void __launch_bounds__(256)
gram_f64_kernel(const T* __restrict__ x, int64_t n, int B, int ld, Sel sel, const double* __restrict__ mean,
                double* __restrict__ gram, int64_t rows_per_cta, const uint8_t* __restrict__ valid) {
  gram_f64_body<T, false>(x, n, B, ld, sel, mean, gram, rows_per_cta, BandMajor{}, valid);
}

template <typename T, class Sel>
__global__ void __launch_bounds__(256)
gram_f64_bm_kernel(const T* __restrict__ x, BandMajor bm, int64_t n, int B, Sel sel, const double* __restrict__ mean,
                   double* __restrict__ gram, int64_t rows_per_cta, const uint8_t* __restrict__ valid) {
  gram_f64_body<T, true>(x, n, B, 0, sel, mean, gram, rows_per_cta, bm, valid);
}

// ---- apply: one warp per pixel; lanes stride over bands for the spectra, then over the 60 components.  valid (u8 [n] or
// nullptr): a no-data pixel stands in as its band means x = mu, i.e. a zero spectra row and the PCA row -shift.
// Feature b < B is raw band raw_band(sel, b) of pixel rows of ld samples
template <typename T, class Sel>
__global__ void __launch_bounds__(256)
preprocess_apply_kernel(const T* __restrict__ x, int64_t n, int B, int ld, Sel sel, int npc, const float* __restrict__ mu,
                        const float* __restrict__ inv_sigma, const float* __restrict__ Us /* [B][npc], U/s */,
                        const float* __restrict__ shift /* [npc], m/s */, const uint8_t* __restrict__ valid,
                        float* __restrict__ cube, float* __restrict__ spectra) {
  extern __shared__ float sm[];                            // per warp: centred spectrum [B]; then the staged band list
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* xc = sm + wid * B;
  const auto bands = stage_bands(sel, reinterpret_cast<uint16_t*>(sm + 8 * B));   // lanes read it divergently
  if constexpr (Sel::kSel) __syncthreads();
  for (int64_t p = blockIdx.x * int64_t(blockDim.x >> 5) + wid; p < n; p += int64_t(gridDim.x) * (blockDim.x >> 5)) {
    if (valid && !valid[p]) {
      if (spectra)
        for (int b = lane; b < B; b += 32) spectra[p * B + b] = 0.f;
      for (int k = lane; k < npc; k += 32) cube[p * npc + k] = -shift[k];
      continue;
    }
    for (int b = lane; b < B; b += 32) {
      const float c = float(x[p * ld + raw_band(bands, b)]) - mu[b];
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

// ---- validity mask (include/cmlpl.h, cmlpl_valid_mask_u8).  A sample is missing when it equals the fill value in the
// sample type; a float32 sample that is not finite is always missing, and nan_only leaves it at that.  A pixel is no-data
// (valid byte 0) when any of its bands is missing.  Missing samples are counted per band into a shared-memory histogram
// [B] that each CTA adds to band_missing once.
template <typename T> __device__ __forceinline__ bool missing(T v, T fill, bool) { return v == fill; }
__device__ __forceinline__ bool missing(float v, float fill, bool nan_only) {
  return !isfinite(v) || (!nan_only && v == fill);
}

// band-interleaved-by-pixel: one warp per pixel, its B contiguous samples on consecutive lanes, 8 loads in flight per lane.
// Feature b < B is raw band raw_band(sel, b) of pixel rows of ld samples
template <typename T, class Sel>
__global__ void __launch_bounds__(256)
valid_mask_kernel(const T* __restrict__ x, int64_t n, int B, int ld, Sel sel, T fill, bool nan_only,
                  uint8_t* __restrict__ valid, unsigned long long* __restrict__ n_valid,
                  unsigned long long* __restrict__ band_missing) {
  extern __shared__ unsigned smiss[];                     // [B] this CTA's missing samples per band; then the band list
  __shared__ unsigned long long scount;
  const auto bands = stage_bands(sel, reinterpret_cast<uint16_t*>(smiss + B));   // lanes read it divergently
  for (int b = threadIdx.x; b < B; b += blockDim.x) smiss[b] = 0;
  if (threadIdx.x == 0) scount = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t nw = int64_t(gridDim.x) * (blockDim.x >> 5);
  unsigned long long cnt = 0;
  for (int64_t p = blockIdx.x * int64_t(blockDim.x >> 5) + (threadIdx.x >> 5); p < n; p += nw) {
    const T* px = x + p * ld;
    bool any = false;
    for (int b0 = 0; b0 < B; b0 += 256) {
      T v[8];
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const int b = b0 + lane + 32 * m;
        v[m] = b < B ? px[raw_band(bands, b)] : fill;
      }
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const int b = b0 + lane + 32 * m;
        if (b < B && missing(v[m], fill, nan_only)) {
          any = true;
          atomicAdd(&smiss[b], 1u);
        }
      }
    }
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) { valid[p] = any ? 0 : 1; cnt += !any; }
  }
  if (lane == 0 && cnt) atomicAdd(&scount, cnt);
  __syncthreads();
  if (threadIdx.x == 0 && scount) atomicAdd(n_valid, scount);
  if (band_missing)
    for (int b = threadIdx.x; b < B; b += blockDim.x)
      if (smiss[b]) atomicAdd(band_missing + b, (unsigned long long)smiss[b]);
}

// band-major (BIL / BSQ): a thread owns one pixel of a row and walks its bands, each load coalesced along the warp's
// consecutive columns (as x16_tile_kernel); rows over blockIdx.y.  Feature b < B is raw band raw_band(sel, b) (warp-uniform)
template <typename T, class Sel>
__global__ void __launch_bounds__(256)
valid_mask_bm_kernel(const T* __restrict__ x, BandMajor bm, int rows, int B, Sel sel, T fill, bool nan_only,
                     uint8_t* __restrict__ valid, unsigned long long* __restrict__ n_valid,
                     unsigned long long* __restrict__ band_missing) {
  extern __shared__ unsigned smiss[];
  __shared__ unsigned long long scount;
  for (int b = threadIdx.x; b < B; b += blockDim.x) smiss[b] = 0;
  if (threadIdx.x == 0) scount = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = c < bm.cols;                            // the warp stays converged for its ballots
  unsigned long long cnt = 0;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const T* px = x + int64_t(r) * bm.rs + (in ? c : 0);
    bool any = false;
    for (int b0 = 0; b0 < B; b0 += 8) {
      T v[8];
#pragma unroll
      for (int m = 0; m < 8; ++m) v[m] = (in && b0 + m < B) ? px[int64_t(raw_band(sel, b0 + m)) * bm.bs] : fill;
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const bool miss = in && b0 + m < B && missing(v[m], fill, nan_only);
        const unsigned bal = __ballot_sync(0xffffffffu, miss);
        any |= miss;
        if (bal && lane == 0) atomicAdd(&smiss[b0 + m], unsigned(__popc(bal)));
      }
    }
    if (in) { valid[int64_t(r) * bm.cols + c] = any ? 0 : 1; cnt += !any; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0 && cnt) atomicAdd(&scount, cnt);
  __syncthreads();
  if (threadIdx.x == 0 && scount) atomicAdd(n_valid, scount);
  if (band_missing)
    for (int b = threadIdx.x; b < B; b += blockDim.x)
      if (smiss[b]) atomicAdd(band_missing + b, (unsigned long long)smiss[b]);
}

__global__ void scale_f64_kernel(double* v, int n, double f) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] *= f;
}

// the masked fit's mean: the column sums over the n_valid valid pixels (counted on the device)
__global__ void scale_by_count_f64_kernel(double* v, int n, const int64_t* __restrict__ count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] *= 1.0 / double(*count);
}

// number of nonzero bytes of valid [n] -> *count (zeroed by the caller)
__global__ void __launch_bounds__(256) count_valid_kernel(const uint8_t* __restrict__ valid, int64_t n,
                                                          unsigned long long* __restrict__ count) {
  unsigned long long c = 0;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    c += valid[i] != 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, c);
}

// mean and centred Gram of a rows x cols cube, pixel-major (bm == nullptr; rows of ld samples) or band-major, over the B
// features sel selects; valid (u8 [rows * cols] or nullptr): the moments of the pixels with a nonzero byte, counted into
// *n_valid
template <typename T, class Sel>
static int fit_impl(const T* x, const BandMajor* bm, int64_t rows, int B, int ld, const Sel& sel, const uint8_t* valid,
                    double* mean, double* gram, int64_t* n_valid, cudaStream_t s) {
  const int64_t n = rows * (bm ? bm->cols : 1);
  CMLPL_CUDA(cudaMemsetAsync(mean, 0, sizeof(double) * B, s));
  CMLPL_CUDA(cudaMemsetAsync(gram, 0, sizeof(double) * B * B, s));
  if (valid) {
    CMLPL_CUDA(cudaMemsetAsync(n_valid, 0, sizeof(int64_t), s));
    int64_t g = (n + 255) / 256; const int64_t cap = int64_t(sm_count()) * 8; if (g > cap) g = cap;
    count_valid_kernel<<<int(g), 256, 0, s>>>(valid, n, reinterpret_cast<unsigned long long*>(n_valid));
    CMLPL_CHECK_LAUNCH("count_valid");
  }
  if (bm) {
    colsum_f64_bm_kernel<T><<<dim3(B, unsigned(rows < 256 ? rows : 256)), 256, 0, s>>>(x, *bm, int(rows), sel, valid, mean);
  } else {
    const int gy = int(n / 256 < 1 ? 1 : (n / 256 > 512 ? 512 : n / 256));
    colsum_f64_kernel<T><<<dim3((B + 31) / 32, gy), 256, 0, s>>>(x, n, B, ld, sel, valid, mean);
  }
  CMLPL_CHECK_LAUNCH("colsum_f64");
  if (valid)
    scale_by_count_f64_kernel<<<(B + 255) / 256, 256, 0, s>>>(mean, B, n_valid);
  else
    scale_f64_kernel<<<(B + 255) / 256, 256, 0, s>>>(mean, B, 1.0 / double(n));
  CMLPL_CHECK_LAUNCH("mean_scale");
  const int tiles = (B + 31) / 32;
  int64_t rows_per_cta = (n + 63) / 64;
  rows_per_cta = (rows_per_cta + 31) / 32 * 32;
  const int gz = int((n + rows_per_cta - 1) / rows_per_cta);
  if (bm)
    gram_f64_bm_kernel<T><<<dim3(tiles, tiles, gz), 256, 0, s>>>(x, *bm, n, B, sel, mean, gram, rows_per_cta, valid);
  else
    gram_f64_kernel<T><<<dim3(tiles, tiles, gz), 256, 0, s>>>(x, n, B, ld, sel, mean, gram, rows_per_cta, valid);
  CMLPL_CHECK_LAUNCH("gram_f64");
  return CMLPL_OK;
}

// sel: the band list of cmlpl_preprocess_fit_sel_f64 (B raw bands, sel->n features), or nullptr for all B bands
static int fit_cube(const char* fn, const void* x, int dtype, int64_t rows, int cols, int B, const PreBands* sel,
                    const uint8_t* valid, double* mean, double* gram, int64_t* n_valid, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && mean && gram, "%s: null pointer", fn);
  const int rc = check_raw_code(fn, "x", x, dtype);
  if (rc != CMLPL_OK) return rc;
  CMLPL_CHECK_ARG(rows > 0 && cols > 0 && rows * cols > 1 && B > 0, "%s: bad dims (rows=%lld cols=%d bands=%d)", fn,
                  static_cast<long long>(rows), cols, B);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int il = dtype & 0xf0;
  const BandMajor bmv = band_major(dtype, B, rows, cols);
  const BandMajor* bm = il == CMLPL_RAW_BIP ? nullptr : &bmv;
  const int64_t r = bm ? rows : rows * cols;                 // pixel-major: one row of cols * B samples per pixel
  return with_sample(dtype, [&](auto sample) {
    using T = decltype(sample);
    return sel ? fit_impl(static_cast<const T*>(x), bm, r, sel->n, B, *sel, valid, mean, gram, n_valid, s)
               : fit_impl(static_cast<const T*>(x), bm, r, B, B, AllBands{}, valid, mean, gram, n_valid, s);
  });
}

// widest spectrum of the mask kernels: their per-band histogram of missing samples sits in shared memory (32 KB)
constexpr int kMaskMaxBands = 8192;

// over the B features sel selects of a cube whose pixel-major rows hold ld samples
template <typename T, class Sel>
static int valid_mask_impl(const T* x, const BandMajor* bm, int64_t rows, int cols, int B, int ld, const Sel& sel, T fill,
                           bool nan_only, uint8_t* valid, int64_t* n_valid, int64_t* band_missing, cudaStream_t s) {
  CMLPL_CUDA(cudaMemsetAsync(n_valid, 0, sizeof(int64_t), s));
  if (band_missing) CMLPL_CUDA(cudaMemsetAsync(band_missing, 0, sizeof(int64_t) * B, s));
  size_t smem = sizeof(unsigned) * B;
  auto* nv = reinterpret_cast<unsigned long long*>(n_valid);
  auto* miss = reinterpret_cast<unsigned long long*>(band_missing);
  const int64_t cap = int64_t(sm_count()) * 8;
  if (bm) {
    const int64_t gx = (cols + 255) / 256;
    int64_t gy = cap * 2 / gx < 1 ? 1 : cap * 2 / gx;
    if (gy > rows) gy = rows;
    if (gy > 65535) gy = 65535;
    valid_mask_bm_kernel<T><<<dim3(unsigned(gx), unsigned(gy)), 256, smem, s>>>(x, *bm, int(rows), B, sel, fill, nan_only,
                                                                               valid, nv, miss);
  } else {
    const int64_t n = rows * cols;
    int64_t g = (n + 7) / 8;
    if (g > cap) g = cap;
    if constexpr (Sel::kSel) {                                // + the list staged after the histogram
      smem += sizeof(uint16_t) * B;
      auto kern = valid_mask_kernel<T, Sel>;
      CMLPL_MAX_DYN_SMEM(kern, smem);
    }
    valid_mask_kernel<T><<<int(g), 256, smem, s>>>(x, n, B, ld, sel, fill, nan_only, valid, nv, miss);
  }
  CMLPL_CHECK_LAUNCH("valid_mask");
  return CMLPL_OK;
}

// preprocess_apply_kernel over x [n, B] (BIP), with or without a validity mask; sel: the band list of
// cmlpl_preprocess_apply_sel (B raw bands, sel->n features), or nullptr for all B bands
static int apply_impl(const char* fn, const void* x, int dtype, int64_t n, int B, const PreBands* sel, int npc,
                      const float* mu, const float* inv_sigma, const float* Us, const float* shift, const uint8_t* valid,
                      float* cube, float* spectra, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && mu && inv_sigma && Us && shift && cube, "%s: null pointer", fn);
  const int nf = sel ? sel->n : B;                           // features per pixel
  CMLPL_CHECK_ARG(n >= 0 && B > 0 && nf <= 1024 && npc > 0 && dtype >= CMLPL_RAW_U16 && dtype <= CMLPL_RAW_I16,
                  "%s: bad args (dtype: BIP uint16, float32 or int16)", fn);
  if (n == 0) return CMLPL_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int64_t grid = (n + 7) / 8; const int64_t cap = int64_t(sm_count()) * 8; if (grid > cap) grid = cap;
  const size_t smem = sizeof(float) * 8 * nf + (sel ? sizeof(uint16_t) * nf : 0);
  with_sample(dtype, [&](auto sample) {
    using T = decltype(sample);
    const T* xt = static_cast<const T*>(x);
    if (sel)
      preprocess_apply_kernel<T><<<int(grid), 256, smem, s>>>(xt, n, nf, B, *sel, npc, mu, inv_sigma, Us, shift, valid, cube,
                                                              spectra);
    else
      preprocess_apply_kernel<T><<<int(grid), 256, smem, s>>>(xt, n, B, B, AllBands{}, npc, mu, inv_sigma, Us, shift, valid, cube,
                                                              spectra);
  });
  CMLPL_CHECK_LAUNCH("preprocess_apply");
  return CMLPL_OK;
}

}  // namespace cmlpl

using namespace cmlpl;

// dtype: sample | interleave (include/cmlpl.h, CMLPL_RAW_*)
extern "C" int cmlpl_preprocess_fit_cube_f64(const void* x, int dtype, int rows, int cols, int B, double* mean,
                                             double* gram, cmlpl_stream_t stream) {
  return fit_cube("preprocess_fit_cube", x, dtype, rows, cols, B, nullptr, nullptr, mean, gram, nullptr, stream);
}

// x [n, B] band-interleaved-by-pixel: the cube fit with rows = n, cols = 1
extern "C" int cmlpl_preprocess_fit_f64(const void* x, int dtype, int64_t n, int B, double* mean, double* gram,
                                        cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG((dtype & 0xf0) != CMLPL_RAW_BIL && (dtype & 0xf0) != CMLPL_RAW_BSQ,
                  "preprocess_fit: x is [n, B] band-interleaved-by-pixel (BIL / BSQ: cmlpl_preprocess_fit_cube_f64)");
  return fit_cube("preprocess_fit", x, dtype, n, 1, B, nullptr, nullptr, mean, gram, nullptr, stream);
}

extern "C" int cmlpl_preprocess_apply(const void* x, int dtype, int64_t n, int B, int npc, const float* mu,
                                      const float* inv_sigma, const float* Us, const float* shift, float* cube,
                                      float* spectra, cmlpl_stream_t stream) {
  return apply_impl("preprocess_apply", x, dtype, n, B, nullptr, npc, mu, inv_sigma, Us, shift, nullptr, cube, spectra, stream);
}

// ---------------------------------------------------------------------------------------------- no-data pixels
// The fill value in the sample type (CMLPL_ERR_ARG unless the type represents it exactly); NaN = non-finite samples only,
// for float32 cubes.  No CUDA call.
static int check_fill(const char* fn, int sample, double fill) {
  if (sample == CMLPL_RAW_F32) {
    CMLPL_CHECK_ARG(isnan(fill) || double(float(fill)) == fill, "%s: fill %.17g is not a float32 value", fn, fill);
    return CMLPL_OK;
  }
  CMLPL_CHECK_ARG(!isnan(fill), "%s: a NaN fill marks non-finite float32 samples; an integer cube needs its fill value", fn);
  const double lo = sample == CMLPL_RAW_U16 ? 0.0 : -32768.0, hi = sample == CMLPL_RAW_U16 ? 65535.0 : 32767.0;
  CMLPL_CHECK_ARG(fill == rint(fill) && fill >= lo && fill <= hi, "%s: fill %.17g is not a%s value", fn, fill,
                  sample == CMLPL_RAW_U16 ? " uint16" : "n int16");
  return CMLPL_OK;
}

// cmlpl_valid_mask_u8 (sel == nullptr) and cmlpl_valid_mask_sel_u8 (the B raw bands' listed ones)
static int valid_mask(const char* fn, const void* raw, int dtype, int64_t rows, int cols, int B, const PreBands* sel,
                      double fill, uint8_t* valid, int64_t* n_valid, int64_t* band_missing, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(raw && valid && n_valid, "%s: null pointer", fn);
  int rc = check_raw_code(fn, "raw", raw, dtype);
  if (rc != CMLPL_OK) return rc;
  const int sample = dtype & 0x0f, il = dtype & 0xf0;
  CMLPL_CHECK_ARG(rows > 0 && cols > 0 && B > 0 && B <= kMaskMaxBands && (il == CMLPL_RAW_BIP || rows < (int64_t(1) << 31)),
                  "%s: bad dims (rows=%lld cols=%d bands=%d; at most %d bands)", fn, static_cast<long long>(rows), cols, B,
                  kMaskMaxBands);
  if ((rc = check_fill(fn, sample, fill)) != CMLPL_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const BandMajor bmv = band_major(dtype, B, rows, cols);
  const BandMajor* bm = il == CMLPL_RAW_BIP ? nullptr : &bmv;
  // (check_fill refuses a NaN fill for the integer types)
  return with_sample(sample, [&](auto sample_type) {
    using T = decltype(sample_type);
    const T* x = static_cast<const T*>(raw);
    const T f = isnan(fill) ? T(0) : T(fill);
    return sel ? valid_mask_impl(x, bm, rows, cols, sel->n, B, *sel, f, bool(isnan(fill)), valid, n_valid, band_missing, s)
               : valid_mask_impl(x, bm, rows, cols, B, B, AllBands{}, f, bool(isnan(fill)), valid, n_valid, band_missing, s);
  });
}

extern "C" int cmlpl_valid_mask_u8(const void* raw, int dtype, int64_t rows, int cols, int B, double fill, uint8_t* valid,
                                   int64_t* n_valid, int64_t* band_missing, cmlpl_stream_t stream) {
  return valid_mask("valid_mask", raw, dtype, rows, cols, B, nullptr, fill, valid, n_valid, band_missing, stream);
}

extern "C" int cmlpl_preprocess_fit_masked_f64(const void* raw, int dtype, int64_t rows, int cols, int B,
                                               const uint8_t* valid, double* mean, double* gram, int64_t* n_valid,
                                               cmlpl_stream_t stream) {
  const char* fn = "preprocess_fit_masked";
  CMLPL_CHECK_ARG(valid && n_valid, "%s: null valid mask or n_valid", fn);
  CMLPL_CHECK_ARG((dtype & 0xf0) == CMLPL_RAW_BIP || rows < (int64_t(1) << 31), "%s: bad dims (rows=%lld)", fn,
                  static_cast<long long>(rows));
  return fit_cube(fn, raw, dtype, rows, cols, B, nullptr, valid, mean, gram, n_valid, stream);
}

extern "C" int cmlpl_preprocess_apply_masked(const void* x, int dtype, int64_t n, int B, int npc, const float* mu,
                                             const float* inv_sigma, const float* Us, const float* shift,
                                             const uint8_t* valid, float* cube, float* spectra, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(valid, "preprocess_apply_masked: null valid mask");
  return apply_impl("preprocess_apply_masked", x, dtype, n, B, nullptr, npc, mu, inv_sigma, Us, shift, valid, cube, spectra,
                    stream);
}

// ---------------------------------------------------------------------------------------------- band selection
// The entry points above over the listed raw bands only (include/cmlpl.h): the list is checked on the host and travels
// by value in the kernel parameters; feature k reads raw band bands_host[k] where the entry point without a list reads
// band k, so the results equal those of the same call on a cube that holds only the listed bands.
extern "C" int cmlpl_valid_mask_sel_u8(const void* raw, int dtype, int64_t rows, int cols, int B, const int* bands_host,
                                       int nsel, double fill, uint8_t* valid, int64_t* n_valid, int64_t* band_missing,
                                       cmlpl_stream_t stream) {
  const char* fn = "valid_mask_sel";
  PreBands sel;
  const int rc = check_band_list(fn, B, bands_host, nsel, kMaskMaxBands, &sel);
  if (rc != CMLPL_OK) return rc;
  return valid_mask(fn, raw, dtype, rows, cols, B, &sel, fill, valid, n_valid, band_missing, stream);
}

extern "C" int cmlpl_preprocess_fit_sel_f64(const void* raw, int dtype, int64_t rows, int cols, int B, const int* bands_host,
                                            int nsel, const uint8_t* valid, double* mean, double* gram, int64_t* n_valid,
                                            cmlpl_stream_t stream) {
  const char* fn = "preprocess_fit_sel";
  PreBands sel;
  const int rc = check_band_list(fn, B, bands_host, nsel, kRawMaxBandsSel, &sel);
  if (rc != CMLPL_OK) return rc;
  CMLPL_CHECK_ARG(!valid || n_valid, "%s: a validity mask needs n_valid", fn);
  CMLPL_CHECK_ARG((dtype & 0xf0) == CMLPL_RAW_BIP || rows < (int64_t(1) << 31), "%s: bad dims (rows=%lld)", fn,
                  static_cast<long long>(rows));
  return fit_cube(fn, raw, dtype, rows, cols, B, &sel, valid, mean, gram, n_valid, stream);
}

extern "C" int cmlpl_preprocess_apply_sel(const void* x, int dtype, int64_t n, int B, const int* bands_host, int nsel, int npc,
                                          const float* mu, const float* inv_sigma, const float* Us, const float* shift,
                                          const uint8_t* valid, float* cube, float* spectra, cmlpl_stream_t stream) {
  const char* fn = "preprocess_apply_sel";
  PreBands sel;
  const int rc = check_band_list(fn, B, bands_host, nsel, 1024, &sel);
  if (rc != CMLPL_OK) return rc;
  return apply_impl(fn, x, dtype, n, B, &sel, npc, mu, inv_sigma, Us, shift, valid, cube, spectra, stream);
}
