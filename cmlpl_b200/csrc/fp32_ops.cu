// fp32 building blocks of BaseNet2 in batch mode (tools/models.py:97-152), NCHW like the
// reference, used by the training forward/backward (SURVEY a5, a12).  All of these are
// one tiled CUDA-core GEMM core (64x64x16 tiles, 4x4 register micro-tiles, fp32 FFMA)
// with different operand-address functors: strided GEMM (nn.Linear fwd/dgrad/wgrad),
// implicit-GEMM convolution forward / data-gradient, and split-K weight-gradient.
// fp32 keeps the training step inside the reference's rtol 1e-5 parity bar.
#include "common.cuh"
#include "gemm_core.cuh"

namespace cmlpl {

// ---------------------------------------------------------------- small kernels
__global__ void avgpool2_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t planes, int h, int w) {
  const int oh = h / 2, ow = w / 2;
  const int64_t total = planes * oh * ow;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t pl = i / (oh * ow); const int r = int(i - pl * oh * ow); const int oy = r / ow, ox = r - oy * ow;
    const float* s = x + pl * h * w + (2 * oy) * w + 2 * ox;
    // same association as ATen's avg_pool2d: sum of the window, then divide
    y[i] = (s[0] + s[1] + s[w] + s[w + 1]) / 4.0f;
  }
}
__global__ void avgpool2_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int64_t planes, int h, int w) {
  const int oh = h / 2, ow = w / 2;
  const int64_t total = planes * h * w;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t pl = i / (h * w); const int r = int(i - pl * h * w); const int y = r / w, xx = r - y * w;
    const int oy = y / 2, ox = xx / 2;
    dx[i] = (oy < oh && ox < ow) ? dy[pl * oh * ow + oy * ow + ox] / 4.0f : 0.f;
  }
}
__global__ void relu_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy, float* __restrict__ dx, int64_t n) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    dx[i] = y[i] > 0.f ? dy[i] : 0.f;
}
// out[n] = sum_m x[m,n]; one warp-column-group per 32 columns, block reduces over rows
__global__ void colsum_kernel(const float* __restrict__ x, float* __restrict__ out, int64_t m, int64_t n) {
  __shared__ float part[8][33];
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rgrp = threadIdx.x >> 5;
  float s = 0.f;
  if (col < n)
    for (int64_t r = rgrp; r < m; r += 8) s += x[r * n + col];
  part[rgrp][threadIdx.x & 31] = s;
  __syncthreads();
  if (rgrp == 0 && col < n) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += part[i][threadIdx.x];
    out[col] = t;
  }
}
// db[co] = sum_{b,pos} dy[b][co][pos]: grid (co, splits); a CTA sums the contiguous planes of every splits-th sample
// and adds its partial to db (zeroed by the caller) -- 64 channels alone cannot fill 148 SMs
__global__ void __launch_bounds__(256)
conv_bias_grad_kernel(const float* __restrict__ dy, float* __restrict__ db, int b, int co, int hw) {
  __shared__ float red[8];
  const int c = blockIdx.x;
  float s = 0.f;
  for (int bi = blockIdx.y; bi < b; bi += gridDim.y) {
    const float* p = dy + (int64_t(bi) * co + c) * hw;
    for (int i = threadIdx.x; i < hw; i += blockDim.x) s += __ldg(p + i);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(db + c, v);
  }
}

// one warp per row.  y = x / max(norm, eps); eps = 0 is models.py:88 (pow(1/2), no epsilon: a zero row gives NaN),
// eps > 0 is F.normalize.  norm stores the unclamped norm.
__global__ void l2norm_kernel(const float* __restrict__ x, float* __restrict__ y, float* __restrict__ norm, int64_t rows,
                              int64_t cols, float eps) {
  const int64_t row = blockIdx.x * int64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + row * cols;
  float s = 0.f;
  for (int64_t c = lane; c < cols; c += 32) s = fmaf(xr[c], xr[c], s);
  s = warp_sum(s);
  const float nr = sqrtf(s);
  if (lane == 0 && norm) norm[row] = nr;
  const float d = nr < eps ? eps : nr;
  for (int64_t c = lane; c < cols; c += 32) y[row * cols + c] = xr[c] / d;
}
// below eps the denominator is the constant eps (clamp_min passes no gradient): dx = dy / eps
__global__ void l2norm_bwd_kernel(const float* __restrict__ y, const float* __restrict__ norm, const float* __restrict__ dy,
                                  float* __restrict__ dx, int64_t rows, int64_t cols, float eps) {
  const int64_t row = blockIdx.x * int64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* yr = y + row * cols; const float* dr = dy + row * cols;
  float s = 0.f;
  for (int64_t c = lane; c < cols; c += 32) s = fmaf(dr[c], yr[c], s);
  s = warp_sum(s);
  const bool clamped = norm[row] < eps;
  if (clamped) s = 0.f;
  const float inv = 1.f / (clamped ? eps : norm[row]);
  for (int64_t c = lane; c < cols; c += 32) dx[row * cols + c] = (dr[c] - yr[c] * s) * inv;
}

static inline int ew_grid(int64_t n) {
  int64_t g = (n + 255) / 256;
  const int64_t cap = int64_t(sm_count()) * 16;
  return int(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace cmlpl

using namespace cmlpl;

extern "C" int cmlpl_sgemm_f32(int M, int N, int K, float alpha, const float* A, int64_t a_rs, int64_t a_cs,
                               const float* B, int64_t b_rs, int64_t b_cs, const float* bias, float beta,
                               float* C, int64_t c_rs, int64_t c_cs, int act, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(M >= 0 && N >= 0 && K >= 0, "sgemm: negative dims");
  // an operand without elements may be null (torch allocates nothing for it): K = 0 gives C = act(bias + beta*C)
  CMLPL_CHECK_ARG((A || int64_t(M) * K == 0) && (B || int64_t(K) * N == 0) && (C || int64_t(M) * N == 0),
                  "sgemm: null pointer");
  StridedA fa{A, a_rs, a_cs};
  StridedB fb{B, b_rs, b_cs};
  StridedC fc{C, c_rs, c_cs, bias, alpha, beta, act};
  return launch_gemm(M, N, K, 1, fa, fb, fc, static_cast<cudaStream_t>(stream), "sgemm");
}

extern "C" int cmlpl_conv2d_f32(const float* x, const float* wgt, const float* bias, const float* res, float* y,
                                int b, int ci, int co, int h, int w, int k, int act, int transpose_w,
                                cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && wgt && y, "conv2d: null pointer");
  CMLPL_CHECK_ARG(k == 1 || k == 3, "conv2d: kernel size %d unsupported (1 or 3)", k);
  CMLPL_CHECK_ARG(b > 0 && ci > 0 && co > 0 && h > 0 && w > 0, "conv2d: bad dims");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int M = b * h * w;
  if (!transpose_w) {
    ConvC fc{y, bias, res, co, h * w, act};
    if (k == 1) return launch_gemm(M, co, ci, 1, ConvA<1, false>{x, ci, h, w}, ConvB<1, false>{wgt, ci, co}, fc, s, "conv1x1");
    return launch_gemm(M, co, ci * 9, 1, ConvA<3, false>{x, ci, h, w}, ConvB<3, false>{wgt, ci, co}, fc, s, "conv3x3");
  }
  // data gradient: x is dL/dy [b,co,h,w]; y is dL/dx [b,ci,h,w]
  ConvC fc{y, bias, res, ci, h * w, act};
  if (k == 1) return launch_gemm(M, ci, co, 1, ConvA<1, true>{x, co, h, w}, ConvB<1, true>{wgt, ci, co}, fc, s, "conv1x1_dgrad");
  return launch_gemm(M, ci, co * 9, 1, ConvA<3, true>{x, co, h, w}, ConvB<3, true>{wgt, ci, co}, fc, s, "conv3x3_dgrad");
}

extern "C" int cmlpl_conv2d_wgrad_f32(const float* x, const float* dy, float* dw, float* db, int b, int ci, int co,
                                      int h, int w, int k, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && dy && dw, "conv2d_wgrad: null pointer");
  CMLPL_CHECK_ARG(k == 1 || k == 3, "conv2d_wgrad: kernel size %d unsupported", k);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int Kp = b * h * w;
  const int N = ci * k * k;
  CMLPL_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * size_t(co) * N, s));
  // enough K-splits to fill the machine
  const int tiles = ((N + TN - 1) / TN) * ((co + TM - 1) / TM);
  int splits = (2 * sm_count() + tiles - 1) / tiles;
  if (splits > (Kp + 255) / 256) splits = (Kp + 255) / 256;
  if (splits < 1) splits = 1;
  AtomicC fc{dw, N};
  int rc;
  if (k == 1) rc = launch_gemm(co, N, Kp, splits, WgradA{dy, co, h * w}, WgradB<1>{x, ci, h, w}, fc, s, "conv1x1_wgrad");
  else rc = launch_gemm(co, N, Kp, splits, WgradA{dy, co, h * w}, WgradB<3>{x, ci, h, w}, fc, s, "conv3x3_wgrad");
  if (rc != CMLPL_OK) return rc;
  if (db) {
    CMLPL_CUDA(cudaMemsetAsync(db, 0, sizeof(float) * size_t(co), s));
    conv_bias_grad_kernel<<<dim3(co, b < 32 ? b : 32), 256, 0, s>>>(dy, db, b, co, h * w);
    CMLPL_CHECK_LAUNCH("conv_bias_grad");
  }
  return rc;
}

extern "C" int cmlpl_avgpool2_f32(const float* x, float* y, int64_t planes, int h, int w, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && y && planes >= 0 && h >= 2 && w >= 2, "avgpool2: bad args");
  if (planes == 0) return CMLPL_OK;
  avgpool2_kernel<<<ew_grid(planes * (h / 2) * (w / 2)), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, planes, h, w);
  CMLPL_CHECK_LAUNCH("avgpool2");
  return CMLPL_OK;
}
extern "C" int cmlpl_avgpool2_bwd_f32(const float* dy, float* dx, int64_t planes, int h, int w, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(dy && dx && planes >= 0 && h >= 2 && w >= 2, "avgpool2_bwd: bad args");
  if (planes == 0) return CMLPL_OK;
  avgpool2_bwd_kernel<<<ew_grid(planes * h * w), 256, 0, static_cast<cudaStream_t>(stream)>>>(dy, dx, planes, h, w);
  CMLPL_CHECK_LAUNCH("avgpool2_bwd");
  return CMLPL_OK;
}
extern "C" int cmlpl_relu_bwd_f32(const float* y, const float* dy, float* dx, int64_t n, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(y && dy && dx && n >= 0, "relu_bwd: bad args");
  if (n == 0) return CMLPL_OK;
  relu_bwd_kernel<<<ew_grid(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(y, dy, dx, n);
  CMLPL_CHECK_LAUNCH("relu_bwd");
  return CMLPL_OK;
}
extern "C" int cmlpl_colsum_f32(const float* x, float* out, int64_t m, int64_t n, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && out && m >= 0 && n >= 0, "colsum: bad args");
  if (n == 0) return CMLPL_OK;
  colsum_kernel<<<int((n + 31) / 32), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, out, m, n);
  CMLPL_CHECK_LAUNCH("colsum");
  return CMLPL_OK;
}
extern "C" int cmlpl_l2norm_f32(const float* x, float* y, float* norm, int64_t rows, int64_t cols, float eps,
                                cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && y && rows >= 0 && cols > 0 && eps >= 0.f, "l2norm: bad args");
  if (rows == 0) return CMLPL_OK;
  l2norm_kernel<<<int((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, norm, rows, cols, eps);
  CMLPL_CHECK_LAUNCH("l2norm");
  return CMLPL_OK;
}
extern "C" int cmlpl_l2norm_bwd_f32(const float* y, const float* norm, const float* dy, float* dx, int64_t rows,
                                    int64_t cols, float eps, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(y && norm && dy && dx && rows >= 0 && cols > 0 && eps >= 0.f, "l2norm_bwd: bad args");
  if (rows == 0) return CMLPL_OK;
  l2norm_bwd_kernel<<<int((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(y, norm, dy, dx, rows, cols, eps);
  CMLPL_CHECK_LAUNCH("l2norm_bwd");
  return CMLPL_OK;
}
