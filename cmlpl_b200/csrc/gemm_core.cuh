// Tiled fp32 CUDA-core GEMM core shared by fp32_ops.cu and scene_infer.cu.
// 64x64x16 tiles, 256 threads, 4x4 register micro-tiles, operand access through functors
// (strided GEMM, implicit-GEMM convolution forward / dgrad / split-K wgrad).
#pragma once
#include "common.cuh"

namespace cmlpl {

constexpr int TM = 64, TN = 64, TK = 16;

// ---------------------------------------------------------------- operand functors
struct StridedA {
  const float* p; int64_t rs, cs;
  __device__ __forceinline__ void prep(int) {}
  __device__ __forceinline__ float at(int m, int k) const { return __ldg(p + m * rs + k * cs); }
};
// rows of the raw cube (uint16 / float32, row stride rs), z-scored on load: A(m,k) = (x[m][k] - mu[k]) * inv_sigma[k];
// valid (u8 per row, or nullptr): a no-data row stands in as its band means, a zero row
template <typename T>
struct RawZA {
  const T* p; int64_t rs; const float* mu; const float* inv_sigma; const uint8_t* valid;
  bool ok_;
  __device__ __forceinline__ void prep(int m) { ok_ = !valid || valid[m]; }
  __device__ __forceinline__ float at(int m, int k) const {
    return ok_ ? (float(__ldg(p + m * rs + k)) - __ldg(mu + k)) * __ldg(inv_sigma + k) : 0.f;
  }
};
// the same from a band-major raw slab (BIL / BSQ): pixel m0 + m of the band is row (m0 + m) / cols, column
// (m0 + m) % cols of the band's rows at p; the k order and the validity rows (valid[m0 + m]) are RawZA's
template <typename T>
struct RawBandZA {
  const T* p; BandMajor bm; int64_t m0; const float* mu; const float* inv_sigma; const uint8_t* valid;
  int64_t off_; bool ok_;
  __device__ __forceinline__ void prep(int m) {
    const int64_t q = m0 + m, r = q / bm.cols;
    off_ = r * bm.rs + (q - r * bm.cols);
    ok_ = !valid || valid[q];
  }
  __device__ __forceinline__ float at(int, int k) const {
    return ok_ ? (float(__ldg(p + off_ + k * bm.bs)) - __ldg(mu + k)) * __ldg(inv_sigma + k) : 0.f;
  }
};
struct StridedB {  // B[k][n]
  const float* p; int64_t rs, cs;
  __device__ __forceinline__ float at(int n, int k) const { return __ldg(p + k * rs + n * cs); }
};

// implicit GEMM A operand for a kxk "same" convolution in NCHW.
//   forward:  A(m,kk) = x[b][ci][y+ky-p][x+kx-p],  kk = (ci*k+ky)*k+kx
//   dgrad  :  A(m,kk) = dy[b][co][y-ky+p][x-kx+p], kk = (co*k+ky)*k+kx
template <int KS, bool DGRAD>
struct ConvA {
  const float* x; int ch, h, w;   // ch = channels of the tensor being read
  int b_, y_, x_; const float* base_;
  __device__ __forceinline__ void prep(int m) {
    const int hw = h * w;
    b_ = m / hw; const int r = m - b_ * hw; y_ = r / w; x_ = r - y_ * w;
    base_ = x + int64_t(b_) * ch * hw;
  }
  __device__ __forceinline__ float at(int, int kk) const {
    const int c = kk / (KS * KS); const int t = kk - c * (KS * KS);
    const int ky = t / KS, kx = t - ky * KS;
    const int p = KS / 2;
    const int yy = DGRAD ? y_ - ky + p : y_ + ky - p;
    const int xx = DGRAD ? x_ - kx + p : x_ + kx - p;
    if (yy < 0 || yy >= h || xx < 0 || xx >= w) return 0.f;
    return __ldg(base_ + (int64_t(c) * h + yy) * w + xx);
  }
};
// B operand: forward B(n=co,kk) = wgt[co][kk];  dgrad B(n=ci,kk=(co,ky,kx)) = wgt[co][ci][ky][kx]
template <int KS, bool DGRAD>
struct ConvB {
  const float* wgt; int ci, co;
  __device__ __forceinline__ float at(int n, int kk) const {
    if (!DGRAD) return __ldg(wgt + int64_t(n) * ci * KS * KS + kk);
    const int c = kk / (KS * KS); const int t = kk - c * (KS * KS);
    return __ldg(wgt + (int64_t(c) * ci + n) * KS * KS + t);
  }
};
// wgrad: dW[co][kk] = sum_m dy[m,co] * xcol[m,kk];  GEMM M'=co, N'=ci*k*k, K'=b*h*w
struct WgradA {  // A(m'=co, k'=pixel)
  const float* dy; int co, hw;
  __device__ __forceinline__ void prep(int) {}
  __device__ __forceinline__ float at(int m, int kp) const {
    const int b = kp / hw, r = kp - b * hw;
    return __ldg(dy + (int64_t(b) * co + m) * hw + r);
  }
};
template <int KS>
struct WgradB {  // B(n'=(ci,ky,kx), k'=pixel)
  const float* x; int ci, h, w;
  __device__ __forceinline__ float at(int n, int kp) const {
    const int hw = h * w;
    const int b = kp / hw, r = kp - b * hw; const int y = r / w, xx0 = r - y * w;
    const int c = n / (KS * KS); const int t = n - c * (KS * KS);
    const int ky = t / KS, kx = t - ky * KS; const int p = KS / 2;
    const int yy = y + ky - p, xx = xx0 + kx - p;
    if (yy < 0 || yy >= h || xx < 0 || xx >= w) return 0.f;
    return __ldg(x + ((int64_t(b) * ci + c) * h + yy) * w + xx);
  }
};

// ---------------------------------------------------------------- epilogues
struct StridedC {
  float* c; int64_t rs, cs; const float* bias; float alpha, beta; int act;
  __device__ __forceinline__ void store(int m, int n, float v) const {
    float* d = c + m * rs + n * cs;
    v *= alpha;
    if (bias) v += __ldg(bias + n);
    if (beta != 0.f) v += beta * *d;
    if (act == 1) v = fmaxf(v, 0.f);
    *d = v;
  }
};
struct ConvC {  // y[b][n][pos]
  float* y; const float* bias; const float* res; int cout, hw; int act;
  __device__ __forceinline__ void store(int m, int n, float v) const {
    const int b = m / hw, r = m - b * hw;
    const int64_t o = (int64_t(b) * cout + n) * hw + r;
    if (bias) v += __ldg(bias + n);
    if (res) v += __ldg(res + o);
    if (act == 1) v = fmaxf(v, 0.f);
    y[o] = v;
  }
};
struct OnesB { __device__ __forceinline__ float at(int, int) const { return 1.f; } };
struct AtomicC {  // split-K accumulation
  float* c; int64_t rs;
  __device__ __forceinline__ void store(int m, int n, float v) const { atomicAdd(c + m * rs + n, v); }
};

// ---------------------------------------------------------------- the GEMM core
// grid: (ceil(N/TN), ceil(M/TM), splits).  K range of split z: [z*kper, min(K,(z+1)*kper)).
template <class FA, class FB, class FC>
__global__ void __launch_bounds__(256)
gemm_tile_kernel(int M, int N, int K, int kper, FA fa, FB fb, FC fc) {
  __shared__ float As[2][TK][TM + 4];
  __shared__ float Bs[2][TK][TN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  const int kbeg = blockIdx.z * kper, kend = min(K, kbeg + kper);
  // loader mapping: thread loads rows (tid & 63) for k = (tid >> 6) + 4*j, j<4
  const int lrow = tid & 63, lk = tid >> 6;
  const int am = m0 + lrow, bn = n0 + lrow;
  const bool am_ok = am < M, bn_ok = bn < N;
  if (am_ok) fa.prep(am);
  // compute mapping: 16x16 threads, 4x4 outputs each
  const int tx = tid & 15, ty = tid >> 4;
  // accumulators as packed fp32 pairs along n: fma.rn.f32x2 (FFMA2) = two fp32 FMAs per issue slot, each rounded like fmaf
  unsigned long long acc2[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc2[i][0] = acc2[i][1] = 0ull;

  float ra[4], rb[4];
  auto gload = [&](int k0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + lk + 4 * j;
      ra[j] = (am_ok && k < kend) ? fa.at(am, k) : 0.f;
      rb[j] = (bn_ok && k < kend) ? fb.at(bn, k) : 0.f;
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      As[buf][lk + 4 * j][lrow] = ra[j];
      Bs[buf][lk + 4 * j][lrow] = rb[j];
    }
  };
  if (kbeg < kend) {
    gload(kbeg);
    sstore(0);
    __syncthreads();
    int buf = 0;
    for (int k0 = kbeg; k0 < kend; k0 += TK) {
      const bool more = k0 + TK < kend;
      if (more) gload(k0 + TK);
#pragma unroll
      for (int k = 0; k < TK; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
        const ulonglong2 b = *reinterpret_cast<const ulonglong2*>(&Bs[buf][k][tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          unsigned long long aa;
          asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(av[i]));
          asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][0]) : "l"(aa), "l"(b.x));
          asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][1]) : "l"(aa), "l"(b.y));
        }
      }
      if (more) {
        sstore(buf ^ 1);
        __syncthreads();
        buf ^= 1;
      }
    }
  }
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) asm("mov.b64 {%0, %1}, %2;" : "=f"(acc[i][2 * j]), "=f"(acc[i][2 * j + 1]) : "l"(acc2[i][j]));
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) fc.store(m, n, acc[i][j]);
    }
  }
}

template <class FA, class FB, class FC>
static int launch_gemm(int M, int N, int K, int splits, FA fa, FB fb, FC fc, cudaStream_t s, const char* name) {
  if (M <= 0 || N <= 0) return CMLPL_OK;
  int kper = (K + splits - 1) / splits;
  kper = (kper + TK - 1) / TK * TK;
  if (kper <= 0) kper = TK;
  splits = K > 0 ? (K + kper - 1) / kper : 1;
  dim3 grid((N + TN - 1) / TN, (M + TM - 1) / TM, splits);
  gemm_tile_kernel<<<grid, 256, 0, s>>>(M, N, K, kper, fa, fb, fc);
  CMLPL_CHECK_LAUNCH(name);
  return CMLPL_OK;
}


}  // namespace cmlpl
