// Fused training step, forward trunk part 1: patch gather + noise + conv0 for every sample of both BaseNet2 peers
// (train.py:157-184 input assembly, tools/models.py:132).  One CTA per sample:
//   loaders   the sample's 20x20x60 window is gathered from the channels-last PCA cube through the MirrowCut index
//             map (tools/hyper_tools.py:35-55, 226-243), `+ noise * sigma` is applied (injected N(0,1) tensor, or the
//             device Philox stream), rounded to fp16 and laid down in shared memory as chunk planes
//             [8 chunks][400 positions][8 channels] -- the UMMA K-major A operand -- and in HBM (x16, the B operand
//             of conv0's weight gradient later)
//   MMA       16 tcgen05.mma (4 position tiles x 4 K-steps, M=128 N=64 K=16) against W0 (fp32 -> fp16 in the prologue)
//   epilogue  TMEM -> +bias -> fp16 -> a0 chunk planes in HBM (input of conv1 and B operand of conv1's weight gradient)
// The patch is never materialised in fp32 and the noise never exists as a tensor in the Philox mode.
// W = 11 (ExtractPatches_for_base, hyper_tools.py:300-317: rows r-5 .. r+5, the same mirror) has 121 positions: one
// position tile, 4 MMAs.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "train_common.cuh"
#include "train_kernels.cuh"

namespace cmlpl {

template <int W>
struct C0Cfg {
  using G = TrainGeom<W>;
  static constexpr int CH = G::TPos * 16;        // bytes per chunk plane (6400 at W = 20)
  static constexpr int NT = (G::TPos + 127) / 128;   // 128-row position tiles (4 at W = 20, 1 at W = 11)
  static constexpr int S_X = 0;
  static constexpr int S_W = 8 * CH + 2048;      // the last tile reads rows up to NT*128-1 of plane 7: slack
  static constexpr int S_BIAS = S_W + 8 * 64 * 16;
  static constexpr int S_BAR = S_BIAS + 256;
  static constexpr int S_TMEM = S_BAR + 16;
  static constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
  static_assert((NT * 128 - G::TPos) * 16 <= 2048, "tile slack");
};
constexpr int kC0Threads = 256;

template <int W>
__global__ void __launch_bounds__(kC0Threads)
train_conv0_kernel(Conv0Args a) {
  using G = TrainGeom<W>;
  using Cfg = C0Cfg<W>;
  constexpr int CH = Cfg::CH, S_X = Cfg::S_X, S_W = Cfg::S_W, S_BIAS = Cfg::S_BIAS, S_BAR = Cfg::S_BAR,
                S_TMEM = Cfg::S_TMEM, THREADS = kC0Threads;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar = sbase + S_BAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);
  const int s = blockIdx.x;                    // sample: net e = s / nb, row i = s % nb
  const int e = s / a.nb, row = s - e * a.nb;

  if (tid == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(sbase + S_TMEM, 256);
  // ---- W0 [64 co][60 ci] fp32 -> fp16 K-major B operand [8 kchunks][64 co][8 ci], bias, slack
  {
    const float* w0 = a.w0[e];
    __half* sw = reinterpret_cast<__half*>(smem + S_W);
    for (int i = tid; i < 64 * 64; i += THREADS) {
      const int co = i >> 6, ci = i & 63;
      sw[((ci >> 3) * 64 + co) * 8 + (ci & 7)] = __float2half_rn(ci < 60 ? __ldg(w0 + co * 60 + ci) : 0.f);
    }
    if (tid < 64) reinterpret_cast<float*>(smem + S_BIAS)[tid] = __ldg(a.b0[e] + tid);
    for (int i = tid; i < 2048 / 16; i += THREADS) reinterpret_cast<uint4*>(smem + 8 * CH)[i] = make_uint4(0, 0, 0, 0);
  }
  if (s == 0) {
    if (tid < 12) a.hist[tid] = 0.f;
    if (tid == 12) a.prm_rw->grad_amax = 0.f;
  }
  // ---- this CTA's slice of the 3x3 weights -> fp16 packs: forward layout [3 dx][8 kchunks][192 rows = (2-dy)*64 + co][8 ci]
  //      (conv_pair_issue.cuh) and backward layout [tap][ci chunk][co][8 ci] (train_bwd_sm100.cu)
  for (int i = s * THREADS + tid; i < 4 * 36864; i += int(gridDim.x) * THREADS) {
    const int t4 = i / 36864, j = i - t4 * 36864;                 // t4 = net * 2 + conv
    const int co = j / 576, r = j - co * 576, ci = r / 9, t = r - ci * 9, dy = t / 3, dx = t - dy * 3;
    const __half h = __float2half_rn(__ldg(a.w3[t4 >> 1][t4 & 1] + j));
    __half* base = reinterpret_cast<__half*>(a.wpack + size_t(t4) * 2 * kWPackBytes);
    base[((dx * 8 + (ci >> 3)) * 192 + (2 - dy) * 64 + co) * 8 + (ci & 7)] = h;
    base[kWPackBytes / 2 + ((t * 8 + (ci >> 3)) * 64 + co) * 8 + (ci & 7)] = h;
  }
  // ---- spectral input: gather + noise (fp32, consumed by the feat_spe GEMM)
  {
    const float sigma = a.prm->noise_scale;
    const int64_t srow = a.cube ? (a.spec_row ? a.spec_row[row] : a.pix[row]) : s;
    const float* src = a.spectra + srow * a.bands;
    const float* nz = a.spec_noise ? a.spec_noise + int64_t(s) * a.bands : nullptr;
    const bool draw = a.cube && !nz && sigma != 0.f;
    float* dst = a.ynoisy + int64_t(s) * a.bands;
    for (int j4 = tid; j4 * 4 < a.bands; j4 += THREADS) {
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      if (draw) {
        const uint2 ctr = spec_noise_counter(s, j4);
        z = philox_normal4(a.prm->seed, a.prm->offset, ctr.x, ctr.y);
      }
      const float zz[4] = {z.x, z.y, z.z, z.w};
      for (int j = 0; j < 4 && j4 * 4 + j < a.bands; ++j) {
        const int b = j4 * 4 + j;
        const float n = nz ? __ldg(nz + b) : zz[j];
        dst[b] = (a.cube && (nz || draw)) ? __fadd_rn(__ldg(src + b), __fmul_rn(n, sigma)) : __ldg(src + b);
      }
    }
  }
  // ---- gather + noise -> fp16 planes (shared memory and HBM)
  {
    const float sigma = a.prm->noise_scale;
    const unsigned long long seed = a.prm->seed, offset = a.prm->offset;
    int r = 0, c = 0;
    if (a.cube) { const int64_t pix = a.pix[row]; r = int(pix / a.cols); c = int(pix - int64_t(r) * a.cols); }
    const float* nz = a.noise ? a.noise + int64_t(s) * 60 * G::TPos : nullptr;
    unsigned char* xg = reinterpret_cast<unsigned char*>(a.x16) + int64_t(s) * G::ActBytes;
    const bool draw = a.cube && !nz && sigma != 0.f;
    // 6400 items (16 channel quads x 400 positions) / 256 threads = 25 per thread, in batches of 5 with all global
    // loads of a batch issued before any is consumed
    constexpr int U = 5;
#pragma unroll 1
    for (int i0 = tid; i0 < 16 * G::TPos; i0 += THREADS * U) {
      float4 b[U], z[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * THREADS;
        const int q = i / G::TPos, p = i - q * G::TPos;        // q: group of 4 channels, p: window position
        b[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        z[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < 15 * G::TPos) {
          if (nz) {
            z[u].x = __ldg(nz + (4 * q + 0) * G::TPos + p); z[u].y = __ldg(nz + (4 * q + 1) * G::TPos + p);
            z[u].z = __ldg(nz + (4 * q + 2) * G::TPos + p); z[u].w = __ldg(nz + (4 * q + 3) * G::TPos + p);
          }
          if (a.cube) {
            const int y = p / W, x = p - y * W;
            const int sr = mirror_index(r - W / 2 + y, a.scene_rows), sc = mirror_index(c - W / 2 + x, a.cols);
            b[u] = __ldg(reinterpret_cast<const float4*>(a.cube + (int64_t(sr) * a.cols + sc) * 60) + q);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * THREADS;
        if (i >= 16 * G::TPos) continue;
        const int q = i / G::TPos, p = i - q * G::TPos;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < 15) {
          if (draw) z[u] = philox_normal4(seed, offset, PHILOX_PATCH, uint32_t(s) * 6000u + uint32_t(i));
          if (a.cube) {
            // x + randn * noise: mul then add, two roundings like torch (train.py:157)
            v.x = __fadd_rn(b[u].x, __fmul_rn(z[u].x, sigma)); v.y = __fadd_rn(b[u].y, __fmul_rn(z[u].y, sigma));
            v.z = __fadd_rn(b[u].z, __fmul_rn(z[u].z, sigma)); v.w = __fadd_rn(b[u].w, __fmul_rn(z[u].w, sigma));
          } else {
            v = z[u];                                       // the caller passed the assembled patches
          }
        }
        const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t*>(&h0); pk.y = *reinterpret_cast<const uint32_t*>(&h1);
        const int off = (q >> 1) * CH + p * 16 + (q & 1) * 8;
        *reinterpret_cast<uint2*>(smem + S_X + off) = pk;
        *reinterpret_cast<uint2*>(xg + off) = pk;
      }
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (tid == 0) {
    constexpr uint32_t kI = make_idesc_f16(128, 64);
#pragma unroll
    for (int t = 0; t < Cfg::NT; ++t)
#pragma unroll
      for (int ks = 0; ks < 4; ++ks)
        umma_f16(tmem + t * 64, make_desc(sbase + S_X + t * 2048 + ks * 2 * CH, CH, 128),
                 make_desc(sbase + S_W + ks * 2 * 1024, 1024, 128), kI, ks);
    umma_commit(bar);
  }
  mbar_wait(bar, 0, 40);
  tc_fence_after();
  {
    const int q4 = warp & 3, chalf = warp >> 2;
    const float* bias = reinterpret_cast<const float*>(smem + S_BIAS) + chalf * 32;
    unsigned char* ag = reinterpret_cast<unsigned char*>(a.a0) + int64_t(s) * G::ActBytes;
#pragma unroll 1
    for (int t = 0; t < Cfg::NT; ++t) {
      const int p = t * 128 + q4 * 32 + lane;
      const uint32_t taddr = tmem + (uint32_t(q4 * 32) << 16) + t * 64 + chalf * 32;
      float v[32];
      tmem_ld16(taddr, v);
      tmem_ld16(taddr + 16, v + 16);
      tmem_ld_wait();
      if (p < G::TPos) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          __half2 h[4];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            h[j] = __floats2half2_rn(v[k * 8 + 2 * j] + bias[k * 8 + 2 * j], v[k * 8 + 2 * j + 1] + bias[k * 8 + 2 * j + 1]);
          *reinterpret_cast<uint4*>(ag + (chalf * 4 + k) * CH + p * 16) = *reinterpret_cast<uint4*>(h);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem, 256); }
}

int launch_train_conv0(const Conv0Args& a, int w, cudaStream_t st) {
  if (w == 11) {
    auto kern = train_conv0_kernel<11>;
    CMLPL_MAX_DYN_SMEM(kern, C0Cfg<11>::SMEM);
    kern<<<2 * a.nb, kC0Threads, C0Cfg<11>::SMEM, st>>>(a);
  } else {
    auto kern = train_conv0_kernel<20>;
    CMLPL_MAX_DYN_SMEM(kern, C0Cfg<20>::SMEM);
    kern<<<2 * a.nb, kC0Threads, C0Cfg<20>::SMEM, st>>>(a);
  }
  CMLPL_CHECK_LAUNCH("train_conv0");
  return CMLPL_OK;
}

}  // namespace cmlpl
