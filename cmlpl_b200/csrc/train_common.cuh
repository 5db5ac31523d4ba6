// Shared by the fused training-step kernels (train_fwd_sm100.cu, train_bwd_sm100.cu, train_head.cu, train_step.cu):
// workspace layout, per-sample activation layouts, the device Philox stream and the gradient scale.
#pragma once
#include "common.cuh"

namespace cmlpl {

// ---- per-sample activation layouts in the workspace (fp16, "chunk-planar": [8 chunks of 8 channels][positions][8])
// A chunk plane row of one position is 16 bytes, so the planes are at the same time
//   * the UMMA no-swizzle K-major operand (K = channels: LBO = plane stride, SBO = 128 B) of the forward / data-gradient
//     convolutions, and
//   * the UMMA no-swizzle MN-major operand (K = positions: LBO = 128 B, SBO = plane stride) of the weight gradients
// (verified on hardware by scripts/micro/mn_major_probe.cu).
constexpr int kTW = 20, kTPos = kTW * kTW, kTPos2 = (kTW / 2) * (kTW / 2);
constexpr int kActBytes = 8 * kTPos * 16;     // x16 / a0 / dz1 / da0 of one sample: 51 200 B
constexpr int kAct2Bytes = 8 * kTPos2 * 16;   // p1 of one sample: 12 800 B
constexpr int kHid = 1024;
constexpr int kCatDim = 64 * 25 + kHid;       // 2624 (tools/models.py:127)
constexpr int kConvFeat = 64 * 25;
constexpr int kWPackBytes = 9 * 64 * 64 * 2;  // one 3x3 conv's weights in fp16: 73 728 B

// Per-window geometry of the trunk kernels.  W = 20 is the reference's BaseNet2 (the constants above, which also size
// the workspace); W = 11 is the odd window of ExtractPatches_for_base (hyper_tools.py:300-317), whose 2x2 average pools
// floor 11 -> 5 -> 2 and drop the last row / column of each map.  A W = 11 step runs in the W = 20 workspace at the
// same region offsets, each region packed densely at the per-sample strides below (include/cmlpl.h).
template <int W>
struct TrainGeom {
  static constexpr int TPos = W * W;                     // conv0 / conv1 positions
  static constexpr int H2 = W / 2;                       // conv2 map
  static constexpr int TPos2 = H2 * H2;
  static constexpr int NP2 = H2 / 2;                     // pooled conv2 map
  static constexpr int ActBytes = 8 * TPos * 16;         // x16 / a0 / dz1 / da0 of one sample
  static constexpr int Act2Bytes = 8 * TPos2 * 16;       // p1 of one sample
  static constexpr int ConvFeat = 64 * NP2 * NP2;        // flattened pooled conv2 output (tools/models.py:141)
  static constexpr int CatDim = ConvFeat + kHid;         // classifier input
};
static_assert(TrainGeom<20>::CatDim == kCatDim && TrainGeom<20>::ActBytes == kActBytes, "W = 20 geometry");
static_assert(TrainGeom<11>::CatDim == 1280 && TrainGeom<11>::ActBytes <= kActBytes, "W = 11 fits the W = 20 workspace");

struct TrainWs {
  size_t x16, a0, p1, m1, m2, cat, dmask, ynoisy, norm, dlogits, dfeat, dcat, dhp, dz1, da0, S, G, dG, probs_orig, wpack, gstage, total;
};
__host__ __device__ inline TrainWs train_ws_layout(int bs, int btu, int B, int C, int queue) {
  TrainWs L;
  const size_t ns = size_t(2) * (bs + btu);
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at = o; o = align256(o + bytes); return at; };
  L.x16 = take(ns * kActBytes);
  L.a0 = take(ns * kActBytes);
  L.p1 = take(ns * kAct2Bytes);
  L.m1 = take(ns * kTPos * 8);
  L.m2 = take(ns * kTPos2 * 8);
  L.cat = take(ns * kCatDim * 4);
  L.dmask = take(ns * kCatDim * 4);
  L.ynoisy = take(ns * size_t(B) * 4);
  L.norm = take(ns * 4);
  L.dlogits = take(ns * size_t(C) * 4);
  L.dfeat = take(size_t(2) * btu * kHid * 4);
  L.dcat = take(ns * kCatDim * 4);
  L.dhp = take(ns * kHid * 4);
  L.dz1 = take(ns * kActBytes);
  L.da0 = take(ns * kActBytes);
  L.S = take(size_t(2) * (2 * ((queue + 127) / 128)) * btu * 33 * 4);   // streaming bank-smoothing partials
  L.G = take(size_t(btu) * btu * 4);
  L.dG = take(size_t(btu) * btu * 4);
  L.probs_orig = take(size_t(2) * btu * C * 4);
  L.wpack = take(size_t(8) * kWPackBytes);     // fp16 3x3 weights [net][conv1|conv2][forward | backward layout]
  L.gstage = take(size_t(4) * 36864 * 4);      // fp32 3x3 weight gradients [net][conv1|conv2][tap][co][ci] (vector reds)
  L.total = o;
  return L;
}

// ---- Philox4x32-10 (Salmon et al., SC'11), counter-based: every consumer derives its counter from the element it
// produces, so the stream does not depend on the launch geometry.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
  }
  return c;
}
// four N(0,1) draws for (stream, index) of the step whose params hold (seed, offset)
__device__ __forceinline__ float4 philox_normal4(unsigned long long seed, unsigned long long offset, uint32_t stream,
                                                 uint32_t index) {
  const uint4 r = philox4x32_10(make_uint4(index, stream, uint32_t(offset), uint32_t(offset >> 32)),
                                make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
  // Box-Muller on (0,1] uniforms
  const float u0 = (float(r.x >> 8) + 1.0f) * (1.0f / 16777216.0f), u1 = float(r.y >> 8) * (1.0f / 16777216.0f);
  const float u2 = (float(r.z >> 8) + 1.0f) * (1.0f / 16777216.0f), u3 = float(r.w >> 8) * (1.0f / 16777216.0f);
  const float ra = sqrtf(-2.0f * __logf(u0)), rb = sqrtf(-2.0f * __logf(u2));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  return make_float4(ra * c0, ra * s0, rb * c1, rb * s1);
}
__device__ __forceinline__ uint4 philox_uniform4(unsigned long long seed, unsigned long long offset, uint32_t stream,
                                                 uint32_t index) {
  return philox4x32_10(make_uint4(index, stream, uint32_t(offset), uint32_t(offset >> 32)),
                       make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
}
enum { PHILOX_PATCH = 1, PHILOX_SPEC = 2, PHILOX_DROP = 3, PHILOX_SPEC_HI = 4 };

// Counter of the spectral noise of band quad j4 of sample s (four bands per draw).  Quads 0..63 keep the original
// (PHILOX_SPEC, s*64 + j4), so every run up to 256 bands draws what it always drew; quad group g = j4 / 64 >= 1 (bands
// 256..511) draws from its own stream PHILOX_SPEC_HI + g - 1 at s*64 + j4 % 64, disjoint from every other sample's
// draws.  Valid up to 512 bands, the bound cmlpl_train_step checks.
__device__ __forceinline__ uint2 spec_noise_counter(int s, int j4) {
  const uint32_t g = uint32_t(j4) >> 6;
  return make_uint2(g == 0 ? uint32_t(PHILOX_SPEC) : uint32_t(PHILOX_SPEC_HI) + g - 1u, uint32_t(s) * 64u + (uint32_t(j4) & 63u));
}

// power-of-two scale that puts gradients whose largest magnitude is `amax` near 2^12 in fp16 (max 65504, smallest
// normal 6.1e-5): the data-gradient sums may grow by 2^4 and values 2^-26 below the maximum are still normal numbers
__device__ __forceinline__ float grad_scale(float amax) {
  if (!(amax > 0.f) || !isfinite(amax)) return 1.f;
  int e;
  frexpf(amax, &e);                       // amax = m * 2^e, m in [0.5, 1)
  return ldexpf(1.f, 12 - e);
}

}  // namespace cmlpl
