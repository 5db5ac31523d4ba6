// Issue helper of the per-pixel tcgen05 conv kernel (patch_cnn_sm100.cu: conv1 and conv2, inference and training).
#pragma once
#include "sm100_ptx.cuh"

namespace cmlpl {

// One PAIR of 128-row accumulator tiles (even-row tile at d_tmem, odd-row tile at d_tmem + 64) of a
// 3x3 convolution.  tcgen05.mma costs ~64 cycles whether N is 64 or 128 (measured,
// scripts/micro/mma_rate.cu), so taps are grouped by the A operand they read:
//   A = (even plane, row i  , dx): feeds dy=1 of the even tile AND dy=0 of the odd tile -> one N=128 MMA
//   A = (odd  plane, row i+1, dx): feeds dy=2 of the even tile AND dy=1 of the odd tile -> one N=128 MMA
//   A = (odd  plane, row i  , dx): dy=0 of the even tile only (N=64)
//   A = (even plane, row i+1, dx): dy=2 of the odd tile only  (N=64)
// (row tables: even outputs y=2i read rows 2i-1, 2i, 2i+1 = odd-plane row i, even-plane row i,
//  odd-plane row i+1; odd outputs y=2i+1 read even-plane row i, odd-plane row i+1, even-plane row i+1.)
// The weights are packed per dx as 192 rows [W(dy=2); W(dy=1); W(dy=0)] x K, so [W2;W1] is rows 0..127,
// [W1;W0] rows 64..191 and the singles are rows 0..63 / 128..191 of the same block: 48 MMAs per pair
// instead of 72, all descriptor offsets immediates.
//   PWX padded row width (entries), CHX bytes between K-chunks, PLANEX bytes per parity plane
//   a_lo low descriptor word of (even plane, entry 1 + first output row of the tile)
//   b_lo low descriptor word of the weight block of dx = 0 (LBO = 192 rows * 16 B)
constexpr int kWRows = 192, kWLbo = kWRows * 16, kWDxBytes = 8 * kWLbo;
template <int PWX, int CHX, int PLANEX>
__device__ __forceinline__ void issue_conv_pair(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo) {
  constexpr uint64_t kHi = (uint64_t(128 >> 4) | (uint64_t(1) << 14)) << 32;   // SBO = 128 B, version 1
  constexpr uint32_t kI128 = make_idesc_f16(128, 128), kI64 = make_idesc_f16(128, 64);
#pragma unroll
  for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const int col = (dx - 1) * 16 + ks * 2 * CHX;
      const uint64_t aE0 = kHi | uint64_t(a_lo + uint32_t(col / 16));
      const uint64_t aE1 = kHi | uint64_t(a_lo + uint32_t((PWX * 16 + col) / 16));
      const uint64_t aO0 = kHi | uint64_t(a_lo + uint32_t((PLANEX + col) / 16));
      const uint64_t aO1 = kHi | uint64_t(a_lo + uint32_t((PLANEX + PWX * 16 + col) / 16));
      const uint32_t b = b_lo + uint32_t((dx * kWDxBytes + ks * 2 * kWLbo) / 16);
      umma_f16(d_tmem, aE0, kHi | uint64_t(b + 64), kI128, (dx | ks) != 0 ? 1u : 0u);   // [W1;W0] -> even|odd
      umma_f16(d_tmem, aO1, kHi | uint64_t(b), kI128, 1u);                               // [W2;W1] -> even|odd
      umma_f16(d_tmem, aO0, kHi | uint64_t(b + 128), kI64, 1u);                          // W0 -> even
      umma_f16(d_tmem + 64, aE1, kHi | uint64_t(b), kI64, 1u);                           // W2 -> odd
    }
  }
}

}  // namespace cmlpl
