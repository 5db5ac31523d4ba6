// conv0 of the scene path on tcgen05: F0 = W . x + b once per PADDED scene position (tools/models.py:102,132 applied to
// the mirror-padded cube, hyper_tools.py:35-55) -> chunk-planar fp16 map [8 chunks][prow_n][pcol_n][8].
// x is either the 60-channel PCA cube (float) or the RAW cube (uint16 / float, K = B bands) with the PCA projection and
// both z-scores folded into W (SURVEY 8-f1): F0 = Wf . (x - mu) + bf.
//
// Persistent CTAs over tiles of 128 consecutive padded positions.  The 256 worker threads read a tile's source pixels
// (mirrored index map, K contiguous values per pixel: fully coalesced), round to fp16 and write the UMMA K-major tile
// [K/8 chunks][128 positions][8] straight into shared memory (two stages); one thread issues K/16 tcgen05.mma
// (M=128, N=64) per tile into one of two TMEM slots; the same workers drain the previous tile (+bias -> fp16 -> F0,
// 16-byte stores coalesced along positions) while their loads for the next tile are in flight.  A band-major raw slab
// (BIL / BSQ) has its own loader: a thread owns one position and reads 8 bands per K-chunk, coalesced along columns.
// Replaces the CUDA-core conv0_tiled_kernel of round 1 (L1-wavefront bound on the strided pixel rows).
// valid (raw cube only; u8 [slab_rows * cols] over the slab's pixels, or nullptr): a position whose mirrored source pixel
// is no-data gets the z-scored operand 0 (hi and lo), i.e. the pixel stands in as its band means and F0 there is the
// folded bias exactly.  The mask byte is read once per tile position; the sample loads keep their order.
#include "common.cuh"
#include "sm100_ptx.cuh"

namespace cmlpl {

namespace c0s {
constexpr int kWorkers = 256, kThreads = kWorkers + 32;
enum { X_FULL0 = 0, X_EMPTY0 = 2, D_FULL0 = 4, D_EMPTY0 = 6 };
}  // namespace c0s

// kSplit (raw cube): both operands are split into fp16 hi + lo parts and every K-step issues hi.hi + hi.lo + lo.hi
// (~2^-21 relative error).  The folded PCA projection is ill-conditioned -- its noise components are differences of
// band values ~10x larger than the result -- so single fp16 operands miss the 1e-3 logit bar (measured at B = 200).
// kBM (raw cube, kSplit only): the slab is band-major (BIL / BSQ, addressed through bm) instead of pixel-major.  The
// kernels read threadIdx.x and pass it in as tid, so the range their launch bounds give it still holds in the body.
template <typename T, bool kVec4, bool kSplit, bool kBM>
__device__ __forceinline__ void
conv0_tc_body(const T* __restrict__ in, int K, int KP, int nstage, int scene_rows, int cols, int slab_row0, int w, int band_row0,
              int prow_n, int pcol_n, const float* __restrict__ wt /* [K][64] */, const float* __restrict__ bias,
              const float* __restrict__ mu, const float* __restrict__ inv_sigma, __half* __restrict__ f0pad, BandMajor bm,
              const uint8_t* __restrict__ valid, const int tid) {
  using namespace c0s;
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const int KC = KP / 8;
  // X chunk planes are 2048 + 16 bytes apart (LBO = 2064): consecutive chunks start 16 B further along the banks, so
  // the loaders' stores (one pixel's K values spread over the chunk planes) do not pile onto the same banks
  constexpr int XCH = 2064;
  const int whalf = KC * 64 * 16, xhalf = (KC * XCH + 127) / 128 * 128;
  const int wbytes = whalf * (kSplit ? 2 : 1), xbytes = xhalf * (kSplit ? 2 : 1);      // [hi | lo]
  const int S_W = 0, S_X = wbytes, S_BIAS = S_X + nstage * xbytes, S_MU = S_BIAS + 256, S_BAR = S_MU + ((KP * 4 + 127) / 128) * 128;
  const int S_TMEM = S_BAR + 64;
  const uint32_t bars = sbase + S_BAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);
  float* smu = reinterpret_cast<float*>(smem + S_MU);      // per input channel: mean (raw cube) or 0
  const int64_t plane = int64_t(prow_n) * pcol_n;
  const int64_t ntiles = (plane + 127) / 128;
  const int lo = window_lo(w);

  // weights [K][64] f32 -> fp16 K-major B operand [KC][64 n][8 k], zero for k >= K
  {
    __half* sw = reinterpret_cast<__half*>(smem + S_W);
    for (int i = tid; i < KP * 64; i += kThreads) {
      const int k = i >> 6, n = i & 63;
      // raw cube: the operand is z-scored per band ((x - mu) * inv_sigma ~ O(1)) and the band's sigma moves into the
      // weight, so neither side of the product falls into fp16's subnormal range (folded weights alone are ~1e-5)
      const float sc = (inv_sigma && k < K) ? 1.f / __ldg(inv_sigma + k) : 1.f;
      const float wv = k < K ? __ldg(wt + k * 64 + n) * sc : 0.f;
      const __half hi = __float2half_rn(wv);
      sw[((k >> 3) * 64 + n) * 8 + (k & 7)] = hi;
      if (kSplit) sw[whalf / 2 + ((k >> 3) * 64 + n) * 8 + (k & 7)] = __float2half_rn(wv - __half2float(hi));
    }
    if (tid < 64) reinterpret_cast<float*>(smem + S_BIAS)[tid] = __ldg(bias + tid);
    for (int i = tid; i < KP; i += kThreads) smu[i] = (mu && i < K) ? __ldg(mu + i) : 0.f;
    // K padding of both X stages (k in [K, KP)) is written once: the loaders only touch k < K
    if (KP > K) {
      const int nh = nstage * (kSplit ? 2 : 1);                 // hi / lo halves of every stage are xhalf apart
      for (int i = tid; i < nh * 128 * (KP - K); i += kThreads) {
        const int st = i / (128 * (KP - K)), r = i - st * 128 * (KP - K);
        const int pos = r / (KP - K), k = K + (r - pos * (KP - K));
        *reinterpret_cast<__half*>(smem + S_X + st * xhalf + (k >> 3) * XCH + pos * 16 + (k & 7) * 2) = __float2half_rn(0.f);
      }
    }
  }
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {                              // (stage 1 is unused when nstage == 1)
      mbar_init(bars + 8 * (X_FULL0 + s), kWorkers);
      mbar_init(bars + 8 * (X_EMPTY0 + s), 1);
      mbar_init(bars + 8 * (D_FULL0 + s), 1);
      mbar_init(bars + 8 * (D_EMPTY0 + s), kWorkers);
    }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(sbase + S_TMEM, 128);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int64_t t_first = blockIdx.x, t_step = gridDim.x;

  if (warp == 8) {
    const uint32_t kI = make_idesc_f16(128, 64);
    int it = 0;
    for (int64_t t = t_first; t < ntiles; t += t_step, ++it) {
      const int s = it & 1, ph = (it >> 1) & 1;                 // TMEM slot
      const int xs_ = nstage == 2 ? s : 0, xph = nstage == 2 ? ph : (it & 1);   // X stage and its phase
      mbar_wait(bars + 8 * (X_FULL0 + xs_), xph, 80);
      mbar_wait(bars + 8 * (D_EMPTY0 + s), ph ^ 1, 81);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t xa = sbase + S_X + xs_ * xbytes, wa = sbase + S_W;
        for (int ks = 0; ks < KP / 16; ++ks) {
          umma_f16(tmem + s * 64, make_desc(xa + ks * 2 * XCH, XCH, 128), make_desc(wa + ks * 2 * 1024, 1024, 128), kI,
                   ks != 0 ? 1u : 0u);
          if (kSplit) {
            umma_f16(tmem + s * 64, make_desc(xa + ks * 2 * XCH, XCH, 128), make_desc(wa + whalf + ks * 2 * 1024, 1024, 128), kI, 1u);
            umma_f16(tmem + s * 64, make_desc(xa + xhalf + ks * 2 * XCH, XCH, 128), make_desc(wa + ks * 2 * 1024, 1024, 128), kI, 1u);
          }
        }
        umma_commit(bars + 8 * (X_EMPTY0 + xs_));
        umma_commit(bars + 8 * (D_FULL0 + s));
      }
      __syncwarp();
    }
  } else {
    const int q4 = warp & 3, chalf = warp >> 2;
    const float* sb = reinterpret_cast<const float*>(smem + S_BIAS) + chalf * 32;
    auto load_tile = [&](int64_t t, int it) {
      const int s = nstage == 2 ? (it & 1) : 0;
      mbar_wait(bars + 8 * (X_EMPTY0 + s), (nstage == 2 ? ((it >> 1) & 1) : (it & 1)) ^ 1, 82);
      unsigned char* xs = smem + S_X + s * xbytes;
      const int64_t p0 = t * 128;
      auto pix_of = [&](int pos) -> int64_t {                   // the position's mirrored source pixel in the slab
        int pp = int(p0) + pos; if (pp >= int(plane)) pp = int(plane) - 1;      // plane < 2^31 (checked by the launcher)
        const int pr = pp / pcol_n, pc = pp - pr * pcol_n;
        const int sr = mirror_index(band_row0 + pr + lo, scene_rows) - slab_row0, sc = mirror_index(pc + lo, cols);
        return int64_t(sr) * cols + sc;
      };
      auto src_of = [&](int pos) -> const T* { return in + pix_of(pos) * K; };
      if constexpr (kBM) {
        // band-major slab: a thread owns one of the tile's 128 positions and reads 8 consecutive bands per K-chunk (each
        // load coalesced along the warp's consecutive columns), then stores the chunk as one 16-byte hi and one lo write.
        // The z-score and the split are those of the pixel-major loader below, so the operand is the same byte for byte.
        const int pos = tid & 127;
        int pp = int(p0) + pos; if (pp >= int(plane)) pp = int(plane) - 1;
        const int pr = pp / pcol_n, pc = pp - pr * pcol_n;
        const int sr = mirror_index(band_row0 + pr + lo, scene_rows) - slab_row0, sc = mirror_index(pc + lo, cols);
        const T* src = in + int64_t(sr) * bm.rs + sc;
        const int kc_end = (K + 7) / 8;                         // chunks past it are K padding, written once above
        const bool ok = !valid || valid[int64_t(sr) * cols + sc];   // the source pixel has data
#pragma unroll 1
        for (int c0 = tid >> 7; c0 < kc_end; c0 += 8) {        // 4 chunks (32 loads) in flight per thread
          float v[4][8];
#pragma unroll
          for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int k = (c0 + 2 * u) * 8 + e;
              v[u][e] = k < K ? float(src[int64_t(k) * bm.bs]) : 0.f;
            }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int kc = c0 + 2 * u;
            if (kc < kc_end) {
              __half2 hi[4], lo2[4];
#pragma unroll
              for (int e = 0; e < 8; e += 2) {
                const int k = kc * 8 + e;
                const float z0 = (ok && k < K) ? (v[u][e] - smu[k]) * __ldg(inv_sigma + k) : 0.f;
                const float z1 = (ok && k + 1 < K) ? (v[u][e + 1] - smu[k + 1]) * __ldg(inv_sigma + k + 1) : 0.f;
                const __half h0 = __float2half_rn(z0), h1 = __float2half_rn(z1);
                hi[e / 2] = __halves2half2(h0, h1);
                lo2[e / 2] = __halves2half2(__float2half_rn(z0 - __half2float(h0)), __float2half_rn(z1 - __half2float(h1)));
              }
              unsigned char* d = xs + kc * XCH + pos * 16;
              *reinterpret_cast<uint4*>(d) = *reinterpret_cast<const uint4*>(hi);
              *reinterpret_cast<uint4*>(d + xhalf) = *reinterpret_cast<const uint4*>(lo2);
            }
          }
        }
      } else if constexpr (kVec4) {
        // K = 60 floats, 16-byte aligned pixels: a half-warp reads one pixel (15 float4 on 15 lanes), 8 pixels per lane
        // in flight; K % 4 == 0 and K <= 64
        const int hw = lane >> 4, q = lane & 15, Q = K / 4;
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int pos = 2 * (warp + 8 * j) + hw;
          v[j] = q < Q ? __ldg(reinterpret_cast<const float4*>(src_of(pos)) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (q < Q) {
          const float m0 = smu[4 * q], m1 = smu[4 * q + 1], m2 = smu[4 * q + 2], m3 = smu[4 * q + 3];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int pos = 2 * (warp + 8 * j) + hw;
            const __half2 h0 = __floats2half2_rn(v[j].x - m0, v[j].y - m1), h1 = __floats2half2_rn(v[j].z - m2, v[j].w - m3);
            uint2 pk;
            pk.x = *reinterpret_cast<const uint32_t*>(&h0); pk.y = *reinterpret_cast<const uint32_t*>(&h1);
            *reinterpret_cast<uint2*>(xs + (q >> 1) * XCH + pos * 16 + (q & 1) * 8) = pk;
          }
        }
      } else {
        // scalar elements (uint16 / unaligned float rows): a warp reads one pixel (K values on consecutive lanes),
        // z-scored on the way (per-lane mean / 1/sigma of its k's stay in registers); K <= 256
        float mr[8], ir[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const int k = lane + 32 * m;
          mr[m] = k < K ? smu[k] : 0.f;
          ir[m] = (inv_sigma && k < K) ? __ldg(inv_sigma + k) : 1.f;
        }
#pragma unroll 1
        for (int j0 = 0; j0 < 16; j0 += 4) {                   // 4 pixels (up to 32 loads) in flight per lane
          float v[4][8];
          bool ok[4];                                           // the source pixel has data
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int64_t px = pix_of(warp + 8 * (j0 + jj));
            const T* src = in + px * K;
#pragma unroll
            for (int m = 0; m < 8; ++m) {
              const int k = lane + 32 * m;
              v[jj][m] = k < K ? float(src[k]) : 0.f;
            }
            ok[jj] = !valid || valid[px];
          }
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int pos = warp + 8 * (j0 + jj);
#pragma unroll
            for (int m = 0; m < 8; ++m) {
              const int k = lane + 32 * m;
              if (k < K) {
                const float z = ok[jj] ? (v[jj][m] - mr[m]) * ir[m] : 0.f;
                const __half hi = __float2half_rn(z);
                unsigned char* d = xs + (k >> 3) * XCH + pos * 16 + (k & 7) * 2;
                *reinterpret_cast<__half*>(d) = hi;
                if (kSplit) *reinterpret_cast<__half*>(d + xhalf) = __float2half_rn(z - __half2float(hi));
              }
            }
          }
        }
      }
      fence_proxy_async();
      mbar_arrive(bars + 8 * (X_FULL0 + s));
    };
    int it = 0;
    if (t_first < ntiles) load_tile(t_first, 0);
    for (int64_t t = t_first; t < ntiles; t += t_step, ++it) {
      if (t + t_step < ntiles) load_tile(t + t_step, it + 1);   // (waits for the stage: immediate with two stages)
      const int s = it & 1;
      mbar_wait(bars + 8 * (D_FULL0 + s), (it >> 1) & 1, 83);
      tc_fence_after();
      float v[32];
      const uint32_t taddr = tmem + (uint32_t(q4 * 32) << 16) + s * 64 + chalf * 32;
      tmem_ld16(taddr, v);
      tmem_ld16(taddr + 16, v + 16);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bars + 8 * (D_EMPTY0 + s));
      const int64_t p = t * 128 + q4 * 32 + lane;
      if (p < plane) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          __half2 h[4];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            h[j] = __floats2half2_rn(v[c * 8 + 2 * j] + sb[c * 8 + 2 * j], v[c * 8 + 2 * j + 1] + sb[c * 8 + 2 * j + 1]);
          *reinterpret_cast<uint4*>(f0pad + (int64_t(chalf * 4 + c) * plane + p) * 8) = *reinterpret_cast<uint4*>(h);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) { tc_fence_after(); tmem_dealloc(tmem, 128); }
}

template <typename T, bool kVec4, bool kSplit>
__global__ void __launch_bounds__(c0s::kThreads, 1)
conv0_tc_kernel(const T* __restrict__ in, int K, int KP, int nstage, int scene_rows, int cols, int slab_row0, int w, int band_row0,
                int prow_n, int pcol_n, const float* __restrict__ wt /* [K][64] */, const float* __restrict__ bias,
                const float* __restrict__ mu, const float* __restrict__ inv_sigma, __half* __restrict__ f0pad,
                const uint8_t* __restrict__ valid) {
  conv0_tc_body<T, kVec4, kSplit, false>(in, K, KP, nstage, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt,
                                         bias, mu, inv_sigma, f0pad, BandMajor{}, valid, threadIdx.x);
}

// the raw cube in BIL / BSQ (split operands)
template <typename T>
__global__ void __launch_bounds__(c0s::kThreads, 1)
conv0_tc_bm_kernel(const T* __restrict__ in, int K, int KP, int nstage, int scene_rows, int cols, int slab_row0, int w,
                   int band_row0, int prow_n, int pcol_n, const float* __restrict__ wt /* [K][64] */,
                   const float* __restrict__ bias, const float* __restrict__ mu, const float* __restrict__ inv_sigma,
                   __half* __restrict__ f0pad, BandMajor bm, const uint8_t* __restrict__ valid) {
  conv0_tc_body<T, false, true, true>(in, K, KP, nstage, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias,
                                      mu, inv_sigma, f0pad, bm, valid, threadIdx.x);
}

// K-sliced variant for the raw cube beyond 256 bands (split hi / lo operands only).  A tile's X operand no longer fits one
// shared-memory stage, so it passes through a two-stage ring of 64-band slices [8 chunks][128 positions][8] (hi | lo):
// the workers load and z-score slice j of a tile while the MMA thread consumes slice j-1, and the 3 x 4 tcgen05.mma of
// every slice accumulate into the tile's TMEM slot.  The folded weights stay resident as fp16 hi + lo ([KC][64][8] each,
// 128 KB at 512 bands).  Tile loop, TMEM slots, mirror index map and epilogue are those of conv0_tc_kernel.
namespace c0k {
constexpr int kSlice = 64, kSliceChunks = kSlice / 8;
constexpr int XCH = 2064;                                     // chunk-plane stride of a slice (as conv0_tc_kernel's)
constexpr int kXHalf = kSliceChunks * XCH;                    // one slice, hi or lo: 16 512 B
constexpr int kMaxK = 512;
}  // namespace c0k

template <typename T, bool kBM>
__device__ __forceinline__ void
conv0_tc_sliced_body(const T* __restrict__ in, int K, int KP, int scene_rows, int cols, int slab_row0, int w, int band_row0,
                     int prow_n, int pcol_n, const float* __restrict__ wt /* [K][64] */, const float* __restrict__ bias,
                     const float* __restrict__ mu, const float* __restrict__ inv_sigma, __half* __restrict__ f0pad,
                     BandMajor bm, const uint8_t* __restrict__ valid, const int tid) {
  using namespace c0s;
  using c0k::kSlice; using c0k::XCH; using c0k::kXHalf;
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const int KC = KP / 8, nslice = (KP + kSlice - 1) / kSlice;
  const int whalf = KC * 64 * 16;
  const int S_W = 0, S_X = 2 * whalf, S_BIAS = S_X + 2 * 2 * kXHalf, S_MU = S_BIAS + 256, S_IS = S_MU + KP * 4,
            S_BAR = S_IS + KP * 4;
  const int S_TMEM = S_BAR + 64;
  const uint32_t bars = sbase + S_BAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);
  float* smu = reinterpret_cast<float*>(smem + S_MU);
  float* sis = reinterpret_cast<float*>(smem + S_IS);
  const int64_t plane = int64_t(prow_n) * pcol_n;
  const int64_t ntiles = (plane + 127) / 128;
  const int lo = window_lo(w);

  // weights [K][64] f32 (times the band's sigma, see conv0_tc_kernel) -> fp16 hi / lo K-major B operands [KC][64 n][8 k]
  {
    __half* sw = reinterpret_cast<__half*>(smem + S_W);
    for (int i = tid; i < KP * 64; i += kThreads) {
      const int k = i >> 6, n = i & 63;
      const float wv = k < K ? __ldg(wt + k * 64 + n) * (1.f / __ldg(inv_sigma + k)) : 0.f;
      const __half hi = __float2half_rn(wv);
      sw[((k >> 3) * 64 + n) * 8 + (k & 7)] = hi;
      sw[whalf / 2 + ((k >> 3) * 64 + n) * 8 + (k & 7)] = __float2half_rn(wv - __half2float(hi));
    }
    if (tid < 64) reinterpret_cast<float*>(smem + S_BIAS)[tid] = __ldg(bias + tid);
    for (int i = tid; i < KP; i += kThreads) {
      smu[i] = i < K ? __ldg(mu + i) : 0.f;
      sis[i] = i < K ? __ldg(inv_sigma + i) : 0.f;       // k >= K: the loaders write 0
    }
  }
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(bars + 8 * (X_FULL0 + s), kWorkers);
      mbar_init(bars + 8 * (X_EMPTY0 + s), 1);
      mbar_init(bars + 8 * (D_FULL0 + s), 1);
      mbar_init(bars + 8 * (D_EMPTY0 + s), kWorkers);
    }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(sbase + S_TMEM, 128);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int64_t t_first = blockIdx.x, t_step = gridDim.x;

  if (warp == 8) {
    const uint32_t kI = make_idesc_f16(128, 64);
    int it = 0, g = 0;                                          // tile count, slice count (ring position)
    for (int64_t t = t_first; t < ntiles; t += t_step, ++it) {
      const int s = it & 1, ph = (it >> 1) & 1;                 // TMEM slot
      mbar_wait(bars + 8 * (D_EMPTY0 + s), ph ^ 1, 91);
      for (int j = 0; j < nslice; ++j, ++g) {
        const int xs_ = g & 1;
        mbar_wait(bars + 8 * (X_FULL0 + xs_), (g >> 1) & 1, 90);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t xa = sbase + S_X + xs_ * 2 * kXHalf, wa = sbase + S_W;
          const int ksteps = (KP - j * kSlice < kSlice ? KP - j * kSlice : kSlice) / 16;
          for (int ks = 0; ks < ksteps; ++ks) {
            const uint32_t wk = wa + (j * (kSlice / 16) + ks) * 2 * 1024;
            umma_f16(tmem + s * 64, make_desc(xa + ks * 2 * XCH, XCH, 128), make_desc(wk, 1024, 128), kI,
                     (j | ks) != 0 ? 1u : 0u);
            umma_f16(tmem + s * 64, make_desc(xa + ks * 2 * XCH, XCH, 128), make_desc(wk + whalf, 1024, 128), kI, 1u);
            umma_f16(tmem + s * 64, make_desc(xa + kXHalf + ks * 2 * XCH, XCH, 128), make_desc(wk, 1024, 128), kI, 1u);
          }
          umma_commit(bars + 8 * (X_EMPTY0 + xs_));
          if (j == nslice - 1) umma_commit(bars + 8 * (D_FULL0 + s));
        }
        __syncwarp();
      }
    }
  } else {
    const int q4 = warp & 3, chalf = warp >> 2;
    const float* sb = reinterpret_cast<const float*>(smem + S_BIAS) + chalf * 32;
    int g = 0;                                                  // slice count (ring position), as the MMA thread's
    // all slices of tile t: a warp reads one pixel's 64 bands of the slice (two per lane), 8 pixels in flight per lane
    auto load_tile = [&](int64_t t) {
      const int64_t p0 = t * 128;
      if constexpr (kBM) {
        // band-major slab: as in conv0_tc_kernel, a thread owns one position and reads 8 consecutive bands per K-chunk,
        // 4 of a slice's 8 chunks; the z-score (0 for k >= K) and split are those of the pixel-major loader below
        const int pos = tid & 127;
        int pp = int(p0) + pos; if (pp >= int(plane)) pp = int(plane) - 1;
        const int pr = pp / pcol_n, pc = pp - pr * pcol_n;
        const int sr = mirror_index(band_row0 + pr + lo, scene_rows) - slab_row0, sc = mirror_index(pc + lo, cols);
        const T* src = in + int64_t(sr) * bm.rs + sc;
        const bool ok = !valid || valid[int64_t(sr) * cols + sc];   // the source pixel has data
#pragma unroll 1
        for (int j = 0; j < nslice; ++j, ++g) {
          const int s = g & 1;
          mbar_wait(bars + 8 * (X_EMPTY0 + s), ((g >> 1) & 1) ^ 1, 92);
          unsigned char* xs = smem + S_X + s * 2 * kXHalf;
          float v[4][8];
#pragma unroll
          for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int k = j * kSlice + ((tid >> 7) + 2 * u) * 8 + e;
              v[u][e] = k < K ? float(src[int64_t(k) * bm.bs]) : 0.f;
            }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int kl = ((tid >> 7) + 2 * u) * 8;             // first band of the chunk within the slice
            __half2 hi[4], lo2[4];
#pragma unroll
            for (int e = 0; e < 8; e += 2) {
              const int k = j * kSlice + kl + e;
              const float z0 = ok ? (v[u][e] - smu[k < KP ? k : 0]) * (k < KP ? sis[k] : 0.f) : 0.f;
              const float z1 = ok ? (v[u][e + 1] - smu[k + 1 < KP ? k + 1 : 0]) * (k + 1 < KP ? sis[k + 1] : 0.f) : 0.f;
              const __half h0 = __float2half_rn(z0), h1 = __float2half_rn(z1);
              hi[e / 2] = __halves2half2(h0, h1);
              lo2[e / 2] = __halves2half2(__float2half_rn(z0 - __half2float(h0)), __float2half_rn(z1 - __half2float(h1)));
            }
            unsigned char* d = xs + (kl >> 3) * XCH + pos * 16;
            *reinterpret_cast<uint4*>(d) = *reinterpret_cast<const uint4*>(hi);
            *reinterpret_cast<uint4*>(d + kXHalf) = *reinterpret_cast<const uint4*>(lo2);
          }
          fence_proxy_async();
          mbar_arrive(bars + 8 * (X_FULL0 + s));
        }
      } else {
        const T* src[16];
        unsigned okm = 0xffffu;                                 // bit jj: pixel jj's source pixel has data
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
          int pp = int(p0) + warp + 8 * jj; if (pp >= int(plane)) pp = int(plane) - 1;     // plane < 2^31 (launcher)
          const int pr = pp / pcol_n, pc = pp - pr * pcol_n;
          const int sr = mirror_index(band_row0 + pr + lo, scene_rows) - slab_row0, sc = mirror_index(pc + lo, cols);
          src[jj] = in + (int64_t(sr) * cols + sc) * K;
          if (valid && !valid[int64_t(sr) * cols + sc]) okm &= ~(1u << jj);
        }
#pragma unroll 1
        for (int j = 0; j < nslice; ++j, ++g) {
          const int s = g & 1;
          mbar_wait(bars + 8 * (X_EMPTY0 + s), ((g >> 1) & 1) ^ 1, 92);
          unsigned char* xs = smem + S_X + s * 2 * kXHalf;
          const int k0 = j * kSlice + lane, k1 = k0 + 32;
          const float m0 = smu[k0 < KP ? k0 : 0], i0 = k0 < KP ? sis[k0] : 0.f;
          const float m1 = smu[k1 < KP ? k1 : 0], i1 = k1 < KP ? sis[k1] : 0.f;
#pragma unroll
          for (int h = 0; h < 16; h += 8) {
            float v[8][2];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              v[jj][0] = k0 < K ? float(src[h + jj][k0]) : 0.f;
              v[jj][1] = k1 < K ? float(src[h + jj][k1]) : 0.f;
            }
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              const int pos = warp + 8 * (h + jj);
#pragma unroll
              for (int m = 0; m < 2; ++m) {
                const int kl = lane + 32 * m;                    // band within the slice
                const float z = (okm >> (h + jj)) & 1 ? (v[jj][m] - (m ? m1 : m0)) * (m ? i1 : i0) : 0.f;   // 0 for k >= K
                const __half hi = __float2half_rn(z);
                unsigned char* d = xs + (kl >> 3) * XCH + pos * 16 + (kl & 7) * 2;
                *reinterpret_cast<__half*>(d) = hi;
                *reinterpret_cast<__half*>(d + kXHalf) = __float2half_rn(z - __half2float(hi));
              }
            }
          }
          fence_proxy_async();
          mbar_arrive(bars + 8 * (X_FULL0 + s));
        }
      }
    };
    int it = 0;
    if (t_first < ntiles) load_tile(t_first);
    for (int64_t t = t_first; t < ntiles; t += t_step, ++it) {
      if (t + t_step < ntiles) load_tile(t + t_step);           // its slices wait for the MMAs of this tile's last slices
      const int s = it & 1;
      mbar_wait(bars + 8 * (D_FULL0 + s), (it >> 1) & 1, 93);
      tc_fence_after();
      float v[32];
      const uint32_t taddr = tmem + (uint32_t(q4 * 32) << 16) + s * 64 + chalf * 32;
      tmem_ld16(taddr, v);
      tmem_ld16(taddr + 16, v + 16);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bars + 8 * (D_EMPTY0 + s));
      const int64_t p = t * 128 + q4 * 32 + lane;
      if (p < plane) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          __half2 h[4];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            h[j] = __floats2half2_rn(v[c * 8 + 2 * j] + sb[c * 8 + 2 * j], v[c * 8 + 2 * j + 1] + sb[c * 8 + 2 * j + 1]);
          *reinterpret_cast<uint4*>(f0pad + (int64_t(chalf * 4 + c) * plane + p) * 8) = *reinterpret_cast<uint4*>(h);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) { tc_fence_after(); tmem_dealloc(tmem, 128); }
}

template <typename T>
__global__ void __launch_bounds__(c0s::kThreads, 1)
conv0_tc_sliced_kernel(const T* __restrict__ in, int K, int KP, int scene_rows, int cols, int slab_row0, int w, int band_row0,
                       int prow_n, int pcol_n, const float* __restrict__ wt /* [K][64] */, const float* __restrict__ bias,
                       const float* __restrict__ mu, const float* __restrict__ inv_sigma, __half* __restrict__ f0pad,
                       const uint8_t* __restrict__ valid) {
  conv0_tc_sliced_body<T, false>(in, K, KP, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias, mu, inv_sigma,
                                 f0pad, BandMajor{}, valid, threadIdx.x);
}

// the raw cube in BIL / BSQ
template <typename T>
__global__ void __launch_bounds__(c0s::kThreads, 1)
conv0_tc_sliced_bm_kernel(const T* __restrict__ in, int K, int KP, int scene_rows, int cols, int slab_row0, int w,
                          int band_row0, int prow_n, int pcol_n, const float* __restrict__ wt /* [K][64] */,
                          const float* __restrict__ bias, const float* __restrict__ mu, const float* __restrict__ inv_sigma,
                          __half* __restrict__ f0pad, BandMajor bm, const uint8_t* __restrict__ valid) {
  conv0_tc_sliced_body<T, true>(in, K, KP, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias, mu, inv_sigma,
                                f0pad, bm, valid, threadIdx.x);
}

template <typename T>
static int launch_conv0_tc_sliced(const T* in, int K, int scene_rows, int cols, int slab_row0, int w, int band_row0,
                                  int prow_n, int pcol_n, const float* wt, const float* bias, const float* mu,
                                  const float* inv_sigma, __half* f0pad, const BandMajor* bm, const uint8_t* valid,
                                  cudaStream_t s) {
  const int KP = (K + 15) / 16 * 16;
  CMLPL_CHECK_ARG(K <= c0k::kMaxK, "conv0: K=%d unsupported by the tensor-core kernel (at most %d)", K, c0k::kMaxK);
  CMLPL_CHECK_ARG(mu && inv_sigma, "conv0: the K-sliced kernel needs the band means and 1/sigma");
  const size_t smem = size_t(KP / 8) * 64 * 16 * 2 + 2 * 2 * c0k::kXHalf + 256 + 2 * size_t(KP) * 4 + 64 + 16 + 128;
  CMLPL_CHECK_ARG(smem <= 227 * 1024, "conv0: K=%d does not fit shared memory", K);
  const int64_t ntiles = (int64_t(prow_n) * pcol_n + 127) / 128;
  int grid = sm_count();
  if (grid > ntiles) grid = int(ntiles);
  if (bm) {
    auto kern = conv0_tc_sliced_bm_kernel<T>;
    CMLPL_MAX_DYN_SMEM(kern, int(smem));
    kern<<<grid, c0s::kThreads, smem, s>>>(in, K, KP, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias, mu,
                                           inv_sigma, f0pad, *bm, valid);
  } else {
    auto kern = conv0_tc_sliced_kernel<T>;
    CMLPL_MAX_DYN_SMEM(kern, int(smem));
    kern<<<grid, c0s::kThreads, smem, s>>>(in, K, KP, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias, mu,
                                           inv_sigma, f0pad, valid);
  }
  CMLPL_CHECK_LAUNCH("conv0_tc_sliced");
  return CMLPL_OK;
}

// bm: the raw slab is band-major (BIL / BSQ; split operands only), or nullptr for pixel-major; valid: the slab's validity
// mask (split operands only), or nullptr
template <typename T, bool kVec4, bool kSplit>
int launch_conv0_tc(const T* in, int K, int scene_rows, int cols, int slab_row0, int w, int band_row0, int prow_n, int pcol_n,
                    const float* wt, const float* bias, const float* mu, const float* inv_sigma, __half* f0pad,
                    const BandMajor* bm, const uint8_t* valid, cudaStream_t s) {
  const int KP = (K + 15) / 16 * 16;
  CMLPL_CHECK_ARG(int64_t(prow_n) * pcol_n < (int64_t(1) << 31) - 256, "conv0: band of %d x %d padded positions is too large",
                  prow_n, pcol_n);
  // beyond 256 bands (raw cube only) the X operand of a tile passes through shared memory in K-slices
  if constexpr (kSplit && !kVec4)
    if (KP > 256)
      return launch_conv0_tc_sliced<T>(in, K, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias, mu,
                                       inv_sigma, f0pad, bm, valid, s);
  CMLPL_CHECK_ARG(!bm || (kSplit && !kVec4), "conv0: band-major input needs the split-operand kernel");
  CMLPL_CHECK_ARG(!valid || (kSplit && !kVec4), "conv0: a validity mask needs the raw-cube kernel");
  CMLPL_CHECK_ARG(KP <= 256 && (!kVec4 || (K % 4 == 0 && K <= 64)), "conv0: K=%d unsupported by the tensor-core kernel", K);
  const int KC = KP / 8;
  const size_t xhalf = (size_t(KC) * 2064 + 127) / 128 * 128, mult = kSplit ? 2 : 1;
  const size_t fixed = size_t(KC) * 64 * 16 * mult + 256 + ((KP * 4 + 127) / 128) * 128 + 64 + 16 + 128;
  const int nstage = fixed + 2 * xhalf * mult <= 227 * 1024 ? 2 : 1;
  const size_t smem = fixed + nstage * xhalf * mult;
  CMLPL_CHECK_ARG(smem <= 227 * 1024, "conv0: K=%d does not fit shared memory", K);
  const int64_t ntiles = (int64_t(prow_n) * pcol_n + 127) / 128;
  int grid = sm_count();
  if (grid > ntiles) grid = int(ntiles);
  if constexpr (kSplit && !kVec4) {
    if (bm) {
      auto kern = conv0_tc_bm_kernel<T>;
      CMLPL_MAX_DYN_SMEM(kern, int(smem));
      kern<<<grid, c0s::kThreads, smem, s>>>(in, K, KP, nstage, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt,
                                             bias, mu, inv_sigma, f0pad, *bm, valid);
      CMLPL_CHECK_LAUNCH("conv0_tc_bm");
      return CMLPL_OK;
    }
  }
  auto kern = conv0_tc_kernel<T, kVec4, kSplit>;
  CMLPL_MAX_DYN_SMEM(kern, int(smem));
  kern<<<grid, c0s::kThreads, smem, s>>>(in, K, KP, nstage, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias, mu,
                                         inv_sigma, f0pad, valid);
  CMLPL_CHECK_LAUNCH("conv0_tc");
  return CMLPL_OK;
}

#define CMLPL_CONV0_INST(T, kVec4, kSplit)                                                                                 \
  template int launch_conv0_tc<T, kVec4, kSplit>(const T*, int, int, int, int, int, int, int, int, const float*, const float*, \
                                                 const float*, const float*, __half*, const BandMajor*, const uint8_t*,   \
                                                 cudaStream_t);
CMLPL_CONV0_INST(float, true, false)
CMLPL_CONV0_INST(float, false, true)
CMLPL_CONV0_INST(uint16_t, false, true)
CMLPL_CONV0_INST(int16_t, false, true)
#undef CMLPL_CONV0_INST

}  // namespace cmlpl
