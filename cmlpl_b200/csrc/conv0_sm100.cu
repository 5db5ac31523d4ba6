// conv0 of the scene path on tcgen05: F0 = W . x + b once per PADDED scene position (tools/models.py:102,132 applied to
// the mirror-padded cube, hyper_tools.py:35-55) -> chunk-planar fp16 map [8 chunks][prow_n][pcol_n][8].
// x is either the 60-channel PCA cube (float) or the RAW cube (uint16 / int16 / float, K = B bands) with the PCA
// projection and both z-scores folded into W (SURVEY 8-f1): F0 = Wf . (x - mu) + bf.
//
// Persistent CTAs over tiles of 128 consecutive padded positions.  The 256 worker threads read a tile's source pixels
// (mirrored index map), round to fp16 and write the UMMA K-major tile [chunks][128 positions][8] straight into shared
// memory; one thread issues the tcgen05.mma (M=128, N=64) of a tile into one of two TMEM slots; the same workers drain
// the previous tile (+bias -> fp16 -> F0, 16-byte stores coalesced along positions) while their loads for the next tile
// are in flight.  A tile's X operand passes through shared memory as nslice slices of S bands, in a ring of nstage
// slice buffers (Conv0Plan): up to 256 bands one slice of all bands, in two buffers when two fit and else in one;
// beyond 256 bands 64-band slices in two buffers, the workers loading slice j while the MMA thread consumes slice j-1.
// The slices of a tile accumulate into its TMEM slot.  The loaders (kLoad) differ in how they read the source: the PCA
// cube as float4 rows; the pixel-major raw cube a pixel per warp (K contiguous values: fully coalesced); the band-major
// raw cube (BIL / BSQ) a position per thread, 8 bands per K-chunk, coalesced along columns.
// Replaces the CUDA-core conv0_tiled_kernel of round 1 (L1-wavefront bound on the strided pixel rows).
// valid (raw cube only; u8 [slab_rows * cols] over the slab's pixels, or nullptr): a position whose mirrored source pixel
// is no-data gets the z-scored operand 0 (hi and lo), i.e. the pixel stands in as its band means and F0 there is the
// folded bias exactly.  The mask byte is read once per tile position; the sample loads keep their order.
// Band selection (Sel = SceneBands, include/cmlpl.h cmlpl_scene_infer_raw_sel): channel k is raw band raw_band(sel, k) of
// pixels of ld samples (pixel-major) or of the band-major slab; the list is staged in shared memory, where the
// pixel-major loaders' lanes index it divergently.  K, the plan and the operands follow the selected count.
#include <type_traits>

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace cmlpl {

namespace c0s {
constexpr int kWorkers = 256, kThreads = kWorkers + 32;
enum { X_FULL0 = 0, X_EMPTY0 = 2, D_FULL0 = 4, D_EMPTY0 = 6 };
// X chunk planes are 2048 + 16 bytes apart (LBO = 2064): consecutive chunks start 16 B further along the banks, so
// the loaders' stores (one pixel's K values spread over the chunk planes) do not pile onto the same banks
constexpr int XCH = 2064;
constexpr int kSlice = 64, kMaxK = 512;                       // slice width beyond 256 bands; widest raw spectrum
// loaders: PCA cube (float4 rows, plain operands); pixel-major raw cube, one slice of up to 256 bands or 64-band
// slices; band-major raw cube, any slicing
enum { kLoadVec4, kLoadPixel, kLoadPixelSlice, kLoadBandMajor };
}  // namespace c0s

// Shared memory of conv0_tc_kernel, the same for the launcher (its size) and the kernel (its offsets): fp16 weights
// [KC][64 n][8 k] (hi | lo when split), the ring of nstage X slice buffers [S/8 chunks][128 positions][8] (hi | lo),
// bias, band means, the band list (u16 [KP], only with a list), barriers and the TMEM address.
struct Conv0Plan {
  int KP, S, nslice, nstage;
  int whalf, xhalf, xstage;                // bytes: weights hi, a slice buffer's hi, a slice buffer
  int x, bias, mu, sel, bar, tmem, bytes;  // offsets; the dynamic shared memory in all
};
__host__ __device__ inline int conv0_xhalf(int S) { return (S / 8 * c0s::XCH + 127) / 128 * 128; }
__host__ __device__ inline Conv0Plan conv0_plan(int K, bool split, bool sel) {
  Conv0Plan P;
  const int mult = split ? 2 : 1;
  P.KP = (K + 15) / 16 * 16;
  P.whalf = P.KP / 8 * 64 * 16;
  const int mu_bytes = (P.KP * 4 + 127) / 128 * 128, sel_bytes = sel ? (P.KP * 2 + 127) / 128 * 128 : 0;
  const int fixed = P.whalf * mult + 256 + mu_bytes + sel_bytes + 64 + 16 + 128;    // + barriers, TMEM address, alignment
  if (P.KP <= 256) {
    P.S = P.KP;
    P.nstage = fixed + 2 * conv0_xhalf(P.S) * mult <= 227 * 1024 ? 2 : 1;
  } else {
    P.S = c0s::kSlice;
    P.nstage = 2;
  }
  P.nslice = (P.KP + P.S - 1) / P.S;
  P.xhalf = conv0_xhalf(P.S);
  P.xstage = P.xhalf * mult;
  P.x = P.whalf * mult;
  P.bias = P.x + P.nstage * P.xstage;
  P.mu = P.bias + 256;
  P.sel = P.mu + mu_bytes;
  P.bar = P.sel + sel_bytes;
  P.tmem = P.bar + 64;
  P.bytes = fixed + P.nstage * P.xstage;
  return P;
}

// Split operands (raw cube): both operands are split into fp16 hi + lo parts and every K-step issues hi.hi + hi.lo +
// lo.hi (~2^-21 relative error).  The folded PCA projection is ill-conditioned -- its noise components are differences
// of band values ~10x larger than the result -- so single fp16 operands miss the 1e-3 logit bar (measured at B = 200).
// bm: the band-major slab's strides (kLoadBandMajor only); ld: samples per pixel of a pixel-major input (K without a list).
template <typename T, int kLoad, class Sel>
__global__ void __launch_bounds__(c0s::kThreads, 1)
conv0_tc_kernel(const T* __restrict__ in, int K, int ld, Sel sel, int scene_rows, int cols, int slab_row0, int w,
                int band_row0, int prow_n, int pcol_n, const float* __restrict__ wt /* [K][64] */,
                const float* __restrict__ bias, const float* __restrict__ mu, const float* __restrict__ inv_sigma,
                __half* __restrict__ f0pad, BandMajor bm, const uint8_t* __restrict__ valid) {
  using namespace c0s;
  constexpr bool kSplit = kLoad != kLoadVec4;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const Conv0Plan P = conv0_plan(K, kSplit, Sel::kSel);
  const auto bands = stage_bands(sel, reinterpret_cast<uint16_t*>(smem + P.sel));   // read after the __syncthreads below
  const int KP = P.KP, sh = P.nstage - 1;                       // slice g of the ring: buffer g & sh, phase (g >> sh) & 1
  const uint32_t bars = sbase + P.bar;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + P.tmem);
  float* smu = reinterpret_cast<float*>(smem + P.mu);          // per input channel: mean (raw cube) or 0
  const int64_t plane = int64_t(prow_n) * pcol_n;
  const int64_t ntiles = (plane + 127) / 128;
  const int lo = window_lo(w);

  // weights [K][64] f32 -> fp16 K-major B operand [KC][64 n][8 k] (hi | lo), zero for k >= K
  {
    __half* sw = reinterpret_cast<__half*>(smem);
    for (int i = tid; i < KP * 64; i += kThreads) {
      const int k = i >> 6, n = i & 63;
      // raw cube: the operand is z-scored per band ((x - mu) * inv_sigma ~ O(1)) and the band's sigma moves into the
      // weight, so neither side of the product falls into fp16's subnormal range (folded weights alone are ~1e-5)
      const float sc = (inv_sigma && k < K) ? 1.f / __ldg(inv_sigma + k) : 1.f;
      const float wv = k < K ? __ldg(wt + k * 64 + n) * sc : 0.f;
      const __half hi = __float2half_rn(wv);
      sw[((k >> 3) * 64 + n) * 8 + (k & 7)] = hi;
      if (kSplit) sw[P.whalf / 2 + ((k >> 3) * 64 + n) * 8 + (k & 7)] = __float2half_rn(wv - __half2float(hi));
    }
    if (tid < 64) reinterpret_cast<float*>(smem + P.bias)[tid] = __ldg(bias + tid);
    for (int i = tid; i < KP; i += kThreads) smu[i] = (mu && i < K) ? __ldg(mu + i) : 0.f;
  }
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {                              // (buffer 1 is unused when nstage == 1)
      mbar_init(bars + 8 * (X_FULL0 + s), kWorkers);
      mbar_init(bars + 8 * (X_EMPTY0 + s), 1);
      mbar_init(bars + 8 * (D_FULL0 + s), 1);
      mbar_init(bars + 8 * (D_EMPTY0 + s), kWorkers);
    }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(sbase + P.tmem, 128);
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
      mbar_wait(bars + 8 * (D_EMPTY0 + s), ph ^ 1, 81);
      for (int j = 0; j < P.nslice; ++j, ++g) {
        const int xs_ = g & sh;
        mbar_wait(bars + 8 * (X_FULL0 + xs_), (g >> sh) & 1, 80);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t xa = sbase + P.x + xs_ * P.xstage;
          const int k0 = j * P.S, ksteps = (KP - k0 < P.S ? KP - k0 : P.S) / 16;
          for (int ks = 0; ks < ksteps; ++ks) {
            const uint32_t xk = xa + ks * 2 * XCH, wk = sbase + (k0 / 16 + ks) * 2 * 1024;
            umma_f16(tmem + s * 64, make_desc(xk, XCH, 128), make_desc(wk, 1024, 128), kI, (j | ks) != 0 ? 1u : 0u);
            if (kSplit) {
              umma_f16(tmem + s * 64, make_desc(xk, XCH, 128), make_desc(wk + P.whalf, 1024, 128), kI, 1u);
              umma_f16(tmem + s * 64, make_desc(xk + P.xhalf, XCH, 128), make_desc(wk, 1024, 128), kI, 1u);
            }
          }
          umma_commit(bars + 8 * (X_EMPTY0 + xs_));
          if (j == P.nslice - 1) umma_commit(bars + 8 * (D_FULL0 + s));
        }
        __syncwarp();
      }
    }
  } else {
    const int q4 = warp & 3, chalf = warp >> 2;
    const float* sb = reinterpret_cast<const float*>(smem + P.bias) + chalf * 32;
    const int xhalf = P.xhalf;
    int g = 0;                                                  // slice count (ring position), as the MMA thread's
    // slab row and column of the mirrored source pixel of position pos of the tile at p0 (positions past the plane
    // repeat its last one; plane < 2^31, checked by the launcher)
    auto src_pixel = [&](int64_t p0, int pos) {
      int pp = int(p0) + pos; if (pp >= int(plane)) pp = int(plane) - 1;
      const int pr = pp / pcol_n, pc = pp - pr * pcol_n;
      return make_int2(mirror_index(band_row0 + pr + lo, scene_rows) - slab_row0, mirror_index(pc + lo, cols));
    };
    // each slice j of a tile: wait for its buffer, fill(j, buffer), hand it to the MMA thread.  A loader fills the
    // slice's bands below KP (the MMAs read no further), with zeros for k >= K.
    auto for_slices = [&](auto&& fill) {
#pragma unroll 1
      for (int j = 0; j < P.nslice; ++j, ++g) {
        const int st = g & sh;
        mbar_wait(bars + 8 * (X_EMPTY0 + st), ((g >> sh) & 1) ^ 1, 82);
        fill(j, smem + P.x + st * P.xstage);
        fence_proxy_async();
        mbar_arrive(bars + 8 * (X_FULL0 + st));
      }
    };
    auto load_tile = [&](int64_t t) {
      const int64_t p0 = t * 128;
      if constexpr (kLoad == kLoadVec4) {
        // K = 60 floats, 16-byte aligned pixels: a half-warp reads one pixel (15 float4 on 15 lanes), 8 pixels per lane
        // in flight; K % 4 == 0 and K <= 64
        for_slices([&](int, unsigned char* xs) {
          const int hw = lane >> 4, q = lane & 15, Q = K / 4;
          float4 v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int2 sp = src_pixel(p0, 2 * (warp + 8 * j) + hw);
            v[j] = q < Q ? __ldg(reinterpret_cast<const float4*>(in + (int64_t(sp.x) * cols + sp.y) * K) + q)
                         : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          if (q < KP / 4) {
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
        });
      } else if constexpr (kLoad == kLoadPixel) {
        // one slice of K <= 256 bands: a warp reads one pixel (K values on consecutive lanes), z-scored on the way
        // (per-lane mean / 1/sigma of its k's stay in registers), 4 pixels (up to 32 loads) in flight per lane
        for_slices([&](int, unsigned char* xs) {
          float mr[8], ir[8];
          int rb[8];                                            // raw band of each of the lane's k's (AllBands: k itself)
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            const int k = lane + 32 * m;
            mr[m] = k < K ? smu[k] : 0.f;
            ir[m] = (inv_sigma && k < K) ? __ldg(inv_sigma + k) : 1.f;
            rb[m] = k < K ? raw_band(bands, k) : 0;
          }
#pragma unroll 1
          for (int j0 = 0; j0 < 16; j0 += 4) {
            float v[4][8];
            bool ok[4];                                         // the source pixel has data
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int2 sp = src_pixel(p0, warp + 8 * (j0 + jj));
              const int64_t px = int64_t(sp.x) * cols + sp.y;
              const T* src = in + px * ld;
#pragma unroll
              for (int m = 0; m < 8; ++m) {
                const int k = lane + 32 * m;
                v[jj][m] = k < K ? float(src[Sel::kSel ? rb[m] : k]) : 0.f;
              }
              ok[jj] = !valid || valid[px];
            }
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int pos = warp + 8 * (j0 + jj);
#pragma unroll
              for (int m = 0; m < 8; ++m) {
                const int k = lane + 32 * m;
                if (k < KP) {
                  const float z = ok[jj] ? (v[jj][m] - mr[m]) * ir[m] : 0.f;
                  const __half hi = __float2half_rn(z);
                  unsigned char* d = xs + (k >> 3) * XCH + pos * 16 + (k & 7) * 2;
                  *reinterpret_cast<__half*>(d) = hi;
                  *reinterpret_cast<__half*>(d + xhalf) = __float2half_rn(z - __half2float(hi));
                }
              }
            }
          }
        });
      } else if constexpr (kLoad == kLoadPixelSlice) {
        // 64-band slices: a warp reads one pixel's 64 bands of the slice (two per lane), 8 pixels in flight per lane
        const T* src[16];
        unsigned okm = 0xffffu;                                 // bit jj: pixel jj's source pixel has data
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
          const int2 sp = src_pixel(p0, warp + 8 * jj);
          const int64_t px = int64_t(sp.x) * cols + sp.y;
          src[jj] = in + px * ld;
          if (valid && !valid[px]) okm &= ~(1u << jj);
        }
        for_slices([&](int j, unsigned char* xs) {
          const int k0 = j * kSlice + lane, k1 = k0 + 32;
          const float m0 = smu[k0 < KP ? k0 : 0], i0 = k0 < K ? __ldg(inv_sigma + k0) : 0.f;
          const float m1 = smu[k1 < KP ? k1 : 0], i1 = k1 < K ? __ldg(inv_sigma + k1) : 0.f;
          const int b0 = k0 < K ? raw_band(bands, k0) : 0, b1 = k1 < K ? raw_band(bands, k1) : 0;
#pragma unroll
          for (int h = 0; h < 16; h += 8) {
            float v[8][2];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              v[jj][0] = k0 < K ? float(src[h + jj][Sel::kSel ? b0 : k0]) : 0.f;
              v[jj][1] = k1 < K ? float(src[h + jj][Sel::kSel ? b1 : k1]) : 0.f;
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
                *reinterpret_cast<__half*>(d + xhalf) = __float2half_rn(z - __half2float(hi));
              }
            }
          }
        });
      } else {
        // band-major slab: a thread owns one of the tile's 128 positions and reads 8 consecutive bands per K-chunk (each
        // load coalesced along the warp's consecutive columns), 4 chunks (32 loads) in flight, then stores each chunk as
        // one 16-byte hi and one lo write.  The z-score and the split are those of the pixel-major loaders, so the
        // operand is the same byte for byte.
        const int pos = tid & 127;
        const int2 sp = src_pixel(p0, pos);
        const T* src = in + int64_t(sp.x) * bm.rs + sp.y;
        const bool ok = !valid || valid[int64_t(sp.x) * cols + sp.y];   // the source pixel has data
        for_slices([&](int j, unsigned char* xs) {
          const int kb = j * P.S, nch = (KP - kb < P.S ? KP - kb : P.S) / 8;   // first band and chunks of the slice
#pragma unroll 1
          for (int c0 = tid >> 7; c0 < nch; c0 += 8) {
            float v[4][8];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int k = kb + (c0 + 2 * u) * 8 + e;
                v[u][e] = k < K ? float(src[int64_t(raw_band(bands, k)) * bm.bs]) : 0.f;
              }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int kc = c0 + 2 * u;
              if (kc < nch) {
                __half2 hi[4], lo2[4];
#pragma unroll
                for (int e = 0; e < 8; e += 2) {
                  const int k = kb + kc * 8 + e;
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
        });
      }
    };
    int it = 0;
    if (t_first < ntiles) load_tile(t_first);
    for (int64_t t = t_first; t < ntiles; t += t_step, ++it) {
      if (t + t_step < ntiles) load_tile(t + t_step);           // its slices wait for the MMAs to free their buffers
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

// kVec4 (PCA cube) with plain operands, or the raw cube with split operands.  bm: the raw slab is band-major (BIL /
// BSQ), or nullptr for pixel-major with ld samples per pixel; valid: the raw slab's validity mask, or nullptr; sel: the
// raw bands of the K channels (AllBands: channel k is band k)
template <typename T, bool kVec4, bool kSplit, class Sel>
int launch_conv0_tc(const T* in, int K, int ld, const Sel& sel, int scene_rows, int cols, int slab_row0, int w, int band_row0,
                    int prow_n, int pcol_n, const float* wt, const float* bias, const float* mu, const float* inv_sigma,
                    __half* f0pad, const BandMajor* bm, const uint8_t* valid, cudaStream_t s) {
  static_assert(kVec4 != kSplit, "conv0 reads the PCA cube with plain operands and the raw cube with split ones");
  static_assert(!(kVec4 && Sel::kSel), "a band list selects raw bands");
  using namespace c0s;
  CMLPL_CHECK_ARG(int64_t(prow_n) * pcol_n < (int64_t(1) << 31) - 256, "conv0: band of %d x %d padded positions is too large",
                  prow_n, pcol_n);
  const Conv0Plan P = conv0_plan(K, kSplit, Sel::kSel);
  if (kSplit && P.KP > 256) {
    CMLPL_CHECK_ARG(K <= kMaxK, "conv0: K=%d unsupported by the tensor-core kernel (at most %d)", K, kMaxK);
    CMLPL_CHECK_ARG(mu && inv_sigma, "conv0: the K-sliced kernel needs the band means and 1/sigma");
  } else {
    CMLPL_CHECK_ARG(!bm || kSplit, "conv0: band-major input needs the split-operand kernel");
    CMLPL_CHECK_ARG(!valid || kSplit, "conv0: a validity mask needs the raw-cube kernel");
    CMLPL_CHECK_ARG(P.KP <= 256 && (!kVec4 || (K % 4 == 0 && K <= 64)), "conv0: K=%d unsupported by the tensor-core kernel", K);
  }
  CMLPL_CHECK_ARG(P.bytes <= 227 * 1024, "conv0: K=%d does not fit shared memory", K);
  const int64_t ntiles = (int64_t(prow_n) * pcol_n + 127) / 128;
  int grid = sm_count();
  if (grid > ntiles) grid = int(ntiles);
  // one instantiation of run per kernel, so that the shared-memory opt-in CMLPL_MAX_DYN_SMEM caches is that kernel's
  auto run = [&](auto load) {
    auto kern = conv0_tc_kernel<T, decltype(load)::value, Sel>;
    CMLPL_MAX_DYN_SMEM(kern, P.bytes);
    kern<<<grid, kThreads, P.bytes, s>>>(in, K, ld, sel, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n, wt, bias, mu,
                                         inv_sigma, f0pad, bm ? *bm : BandMajor{}, valid);
    CMLPL_CHECK_LAUNCH("conv0_tc");
    return CMLPL_OK;
  };
  if constexpr (kVec4) return run(std::integral_constant<int, kLoadVec4>{});
  else if (bm) return run(std::integral_constant<int, kLoadBandMajor>{});
  else if (P.nslice > 1) return run(std::integral_constant<int, kLoadPixelSlice>{});
  else return run(std::integral_constant<int, kLoadPixel>{});
}

#define CMLPL_CONV0_INST(T, kVec4, kSplit, Sel)                                                                             \
  template int launch_conv0_tc<T, kVec4, kSplit, Sel>(const T*, int, int, const Sel&, int, int, int, int, int, int, int,    \
                                                      const float*, const float*, const float*, const float*, __half*,      \
                                                      const BandMajor*, const uint8_t*, cudaStream_t);
CMLPL_CONV0_INST(float, true, false, AllBands)
CMLPL_CONV0_INST(float, false, true, AllBands)
CMLPL_CONV0_INST(uint16_t, false, true, AllBands)
CMLPL_CONV0_INST(int16_t, false, true, AllBands)
CMLPL_CONV0_INST(float, false, true, SceneBands)
CMLPL_CONV0_INST(uint16_t, false, true, SceneBands)
CMLPL_CONV0_INST(int16_t, false, true, SceneBands)
#undef CMLPL_CONV0_INST

}  // namespace cmlpl
