// Tensor-core head of the scene path (sm_100a): the spectral branch relu(feat_spe(x)) (tools/models.py:142-143)
// and its classifier columns (models.py:150) as two chained tcgen05 GEMMs with fp16 operands / fp32 accumulate,
// then the sum of all logit partials + argmax (models.py:144,150; hyper_tools.py:426).
//   x16_tile(_raw)_kernel  : spectra (or the z-scored raw cube) -> fp16 A-operand tiles in the UMMA "no-swizzle
//                            K-major" layout [m-tile][K/8 chunks][128 rows][8 halves], so that a tile is one
//                            contiguous block the loader moves with cp.async.bulk (UBLKCP) and tcgen05.mma reads as is
//   spectral_logits_kernel : part = Wc_spe . relu(Wspe . x + b) per hidden quarter, the hidden features never in HBM
//   head_sum_kernel        : logits = bc + spectral partials + the gathered conv partials of pool2_cls_kernel, argmax
// valid (raw cube; u8 [n] over the band's pixels, or nullptr): the conversion writes zero rows for no-data pixels (their
// band means, z-scored), and the head labels them CMLPL_NODATA_LABEL
#include "common.cuh"
#include "sm100_ptx.cuh"

namespace cmlpl {

// ------------------------------------------------------------------ spectra -> fp16 tiles
__global__ void x16_tile_kernel(const float* __restrict__ X, int64_t n, int B, int KC, int64_t total,
                                __half* __restrict__ out) {
  for (int64_t t = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; t < total; t += int64_t(gridDim.x) * blockDim.x) {
    const int row = int(t & 127);
    const int64_t r = t >> 7;
    const int kc = int(r % KC);
    const int64_t p = (r / KC) * 128 + row;
    __half2 h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = kc * 8 + 2 * e;
      const float a = (p < n && k < B) ? __ldg(X + p * B + k) : 0.f;
      const float b = (p < n && k + 1 < B) ? __ldg(X + p * B + k + 1) : 0.f;
      h[e] = __floats2half2_rn(a, b);
    }
    *reinterpret_cast<uint4*>(out + t * 8) = *reinterpret_cast<uint4*>(h);
  }
}

// same from the raw cube: x16 = (raw - mu) * inv_sigma  (featureNormalize(X, 1), hyper_tools.py:292)
template <typename T>
__global__ void x16_tile_raw_kernel(const T* __restrict__ X, int64_t n, int B, int KC, int64_t total,
                                    const float* __restrict__ mu, const float* __restrict__ inv_sigma,
                                    const uint8_t* __restrict__ valid, __half* __restrict__ out) {
  for (int64_t t = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; t < total; t += int64_t(gridDim.x) * blockDim.x) {
    const int row = int(t & 127);
    const int64_t r = t >> 7;
    const int kc = int(r % KC);
    const int64_t p = (r / KC) * 128 + row;
    const bool in = p < n && (!valid || valid[p]);
    __half2 h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = kc * 8 + 2 * e;
      const float a = (in && k < B) ? (float(X[p * B + k]) - __ldg(mu + k)) * __ldg(inv_sigma + k) : 0.f;
      const float b = (in && k + 1 < B) ? (float(X[p * B + k + 1]) - __ldg(mu + k + 1)) * __ldg(inv_sigma + k + 1) : 0.f;
      h[e] = __floats2half2_rn(a, b);
    }
    *reinterpret_cast<uint4*>(out + t * 8) = *reinterpret_cast<uint4*>(h);
  }
}

// same from a band-major raw slab (BIL / BSQ, include/cmlpl.h): pixel p of the band is row p / cols, column p % cols of
// the band's rows at X; with rows as the fastest index, a warp's loads of one band are consecutive columns
template <typename T>
__global__ void x16_tile_raw_bm_kernel(const T* __restrict__ X, BandMajor bm, int64_t n, int B, int KC, int64_t total,
                                       const float* __restrict__ mu, const float* __restrict__ inv_sigma,
                                       const uint8_t* __restrict__ valid, __half* __restrict__ out) {
  for (int64_t t = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; t < total; t += int64_t(gridDim.x) * blockDim.x) {
    const int row = int(t & 127);
    const int64_t r = t >> 7;
    const int kc = int(r % KC);
    const int64_t p = (r / KC) * 128 + row;
    const int64_t pr = p / bm.cols;
    const T* x = X + pr * bm.rs + (p - pr * bm.cols);
    const bool in = p < n && (!valid || valid[p]);
    __half2 h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = kc * 8 + 2 * e;
      const float a = (in && k < B) ? (float(x[k * bm.bs]) - __ldg(mu + k)) * __ldg(inv_sigma + k) : 0.f;
      const float b = (in && k + 1 < B) ? (float(x[(k + 1) * bm.bs]) - __ldg(mu + k + 1)) * __ldg(inv_sigma + k + 1) : 0.f;
      h[e] = __floats2half2_rn(a, b);
    }
    *reinterpret_cast<uint4*>(out + t * 8) = *reinterpret_cast<uint4*>(h);
  }
}

// ------------------------------------------------------------------ spectral logits: Wc_spe . relu(Wspe . x + b), hidden never in HBM
// spectral_logits_kernel fuses the two GEMMs of the spectral branch (models.py:142-143 and the spectral columns of
// models.py:150): a CTA owns one quarter (256) of the 1024 hidden features and walks pixel tiles of 128.
//   MMA1 (M=128, N=128, K=B)  hidden half-tile -> TMEM (ring of 3 accumulator slots)
//   epilogue                   bias + ReLU -> fp16, written back IN PLACE into the slot it came from (tcgen05.st): a thread
//                              packs the 64 fp32 columns it has read into the first 32 of them, i.e. the half-tile sits in
//                              columns [0,32) and [64,96) of the slot as a K-major A operand
//   MMA2 (M=128, N=NC, K=128)  classifier columns of those hidden features, A operand FROM TENSOR MEMORY, accumulated over
//                              both halves -> TMEM; its commit hands the slot back to MMA1 (NC = 16, or 32 for 17-32 classes)
//   readout                    part[quarter][pixel][NC] f32: the head adds the 4 quarter partials (53 MB at NC = 16 instead
//                              of the 425 MB hidden tensor written and read back)
// The hidden features touch neither HBM nor shared memory, whose space goes to the input-tile ring.
// NC = 32 (17-32 classes): MMA2 is N = 32, and a logits stage holds ONE 32-column accumulator in place of two of 16 --
// the 128 TMEM columns above the MMA1 ring keep four stages of 32 columns either way.
namespace spl {
constexpr int kEpi = 512, kThreads = kEpi + 96;      // warps 0-15 epilogue, warp 16 loader, warp 17 MMA1 issuer (+ TMEM), warp 18 MMA2 issuer
constexpr int kLoadWarp = kEpi / 32, kMmaWarp = kLoadWarp + 1, kMma2Warp = kLoadWarp + 2;
__host__ __device__ constexpr int wc_bytes(int NC) { return 32 * NC * 16; }   // classifier columns of this quarter: 32 k-chunks x NC classes x 16 B
constexpr int D2COL = 384;                           // TMEM: MMA1 ring at 0/128/256, 4 logits stages x 32 columns at 384..511
enum { A_FULL0 = 0, A_EMPTY0 = 4, D1_FULL0 = 8, D1_EMPTY0 = 11, H_FULL0 = 14, L_FULL0 = 20, L_EMPTY0 = 24, W_FULL = 28 };   // nA <= 4, 4 logits stages
}  // namespace spl

template <int NC>
__global__ void __launch_bounds__(spl::kThreads, 1)
spectral_logits_kernel(const __half* __restrict__ x16, int64_t mtiles, int KC, int nA,
                       const __half* __restrict__ w1t, const float* __restrict__ bspe,
                       const __half* __restrict__ wc_spe16, float* __restrict__ part) {
  using namespace spl;
  static_assert(NC == 16 || NC == 32, "spectral_logits: class width 16 or 32");
  constexpr int WCBYTES = wc_bytes(NC);
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t wbytes = uint32_t(KC) * 4096, abytes = uint32_t(KC) * 2048;
  const uint32_t S_W = 0, S_A = wbytes, S_WC = S_A + uint32_t(nA) * abytes, S_BIAS = S_WC + WCBYTES, S_BAR = S_BIAS + 1024,
                 S_TMEM = S_BAR + 256;
  const uint32_t bars = sbase + S_BAR;
  const int ntile = blockIdx.x & 3;
  const int64_t mt0 = blockIdx.x >> 2, mstep = gridDim.x >> 2;
  const int64_t my_tiles = mt0 < mtiles ? (mtiles - mt0 + mstep - 1) / mstep : 0;
  const uint32_t U = uint32_t(2 * my_tiles);           // units = (tile, hidden half)

  {
    float* sb = reinterpret_cast<float*>(smem + S_BIAS);
    if (tid < 256) sb[tid] = bspe[ntile * 256 + tid];
  }
  if (tid == 0) {
    mbar_init(bars + 8 * W_FULL, 1);
    fence_barrier_init();
    mbar_arrive_expect_tx(bars + 8 * W_FULL, wbytes + WCBYTES);   // this quarter's feat_spe rows and classifier columns
    const unsigned char* gw = reinterpret_cast<const unsigned char*>(w1t) + size_t(ntile) * wbytes;
    for (uint32_t o = 0; o < wbytes; o += 8192) bulk_g2s(sbase + S_W + o, gw + o, wbytes - o < 8192 ? wbytes - o : 8192, bars + 8 * W_FULL);
    bulk_g2s(sbase + S_WC, reinterpret_cast<const unsigned char*>(wc_spe16) + size_t(ntile) * WCBYTES, WCBYTES, bars + 8 * W_FULL);
    for (int i = 0; i < 4; ++i) { mbar_init(bars + 8 * (A_FULL0 + i), 1); mbar_init(bars + 8 * (A_EMPTY0 + i), 1); }
    // two epilogue groups of eight warps take alternate units; a slot goes MMA1 -> (D1_FULL) -> epilogue group ->
    // (H_FULL) -> MMA2 -> (D1_EMPTY) -> MMA1
    for (int i = 0; i < 3; ++i) { mbar_init(bars + 8 * (D1_FULL0 + i), 1); mbar_init(bars + 8 * (D1_EMPTY0 + i), 1); }
    for (int i = 0; i < 3; ++i) mbar_init(bars + 8 * (H_FULL0 + i), kEpi / 2);
    for (int i = 0; i < 4; ++i) { mbar_init(bars + 8 * (L_FULL0 + i), 1); mbar_init(bars + 8 * (L_EMPTY0 + i), 128); }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(sbase + S_TMEM, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);

  if (warp == kLoadWarp) {
    // ================================================================ loader: one bulk copy per pixel tile
    if (lane == 0) {
      [[maybe_unused]] uint32_t ntr = 0;
      for (uint32_t j = 0; j < uint32_t(my_tiles); ++j) {
        const uint32_t s = j % uint32_t(nA), ph = (j / uint32_t(nA)) & 1;
        mbar_wait(bars + 8 * (A_EMPTY0 + s), ph ^ 1, 91);
        CMLPL_TR(4, ntr, j);
        mbar_arrive_expect_tx(bars + 8 * (A_FULL0 + s), abytes);
        // one bulk copy moves ~6-7 GB/s however large it is: the tile goes as KC/2 copies of 4 KB in flight together
        const __half* src = x16 + (mt0 + int64_t(j) * mstep) * int64_t(KC) * 1024;
        for (int c = 0; c < KC / 2; ++c)
          bulk_g2s(sbase + S_A + s * abytes + c * 4096, src + c * 2048, 4096, bars + 8 * (A_FULL0 + s));
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA1 issuer
    if (tmem != 0) { printf("spectral_logits: unexpected TMEM base %u\n", tmem); __trap(); }
    constexpr uint64_t kHi = (uint64_t(128 >> 4) | (uint64_t(1) << 14)) << 32;
    constexpr uint32_t idesc1 = make_idesc_f16(128, 128);
    // gated by the input tile and by the slot's previous MMA2; runs up to the full ring (3 units) ahead
    mbar_wait(bars + 8 * W_FULL, 0, 90);                 // weights have landed
    [[maybe_unused]] uint32_t ntr = 0;
    for (uint32_t u = 0; u < U; ++u) {
      const uint32_t ti = u >> 1, hh = u & 1, d = u % 3, s = ti % uint32_t(nA);
      if (lane == 0) CMLPL_TR(0, ntr, u * 4);
      if (hh == 0) mbar_wait(bars + 8 * (A_FULL0 + s), (ti / uint32_t(nA)) & 1, 92);
      if (lane == 0) CMLPL_TR(0, ntr, u * 4 + 1);
      mbar_wait(bars + 8 * (D1_EMPTY0 + d), ((u / 3) & 1) ^ 1, 93);
      tc_fence_after();
      if (lane == 0) CMLPL_TR(0, ntr, u * 4 + 2);
      if (elect_one_sync()) {
        uint32_t a_lo = ((sbase + S_A + s * abytes) >> 4) | (uint32_t(2048 >> 4) << 16);
        uint32_t b_lo = ((sbase + S_W + hh * 2048) >> 4) | (uint32_t(4096 >> 4) << 16);
        for (int ks = 0; ks < KC / 2; ++ks) {
          umma_f16(d * 128, kHi | a_lo, kHi | b_lo, idesc1, ks ? 1u : 0u);
          a_lo += 4096 >> 4; b_lo += 8192 >> 4;
        }
        umma_commit(bars + 8 * (D1_FULL0 + d));
        if (hh == 1) umma_commit(bars + 8 * (A_EMPTY0 + s));
      }
      __syncwarp();
      if (lane == 0) CMLPL_TR(0, ntr, u * 4 + 3);
    }
  } else if (warp == kMma2Warp) {
    // ================================================================ MMA2 issuer: classifier columns over the hidden half-tiles (A from TMEM)
    constexpr uint64_t kHi = (uint64_t(128 >> 4) | (uint64_t(1) << 14)) << 32;
    constexpr uint32_t idesc2 = make_idesc_f16(128, NC);
    constexpr uint32_t kcb = NC * 16;                  // bytes per k-chunk of the classifier columns (LBO)
    mbar_wait(bars + 8 * W_FULL, 0, 90);
    [[maybe_unused]] uint32_t ntr = 0;
    for (uint32_t u = 0; u < U; ++u) {
      const uint32_t ti = u >> 1, hh = u & 1, d = u % 3, ls = ti & 3;
      if (lane == 0) CMLPL_TR(1, ntr, u * 4);
      mbar_wait(bars + 8 * (H_FULL0 + d), (u / 3) & 1, 94);
      if (hh == 0) mbar_wait(bars + 8 * (L_EMPTY0 + ls), ((ti >> 2) & 1) ^ 1, 95);
      tc_fence_after();
      if (lane == 0) CMLPL_TR(1, ntr, u * 4 + 2);
      if (elect_one_sync()) {
        uint32_t b_lo = ((sbase + S_WC + hh * 16 * kcb) >> 4) | (uint32_t(kcb >> 4) << 16);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          // k-step ks = hidden features 16 ks .. 16 ks + 15 of the half-tile = 8 packed columns; NC = 16: two independent
          // accumulators (even / odd k-steps), the readout adds them; NC = 32: one accumulator
          const uint32_t dcol = D2COL + ls * 32 + (NC == 16 ? (ks & 1) * 16 : 0);
          const uint32_t acc = NC == 16 ? (hh | (ks >> 1)) : (hh | ks);
          umma_f16_ta(dcol, d * 128 + (ks >> 2) * 64 + (ks & 3) * 8, kHi | b_lo, idesc2, acc ? 1u : 0u);
          b_lo += (2 * kcb) >> 4;
        }
        umma_commit(bars + 8 * (D1_EMPTY0 + d));
        if (hh == 1) umma_commit(bars + 8 * (L_FULL0 + ls));
      }
      __syncwarp();
      if (lane == 0) CMLPL_TR(1, ntr, u * 4 + 3);
    }
  } else {
    // ================================================================ epilogue (warps 0-15)
    // two groups of eight warps, group 0 takes the first hidden halves (even units), group 1 the second halves; a thread
    // owns one pixel row x 64 columns of the slot
    const int grp = warp >> 3, q = warp & 3, ch = (warp >> 2) & 1, L = q * 32 + lane;
    const uint32_t lane_addr = uint32_t(q * 32) << 16;
    const float* sb = reinterpret_cast<const float*>(smem + S_BIAS);
    auto readout = [&](uint32_t ti) {                  // partial logits of tile ti (four warps: one lane quarter each)
      const uint32_t ls = ti & 3;
      mbar_wait(bars + 8 * (L_FULL0 + ls), (ti >> 2) & 1, 96);
      tc_fence_after();
      float v[32];
      tmem_ld16(lane_addr + D2COL + ls * 32, v);
      tmem_ld16(lane_addr + D2COL + ls * 32 + 16, v + 16);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bars + 8 * (L_EMPTY0 + ls));
      if (NC == 16) {
#pragma unroll
        for (int c = 0; c < 16; ++c) v[c] += v[16 + c];
      }
      float4* dst = reinterpret_cast<float4*>(part) + ((int64_t(ntile) * mtiles + (mt0 + int64_t(ti) * mstep)) * 128 + L) * (NC / 4);
#pragma unroll
      for (int k = 0; k < NC / 4; ++k) dst[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    };
    [[maybe_unused]] uint32_t ntr = 0;
    const bool tracer = (warp & 7) == 0 && lane == 0;
    for (uint32_t u = uint32_t(grp); u < U; u += 2) {
      const uint32_t ti = u >> 1, hh = u & 1, d = u % 3;
      if (hh == 1 && ch == 0 && ti > 1) readout(ti - 2);      // deferred by two tiles (4 logits stages): its MMA2 has long completed
      if (tracer) CMLPL_TR(2 + grp, ntr, u * 4);
      mbar_wait(bars + 8 * (D1_FULL0 + d), (u / 3) & 1, 97);
      tc_fence_after();
      if (tracer) CMLPL_TR(2 + grp, ntr, u * 4 + 1);
      const float* bb = sb + hh * 128 + ch * 64;
      const uint32_t col0 = lane_addr + d * 128 + ch * 64;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        float v0[16], v1[16];
        tmem_ld16(col0 + g * 32, v0);
        tmem_ld16(col0 + g * 32 + 16, v1);
        tmem_ld_wait();
        uint32_t h[16];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const __half2 a = __floats2half2_rn(fmaxf(v0[2 * e] + bb[g * 32 + 2 * e], 0.f), fmaxf(v0[2 * e + 1] + bb[g * 32 + 2 * e + 1], 0.f));
          const __half2 b = __floats2half2_rn(fmaxf(v1[2 * e] + bb[g * 32 + 16 + 2 * e], 0.f),
                                              fmaxf(v1[2 * e + 1] + bb[g * 32 + 16 + 2 * e + 1], 0.f));
          h[e] = *reinterpret_cast<const uint32_t*>(&a);
          h[8 + e] = *reinterpret_cast<const uint32_t*>(&b);
        }
        tmem_st16u(col0 + g * 16, h);                    // packed pair c of the chunk -> column c: trails this thread's own reads
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(bars + 8 * (H_FULL0 + d));
      if (tracer) CMLPL_TR(2 + grp, ntr, u * 4 + 3);
    }
    if (grp == 1 && ch == 0) {
      if (my_tiles > 1) readout(uint32_t(my_tiles - 2));
      if (my_tiles > 0) readout(uint32_t(my_tiles - 1));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ------------------------------------------------------------------ head of the dense path: sums + argmax
// logits(p) = bc + sum over the 4 hidden quarters of part[q][p] + the 5 gathered conv partials M[I][r'+2I, c'] of pixel p
// (row maps of pool2_cls_kernel); first index wins ties (hyper_tools.py:426).  One thread per pixel:
// adjacent lanes read adjacent 16-byte quads of the two parity planes of a row.  NC = class width of part / lmap (16, 32).
template <int NC>
__global__ void __launch_bounds__(256)
head_sum_kernel(const float* __restrict__ part, int64_t mtiles, const float* __restrict__ lmap, int cols, int PR2, int PC2,
                int64_t n, int C, int ncell /* pooled rows: 5 (w = 20) or 2 (w = 11) */, const float* __restrict__ bc,
                const uint8_t* __restrict__ valid, uint8_t* __restrict__ labels, float* __restrict__ logits) {
  constexpr int NQ = NC / 4;                           // class quads per map entry
  const int64_t p = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (p >= n) return;
  const int nq = (C + 3) >> 2;                         // class quads that hold real classes
  float v[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) v[c] = 0.f;
  const int r = int(p / cols), c0 = int(p - int64_t(r) * cols);
  const int64_t psz = int64_t(PR2) * PC2;
  const float4* base = reinterpret_cast<const float4*>(lmap) + int64_t((r & 1) * 2 + (c0 & 1)) * 5 * NQ * psz +
                       int64_t(r >> 1) * PC2 + (c0 >> 1);
#pragma unroll
  for (int I = 0; I < 5; ++I) {
    if (I >= ncell) break;
    const float4* q = base + int64_t(I * NQ) * psz + (2 * I) * PC2;
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
      if (k < nq) {
        const float4 t = __ldg(q + int64_t(k) * psz);
        v[4 * k] += t.x; v[4 * k + 1] += t.y; v[4 * k + 2] += t.z; v[4 * k + 3] += t.w;
      }
    }
  }
#pragma unroll
  for (int qd = 0; qd < 4; ++qd) {
    const float4* s = reinterpret_cast<const float4*>(part) + (int64_t(qd) * mtiles * 128 + p) * NQ;
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
      if (k < nq) {
        const float4 t = __ldg(s + k);
        v[4 * k] += t.x; v[4 * k + 1] += t.y; v[4 * k + 2] += t.z; v[4 * k + 3] += t.w;
      }
    }
  }
  float best = -INFINITY; int arg = 0;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (c < C) {
      const float z = v[c] + __ldg(bc + c);
      if (logits) logits[p * C + c] = z;
      if (z > best) { best = z; arg = c; }
    }
  }
  labels[p] = (valid && !valid[p]) ? uint8_t(CMLPL_NODATA_LABEL) : uint8_t(arg);
}

}  // namespace cmlpl

using namespace cmlpl;

CMLPL_TRACE_EXPORT(cmlpl_debug_spl_trace)

namespace cmlpl {

// shared-memory plan of spectral_logits_kernel for KC input k-chunks and class width NC: as many input tiles in flight as
// fit (<= 4).  224 bands (KC = 28) leave room for one at either width.
static bool spectral_logits_plan(int KC, int NC, int* nA, size_t* smem) {
  for (int a = 4; a >= 1; --a) {
    const size_t b = size_t(KC) * 4096 + size_t(a) * KC * 2048 + spl::wc_bytes(NC) + 1024 + 256 + 64;
    if (b <= 232448) { *nA = a; *smem = b; return true; }
  }
  return false;
}

// x16_tile(_raw) + spectral_logits_kernel: x16 is scratch for the fp16 input tiles, part f32 [4][ceil(n/128)*128][NC].
// dtype: -1 = preprocessed f32 spectra, else the raw sample type (CMLPL_RAW_U16 / F32 / I16); bm: band-major raw rows, or
// nullptr for pixel-major [n][B]; valid: u8 [n] of the raw rows (no-data pixels convert to zero rows), or nullptr
int launch_spectral_logits(const void* x, int dtype, const BandMajor* bm, int64_t n, int num_features, int num_classes,
                           int w, const float* mu, const float* inv_sigma, const uint8_t* valid, const void* packed,
                           void* x16, float* part, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(x && packed && x16 && part, "spectral_logits_tc: null pointer");
  CMLPL_CHECK_ARG(n > 0 && num_features > 0, "spectral_logits_tc: bad dims");
  CMLPL_CHECK_ARG(num_classes <= 32, "spectral_logits_tc: needs <= 32 classes, got %d", num_classes);
  const PackedLayout L = packed_layout(num_features, num_classes, w);
  const int KC = L.kc_spe_in;
  int nA = 0; size_t smem = 0;
  CMLPL_CHECK_ARG(spectral_logits_plan(KC, L.nc, &nA, &smem), "spectral_logits_tc: %d bands do not fit shared memory", num_features);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t mtiles = (n + 127) / 128, total = mtiles * KC * 128;
  int64_t g = (total + 255) / 256; const int64_t cap = int64_t(sm_count()) * 16; if (g > cap) g = cap;
  __half* o = static_cast<__half*>(x16);
  if (dtype < 0)
    x16_tile_kernel<<<int(g), 256, 0, s>>>(static_cast<const float*>(x), n, num_features, KC, total, o);
  else if (bm && dtype == CMLPL_RAW_U16)
    x16_tile_raw_bm_kernel<uint16_t><<<int(g), 256, 0, s>>>(static_cast<const uint16_t*>(x), *bm, n, num_features, KC, total, mu, inv_sigma, valid, o);
  else if (bm && dtype == CMLPL_RAW_I16)
    x16_tile_raw_bm_kernel<int16_t><<<int(g), 256, 0, s>>>(static_cast<const int16_t*>(x), *bm, n, num_features, KC, total, mu, inv_sigma, valid, o);
  else if (bm)
    x16_tile_raw_bm_kernel<float><<<int(g), 256, 0, s>>>(static_cast<const float*>(x), *bm, n, num_features, KC, total, mu, inv_sigma, valid, o);
  else if (dtype == CMLPL_RAW_U16)
    x16_tile_raw_kernel<uint16_t><<<int(g), 256, 0, s>>>(static_cast<const uint16_t*>(x), n, num_features, KC, total, mu, inv_sigma, valid, o);
  else if (dtype == CMLPL_RAW_I16)
    x16_tile_raw_kernel<int16_t><<<int(g), 256, 0, s>>>(static_cast<const int16_t*>(x), n, num_features, KC, total, mu, inv_sigma, valid, o);
  else
    x16_tile_raw_kernel<float><<<int(g), 256, 0, s>>>(static_cast<const float*>(x), n, num_features, KC, total, mu, inv_sigma, valid, o);
  CMLPL_CHECK_LAUNCH("x16_tile");
  int grid = sm_count() / 4 * 4;
  if (grid > mtiles * 4) grid = int(mtiles * 4);
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const __half* w1s = reinterpret_cast<const __half*>(pk + L.w1s);
  const float* bspe = reinterpret_cast<const float*>(pk + L.bspe);
  const __half* wc_spe16 = reinterpret_cast<const __half*>(pk + L.wc16 + size_t(L.conv_pos) * 8 * L.nc * 16);
  if (L.nc == 16) {
    CMLPL_MAX_DYN_SMEM(spectral_logits_kernel<16>, int(smem));
    spectral_logits_kernel<16><<<grid, spl::kThreads, smem, s>>>(static_cast<const __half*>(x16), mtiles, KC, nA, w1s, bspe,
                                                                 wc_spe16, part);
  } else {
    CMLPL_MAX_DYN_SMEM(spectral_logits_kernel<32>, int(smem));
    spectral_logits_kernel<32><<<grid, spl::kThreads, smem, s>>>(static_cast<const __half*>(x16), mtiles, KC, nA, w1s, bspe,
                                                                 wc_spe16, part);
  }
  CMLPL_CHECK_LAUNCH("spectral_logits");
  return CMLPL_OK;
}

}  // namespace cmlpl

// Fused spectral branch of the dense path: part f32 [4 hidden quarters][ceil(n/128)*128][NC] partial spectral logits, NC =
// 16 for <= 16 classes and 32 for 17-32 (spectral_logits_kernel; the 1024 hidden features stay on chip).  x16 is
// scratch for the fp16 input tiles.
extern "C" int cmlpl_spectral_logits_tc(const float* spectra, int64_t n, int num_features, int num_classes, int w,
                                        const void* packed, void* x16, float* part, cmlpl_stream_t stream) {
  return launch_spectral_logits(spectra, -1, nullptr, n, num_features, num_classes, w, nullptr, nullptr, nullptr, packed, x16,
                                part, stream);
}

namespace cmlpl {

// head_sum_kernel over the band's pixels; valid: u8 [band_rows * cols] (no-data pixels get CMLPL_NODATA_LABEL) or nullptr
int launch_head_sum(const float* part, const float* lmap, int cols, int band_rows, int num_features, int num_classes, int w,
                    const void* packed, const uint8_t* valid, uint8_t* labels, float* logits, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(part && lmap && packed && labels, "head_sum_lmap: null pointer");
  CMLPL_CHECK_ARG((w == 20 || w == 11) && cols > 0 && band_rows > 0, "head_sum_lmap: bad dims (w must be 20 or 11)");
  CMLPL_CHECK_ARG(num_classes > 0 && num_classes <= 32, "head_sum_lmap: needs 1..32 classes, got %d", num_classes);
  const PackedLayout L = packed_layout(num_features, num_classes, w);
  const int64_t n = int64_t(band_rows) * cols, mtiles = (n + 127) / 128;
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const unsigned grid = unsigned((n + 255) / 256);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int PR2 = (band_rows + w) / 2, PC2 = (cols + w) / 2, ncell = w == 20 ? 5 : 2;
  const float* bc = reinterpret_cast<const float*>(pk + L.bc);
  if (L.nc == 16)
    head_sum_kernel<16><<<grid, 256, 0, s>>>(part, mtiles, lmap, cols, PR2, PC2, n, num_classes, ncell, bc, valid, labels, logits);
  else
    head_sum_kernel<32><<<grid, 256, 0, s>>>(part, mtiles, lmap, cols, PR2, PC2, n, num_classes, ncell, bc, valid, labels, logits);
  CMLPL_CHECK_LAUNCH("head_sum");
  return CMLPL_OK;
}

}  // namespace cmlpl

// Head of the dense path without a GEMM: quarter partials of cmlpl_spectral_logits_tc + the 5 gathered conv partials
// per pixel from lmap (cmlpl_pool2_cls_f16) + bias, argmax.  Pixels are the band's raster order.
extern "C" int cmlpl_head_sum_lmap(const float* part, const float* lmap, int cols, int band_rows, int num_features,
                                   int num_classes, int w, const void* packed, uint8_t* labels, float* logits,
                                   cmlpl_stream_t stream) {
  return launch_head_sum(part, lmap, cols, band_rows, num_features, num_classes, w, packed, nullptr, labels, logits, stream);
}
