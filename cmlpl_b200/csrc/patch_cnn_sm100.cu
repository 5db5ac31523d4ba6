// patch_cnn: conv1 -> (+res, ReLU, 2x2 avg-pool) -> conv2 -> (+res, ReLU, 2x2 avg-pool)
// for every pixel's w x w window of the conv0 map (tools/models.py:133-140 applied to the
// patch hyper_tools.py:226-243 would have materialised).  sm_100a only: tcgen05.mma
// (kind::f16, fp16 operands = TF32's 11-bit significand, fp32 accumulate in TMEM).
//
// Persistent kernel, one CTA per SM, warp-specialised:
//   warps 0-7   epilogue  (TMEM -> registers: bias + residual + ReLU + pool -> next stage);
//               warp w reads TMEM lane quadrant w%4 and the 32 output channels of half w/4
//   warps 8-9   loaders   (cp.async 16 B straight into the zero-padded parity planes: 8 pixels x 8
//               channel chunks per step; the (row, column) pattern repeats every two window rows,
//               so per-thread offsets are computed once)
//   warp  10    MMA issuer (one elected lane) + TMEM allocator
//
// Implicit GEMM without im2col: activations live in shared memory in the UMMA "no swizzle,
// K-major" canonical layout with SBO = 128 B, i.e. for every 16-byte K-chunk (8 channels) a
// *linear* array of positions, 16 B apart.  A 3x3 tap is then nothing but a different start
// address of the A descriptor (row-major positions with a zero-padded border), so the nine
// taps x four K-steps of a tile are back-to-back tcgen05.mma (M=128, K=16) on the same buffer
// (taps that read the same rows for the even- and odd-row tile are fused into N=128 MMAs).  Rows are split by parity into two planes (even rows / odd rows) so that the
// two rows of every 2x2 pooling window land in the SAME TMEM lane of two accumulator tiles
// and the two columns in adjacent lanes: pooling is one add + one shfl_xor in the epilogue.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "conv_pair_issue.cuh"
#include "train_common.cuh"
#include "train_kernels.cuh"

namespace cmlpl {

template <int W>
struct PatchCfg {
  // W = 20: the reference's window (tools/models.py:127 fixes 2624 classifier inputs).  Odd W (W = 11, BASELINE
  // configs[4]) follows ExtractPatches_for_base (hyper_tools.py:300-317) and the floor semantics of avg_pool2d: the
  // last row / column of an odd map feeds the convolution taps of its neighbours but no pooling window.
  // Padded row widths are EVEN so that the two columns of a pooling window are lanes L and L^1 of a tile.
  // ---- conv1 input: W x W, parity planes of (W/2+1) rows x PW1 padded columns
  static constexpr int H1 = W;
  static constexpr int NP1 = W / 2;                 // output row pairs (= pooled rows)
  static constexpr int PW1 = (W + 3) & ~1;
  static constexpr int PR1 = W / 2 + 1;
  static constexpr int ENT1 = 1 + PR1 * PW1;        // +1 leading zero entry (x = -1 of row 0)
  static constexpr int CH1 = ENT1 * 16;             // bytes between 16-B K-chunks (= LBO)
  static constexpr int PLANE1 = 8 * CH1;
  static constexpr int M1 = NP1 * PW1;              // outputs per parity
  static constexpr int NT1 = (M1 + 127) / 128;      // 128-row tiles per parity
  // ---- conv2 input: W/2 x W/2
  static constexpr int H2 = W / 2;
  static constexpr int NP2 = H2 / 2;
  static constexpr int PW2 = (H2 + 3) & ~1;
  static constexpr int PR2 = H2 / 2 + 1;
  static constexpr int ENT2 = 1 + PR2 * PW2;
  static constexpr int CH2 = ENT2 * 16;
  static constexpr int PLANE2 = 8 * CH2;
  static constexpr int M2 = NP2 * PW2;
  static_assert(M2 <= 128, "conv2 parity plane must fit one tile");
  static constexpr int P = NP2 * NP2;               // pooled positions written per pixel
  // ---- TMEM columns (fp32 accumulators, 64 per tile)
  static constexpr int TM_C1 = 0;                   // (half h, parity q) -> (h*2+q)*64
  static constexpr int TM_C2 = NT1 * 2 * 64;        // parity q -> TM_C2 + q*64
  static constexpr int TM_COLS = 512;
  static_assert(TM_C2 + 128 <= TM_COLS, "TMEM budget");
  // ---- shared memory map (bytes)
  static constexpr int WBYTES = 9 * 8 * 64 * 8 * 2;  // one conv's weights, 73 728 B
  static constexpr int S_W1 = 0;
  static constexpr int S_W2 = S_W1 + WBYTES;
  static constexpr int S_A2 = S_W2 + WBYTES;
  static constexpr int S_A1 = S_A2 + 2 * PLANE2;
  static constexpr int S_BIAS = S_A1 + 2 * PLANE1;   // b1[64] b2[64] f32
  static constexpr int S_BAR = S_BIAS + 512;         // 16 mbarriers
  static constexpr int S_TMEM = S_BAR + 128;         // tmem base address
  // the last 128-row tile reads up to entry 128*NT1-1 + PW1+1 (+1 leading) of a chunk plane;
  // whatever lies beyond ENT1 only feeds discarded output rows but must be mapped memory.
  static constexpr int OVER1 = (128 * NT1 + PW1 + 2 - ENT1) * 16;
  static constexpr int S_END0 = S_TMEM + 16;
  static constexpr int S_END = (S_A1 + 2 * PLANE1 + (OVER1 > 0 ? OVER1 : 0)) > S_END0
                                   ? (S_A1 + 2 * PLANE1 + (OVER1 > 0 ? OVER1 : 0)) : S_END0;
  static constexpr int SMEM = (S_END + 127) / 128 * 128;
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
};

enum { BAR_A1_FULL = 0, BAR_A1_EMPTY, BAR_C1_FULL0, BAR_C1_FULL1, BAR_C1_EMPTY0, BAR_C1_EMPTY1,
       BAR_A2_FULL, BAR_C2_FULL, BAR_C2_EMPTY, BAR_COUNT };

constexpr int kEpiThreads = 256, kLoadThreads = 64, kThreads = kEpiThreads + kLoadThreads + 32;
constexpr int kEpiWarps = kEpiThreads / 32, kLoadWarp0 = kEpiWarps, kMmaWarp = kEpiWarps + kLoadThreads / 32;

// TRAIN = the forward trunk of the fused training step (tools/models.py:133-140 in batch mode): every "pixel" is one
// sample of one of the two BaseNet2 peers whose conv0 output a0 [8 chunks][W x W][8] lies in the workspace.  The CTAs
// are split between the nets (each keeps ONE net's weights, converted from the fp32 parameters in the prologue) and
// the epilogues additionally save what the backward pass needs: the ReLU masks of both blocks as bits, the pooled
// conv1 output p1 (B operand of conv2's weight gradient) and the pooled conv2 output as fp32 in the classifier's
// flatten order (tools/models.py:141).
template <int W, bool TRAIN>
__global__ void __launch_bounds__(kThreads, 1)
patch_cnn_kernel(const __half* __restrict__ f0pad, int cols, int band_rows,
                 const unsigned char* __restrict__ packed_w1, const unsigned char* __restrict__ packed_w2,
                 const float* __restrict__ b1g, const float* __restrict__ b2g, __half* __restrict__ p2out,
                 TrainCnnArgs ta) {
  using Cfg = PatchCfg<W>;
  using G = TrainGeom<W>;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + Cfg::S_BAR;
  float* sbias = reinterpret_cast<float*>(smem + Cfg::S_BIAS);
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + Cfg::S_TMEM);

  // TRAIN: the grid is split evenly between the two nets; p runs over the GLOBAL sample index net*nb + row
  const int cpn = TRAIN ? int(gridDim.x >> 1) : 1;
  const int net = TRAIN ? int(blockIdx.x) / cpn : 0;
  const int64_t npix = TRAIN ? int64_t(ta.nb) : int64_t(band_rows) * cols;
  const int64_t nctas = TRAIN ? cpn : gridDim.x;
  const int64_t cta = TRAIN ? int(blockIdx.x) - net * cpn : blockIdx.x;
  const int64_t per = (npix + nctas - 1) / nctas;
  const int64_t p_lo = cta * per;
  const int64_t p_begin = (TRAIN ? int64_t(net) * ta.nb : 0) + (p_lo < npix ? p_lo : npix);
  const int64_t p_end = (TRAIN ? int64_t(net) * ta.nb : 0) + ((p_lo + per < npix) ? p_lo + per : npix);
  const int pitch = TRAIN ? W : cols + W - 1;   // padded map width in pixels
  const int plane_rows = TRAIN ? W : band_rows + W - 1;   // padded map height (rows per chunk plane)

  // ---------------------------------------------------------------- one-time setup
  if constexpr (TRAIN) {
    // this net's fp16 forward packs [3 dx][8 kchunks][192 rows][8 ci] (written by train_conv0_kernel this step)
    packed_w1 = ta.wpack + size_t(net * 2 + 0) * 2 * kWPackBytes;
    packed_w2 = ta.wpack + size_t(net * 2 + 1) * 2 * kWPackBytes;
  }
  {    // weights -> smem (already in UMMA layout), zero the activation planes, biases
    const uint4* g1 = reinterpret_cast<const uint4*>(packed_w1);
    const uint4* g2 = reinterpret_cast<const uint4*>(packed_w2);
    uint4* s1 = reinterpret_cast<uint4*>(smem + Cfg::S_W1);
    uint4* s2 = reinterpret_cast<uint4*>(smem + Cfg::S_W2);
    for (int i = tid; i < Cfg::WBYTES / 16; i += kThreads) { s1[i] = __ldg(g1 + i); s2[i] = __ldg(g2 + i); }
    uint4* z = reinterpret_cast<uint4*>(smem + Cfg::S_A2);
    const int zn = (Cfg::SMEM - Cfg::S_A2) / 16;
    for (int i = tid; i < zn; i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  __syncthreads();
  if constexpr (TRAIN) { b1g = ta.b1[net]; b2g = ta.b2[net]; }
  if (tid < 64) { sbias[tid] = b1g[tid]; sbias[64 + tid] = b2g[tid]; }
  if (tid == 0) {
    mbar_init(bars + 8 * BAR_A1_FULL, kLoadThreads);
    mbar_init(bars + 8 * BAR_A1_EMPTY, 1 + kEpiThreads);   // conv1 MMAs done + residuals read
    mbar_init(bars + 8 * BAR_C1_FULL0, 1);
    mbar_init(bars + 8 * BAR_C1_FULL1, 1);
    mbar_init(bars + 8 * BAR_C1_EMPTY0, kEpiThreads);
    mbar_init(bars + 8 * BAR_C1_EMPTY1, kEpiThreads);
    mbar_init(bars + 8 * BAR_A2_FULL, kEpiThreads);
    mbar_init(bars + 8 * BAR_C2_FULL, 1);
    mbar_init(bars + 8 * BAR_C2_EMPTY, kEpiThreads);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(sbase + Cfg::S_TMEM, Cfg::TM_COLS);
  fence_proxy_async();   // weights / zeros written through the generic proxy, read by the MMA (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp >= kLoadWarp0 && warp < kMmaWarp) {
    // ================================================================ LOADERS
    // F0 is chunk-planar in HBM ([8 chunks][rows][cols][8 halves]).  64 threads = 8 chunks x 8 pixels per
    // step; 5 steps cover two window rows (40 pixels) and the pattern repeats for each of the W/2 row
    // pairs: global += 2 rows, both planes += one plane row.  Per-thread offsets are computed once.
    constexpr bool kPairs = (W % 2 == 0) && ((2 * W) % 8 == 0);     // row-pair pattern (W = 20)
    constexpr int STEPS = kPairs ? 2 * W / 8 : (W * W + 7) / 8;     // otherwise: the whole window, 8 pixels per step
    const int lt = tid - kEpiThreads;                        // 0..63
    const int lch = lt >> 3, lpx = lt & 7;
    int64_t goff[STEPS];                                     // halves, relative to the window origin of chunk 0
    uint32_t soff[STEPS];                                    // smem byte address (row pair 0 in the pair pattern)
#pragma unroll
    for (int st = 0; st < STEPS; ++st) {
      const int pix = st * 8 + lpx;                          // 0 .. 2W-1 within the row pair, or 0 .. W*W-1
      const int y = pix / W, x = pix - y * W;
      goff[st] = ((int64_t(lch) * plane_rows + y) * pitch + x) * 8;
      // window row y -> plane y&1, plane row (y + (y&1)) / 2: even plane row g holds y = 2g, odd plane row g+1 holds 2g+1
      soff[st] = sbase + Cfg::S_A1 + (y & 1) * Cfg::PLANE1 + lch * Cfg::CH1 + (1 + ((y + (y & 1)) >> 1) * Cfg::PW1 + x) * 16;
    }
    uint32_t ph = 0;
    for (int64_t p = p_begin; p < p_end; ++p, ph ^= 1) {
      const __half* src;
      if constexpr (TRAIN) {
        src = ta.a0 + p * int64_t(G::ActBytes / 2);
      } else {
        const int rb = int(p / cols), c = int(p - int64_t(rb) * cols);
        src = f0pad + (int64_t(rb) * pitch + c) * 8;
      }
      mbar_wait(bars + 8 * BAR_A1_EMPTY, ph ^ 1, 1);         // conv1 MMAs + residual reads of the previous patch done
      // hold the copies back until the previous patch's conv1 epilogue has finished: the LSU queue is
      // shared with the epilogue's shared-memory traffic, and the load still hides under conv2
      if (p > p_begin) mbar_wait(bars + 8 * BAR_A2_FULL, ph ^ 1, 10);
      if constexpr (kPairs) {
#pragma unroll
        for (int g = 0; g < W / 2; ++g) {
#pragma unroll
          for (int st = 0; st < STEPS; ++st)
            cp_async16(soff[st] + g * Cfg::PW1 * 16, src + goff[st] + int64_t(2 * g) * pitch * 8);
        }
      } else {
#pragma unroll
        for (int st = 0; st < STEPS; ++st)
          if (st * 8 + lpx < W * W) cp_async16(soff[st], src + goff[st]);
      }
      cp_async_wait_all();
      fence_proxy_async();                                   // generic-proxy writes -> visible to the MMA
      mbar_arrive(bars + 8 * BAR_A1_FULL);
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA ISSUER
    // The whole warp walks the protocol (so every address stays warp-uniform); one elected lane
    // issues the MMAs and the commits.  A 512-column allocation necessarily starts at column 0.
    if (tmem != 0) { printf("patch_cnn: unexpected TMEM base %u\n", tmem); __trap(); }
    const uint32_t a1_lo = ((sbase + Cfg::S_A1 + 16) >> 4) | (uint32_t(Cfg::CH1 >> 4) << 16);
    const uint32_t a2_lo = ((sbase + Cfg::S_A2 + 16) >> 4) | (uint32_t(Cfg::CH2 >> 4) << 16);
    const uint32_t w1_lo = ((sbase + Cfg::S_W1) >> 4) | (uint32_t(kWLbo >> 4) << 16);
    const uint32_t w2_lo = ((sbase + Cfg::S_W2) >> 4) | (uint32_t(kWLbo >> 4) << 16);
    uint32_t ph = 0;
    for (int64_t p = p_begin; p < p_end; ++p, ph ^= 1) {
      mbar_wait(bars + 8 * BAR_A1_FULL, ph, 2);
      // ---- conv1: NT1 halves x 2 parities
#pragma unroll
      for (int h = 0; h < Cfg::NT1; ++h) {
        mbar_wait(bars + 8 * (BAR_C1_EMPTY0 + h), ph ^ 1, 3);     // epilogue drained this half (prev patch)
        tc_fence_after();
        if (elect_one_sync()) {
          issue_conv_pair<Cfg::PW1, Cfg::CH1, Cfg::PLANE1>(Cfg::TM_C1 + h * 128, a1_lo + h * 128, w1_lo);
          umma_commit(bars + 8 * (BAR_C1_FULL0 + h));
          if (h == Cfg::NT1 - 1) umma_commit(bars + 8 * BAR_A1_EMPTY);   // every conv1 read of A1 has completed
        }
        __syncwarp();
      }
      // ---- conv2: 2 parities, one 128-row tile each
      mbar_wait(bars + 8 * BAR_A2_FULL, ph, 4);
      mbar_wait(bars + 8 * BAR_C2_EMPTY, ph ^ 1, 5);
      tc_fence_after();
      if (elect_one_sync()) {
        issue_conv_pair<Cfg::PW2, Cfg::CH2, Cfg::PLANE2>(Cfg::TM_C2, a2_lo, w2_lo);
        umma_commit(bars + 8 * BAR_C2_FULL);
      }
      __syncwarp();
    }
  } else {
    // ================================================================ EPILOGUE (warps 0-7)
    const int L = (warp & 3) * 32 + lane;                    // TMEM lane == row of the tile
    const int chalf = warp >> 2;                             // which 32 output channels this warp handles
    const uint32_t lane_addr = tmem + (uint32_t((warp & 3) * 32) << 16) + chalf * 32;
    const float* bias1 = sbias + chalf * 32;
    const float* bias2 = sbias + 64 + chalf * 32;
    uint32_t ph = 0;
    // bias + residual + ReLU on both rows of the pooling window, sum, add the horizontal neighbour
    uint32_t mbits_e = 0, mbits_o = 0;   // TRAIN: ReLU masks (even / odd row of the pooling window), 16 bits per call
    float pooled[16];                    // TRAIN reads the fp32 pooled values of the last call
    auto pool16 = [&](const float* e, const float* o, const uint4* re, const uint4* ro, const float* bias,
                      uint4& out_lo, uint4& out_hi) {
      const __half2* he = reinterpret_cast<const __half2*>(re);
      const __half2* ho = reinterpret_cast<const __half2*>(ro);
      mbits_e = 0; mbits_o = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float2 fe = __half22float2(he[j]), fo = __half22float2(ho[j]);
        const float b0 = bias[2 * j], b1 = bias[2 * j + 1];
        const float e0 = e[2 * j] + b0 + fe.x, o0 = o[2 * j] + b0 + fo.x;
        const float e1 = e[2 * j + 1] + b1 + fe.y, o1 = o[2 * j + 1] + b1 + fo.y;
        if constexpr (TRAIN) {
          mbits_e |= (e0 > 0.f ? 1u : 0u) << (2 * j) | (e1 > 0.f ? 1u : 0u) << (2 * j + 1);
          mbits_o |= (o0 > 0.f ? 1u : 0u) << (2 * j) | (o1 > 0.f ? 1u : 0u) << (2 * j + 1);
        }
        pooled[2 * j] = fmaxf(e0, 0.f) + fmaxf(o0, 0.f);
        pooled[2 * j + 1] = fmaxf(e1, 0.f) + fmaxf(o1, 0.f);
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) pooled[j] = (pooled[j] + __shfl_xor_sync(0xffffffffu, pooled[j], 1)) * 0.25f;
      __half2 hv[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) hv[j] = __floats2half2_rn(pooled[2 * j], pooled[2 * j + 1]);
      out_lo = *reinterpret_cast<uint4*>(&hv[0]);
      out_hi = *reinterpret_cast<uint4*>(&hv[4]);
    };
    for (int64_t p = p_begin; p < p_end; ++p, ph ^= 1) {
      if constexpr (TRAIN && (W & 1)) {
        // floor pooling drops the last row / column of both maps: no gradient reaches them, so their ReLU mask bits
        // are stored as 0 (m1: 2W-1 positions, m2: 2*H2-1 positions, two words each)
        if (tid < 2 * (2 * W - 1)) {
          const int k = tid >> 1, y = k < W ? W - 1 : k - W, x = k < W ? k : W - 1;
          ta.m1[(p * G::TPos + y * W + x) * 2 + (tid & 1)] = 0u;
        }
        if (tid < 2 * (2 * Cfg::H2 - 1)) {
          const int k = tid >> 1, y = k < Cfg::H2 ? Cfg::H2 - 1 : k - Cfg::H2, x = k < Cfg::H2 ? k : Cfg::H2 - 1;
          ta.m2[(p * G::TPos2 + y * Cfg::H2 + x) * 2 + (tid & 1)] = 0u;
        }
      }
      mbar_wait(bars + 8 * BAR_A1_FULL, ph, 9);             // the residuals are read back from A1
      // ------------------------------------------------ conv1 epilogue -> A2 (pooled, fp16)
#pragma unroll 1
      for (int h = 0; h < Cfg::NT1; ++h) {
        const int m = h * 128 + L;
        const int i = m / Cfg::PW1, x = m - i * Cfg::PW1;
        const bool valid = (m < Cfg::M1) && (x < 2 * Cfg::NP1);
        const bool writer = valid && ((x & 1) == 0);
        // residual = conv0 output at the same position (models.py:133,135), rows 2i and 2i+1: read it
        // back from the A1 planes (same fp16 values the MMA consumes) before waiting for the
        // accumulators.  A1 is stable until the loader is released, and the loader's release needs
        // this thread's arrival below (after the last half's residual is in registers).
        uint4 re[4], ro[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { re[k] = make_uint4(0, 0, 0, 0); ro[k] = make_uint4(0, 0, 0, 0); }
        if (valid) {
          const unsigned char* rE = smem + Cfg::S_A1 + (chalf * 4) * Cfg::CH1 + (1 + i * Cfg::PW1 + x) * 16;
          const unsigned char* rO = smem + Cfg::S_A1 + Cfg::PLANE1 + (chalf * 4) * Cfg::CH1 +
                                    (1 + (i + 1) * Cfg::PW1 + x) * 16;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            re[k] = *reinterpret_cast<const uint4*>(rE + k * Cfg::CH1);
            ro[k] = *reinterpret_cast<const uint4*>(rO + k * Cfg::CH1);
          }
        }
        if (h == Cfg::NT1 - 1) {
          // make sure the loads have landed (consume them) before telling the loader A1 may be rewritten
          uint32_t sink = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) sink |= re[k].x ^ ro[k].w;
          asm volatile("" ::"r"(sink) : "memory");
          mbar_arrive(bars + 8 * BAR_A1_EMPTY);
        }
        // destination in the conv2 planes: pooled pixel (py=i, px=x/2), chunks chalf*4 .. chalf*4+3
        const int q2 = i & 1, prow2 = (i + q2) >> 1;
        unsigned char* dst = smem + Cfg::S_A2 + q2 * Cfg::PLANE2 + (chalf * 4) * Cfg::CH2 +
                             (1 + prow2 * Cfg::PW2 + (x >> 1)) * 16;
        mbar_wait(bars + 8 * (BAR_C1_FULL0 + h), ph, 6);
        tc_fence_after();
        // two 16-channel groups one after the other keeps only 32 accumulators live
        float e[16], o[16];
        uint4 w0, w1;
        tmem_ld16(lane_addr + Cfg::TM_C1 + (h * 2 + 0) * 64, e);
        tmem_ld16(lane_addr + Cfg::TM_C1 + (h * 2 + 1) * 64, o);
        tmem_ld_wait();
        pool16(e, o, &re[0], &ro[0], bias1, w0, w1);
        if (writer) {
          *reinterpret_cast<uint4*>(dst) = w0;
          *reinterpret_cast<uint4*>(dst + Cfg::CH2) = w1;
        }
        uint32_t me = mbits_e, mo = mbits_o;
        unsigned char* p1g = nullptr;
        if constexpr (TRAIN) {
          // pooled conv1 output of this sample: p1 [8 chunks][(W/2)x(W/2)][8]
          p1g = reinterpret_cast<unsigned char*>(ta.p1) + p * int64_t(G::Act2Bytes) + (chalf * 4) * (G::TPos2 * 16) +
                (i * (W / 2) + (x >> 1)) * 16;
          if (writer) {
            *reinterpret_cast<uint4*>(p1g) = w0;
            *reinterpret_cast<uint4*>(p1g + G::TPos2 * 16) = w1;
          }
        }
        tmem_ld16(lane_addr + Cfg::TM_C1 + (h * 2 + 0) * 64 + 16, e);
        tmem_ld16(lane_addr + Cfg::TM_C1 + (h * 2 + 1) * 64 + 16, o);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(bars + 8 * (BAR_C1_EMPTY0 + h));         // accumulators are in registers: free the tiles
        pool16(e, o, &re[2], &ro[2], bias1 + 16, w0, w1);
        if (writer) {
          *reinterpret_cast<uint4*>(dst + 2 * Cfg::CH2) = w0;
          *reinterpret_cast<uint4*>(dst + 3 * Cfg::CH2) = w1;
        }
        if constexpr (TRAIN) {
          if (writer) {
            *reinterpret_cast<uint4*>(p1g + 2 * G::TPos2 * 16) = w0;
            *reinterpret_cast<uint4*>(p1g + 3 * G::TPos2 * 16) = w1;
          }
          if (valid) {   // m1 [sample][y][x][half]: bit c%32 of word c/32 = (a1[c][y][x] > 0), rows y = 2i, 2i+1
            uint32_t* mg = ta.m1 + (p * G::TPos + (2 * i) * W + x) * 2 + chalf;
            mg[0] = me | (mbits_e << 16);
            mg[2 * W] = mo | (mbits_o << 16);
          }
        }
      }
      fence_proxy_async();
      mbar_arrive(bars + 8 * BAR_A2_FULL);
      mbar_wait(bars + 8 * BAR_A2_FULL, ph, 7);              // every epilogue thread's A2 writes are visible
      // ------------------------------------------------ conv2 epilogue -> P2 (global, fp16)
      {
        const int m = L;
        const int i = m / Cfg::PW2, x = m - i * Cfg::PW2;
        const bool valid = (m < Cfg::M2) && (x < 2 * Cfg::NP2);
        const bool writer = valid && ((x & 1) == 0);
        // residual = pooled conv1 output (models.py:137,139): rows 2i (even plane row i), 2i+1 (odd plane row i+1)
        uint4 re[4], ro[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { re[k] = make_uint4(0, 0, 0, 0); ro[k] = make_uint4(0, 0, 0, 0); }
        if (valid) {
          const unsigned char* rE = smem + Cfg::S_A2 + (chalf * 4) * Cfg::CH2 + (1 + i * Cfg::PW2 + x) * 16;
          const unsigned char* rO = smem + Cfg::S_A2 + Cfg::PLANE2 + (chalf * 4) * Cfg::CH2 +
                                    (1 + (i + 1) * Cfg::PW2 + x) * 16;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            re[k] = *reinterpret_cast<const uint4*>(rE + k * Cfg::CH2);
            ro[k] = *reinterpret_cast<const uint4*>(rO + k * Cfg::CH2);
          }
        }
        // row-major [pixel][pos][64]
        const int pos = i * Cfg::NP2 + (x >> 1);
        __half* dst = p2out + (p * Cfg::P + pos) * 64 + chalf * 32;
        mbar_wait(bars + 8 * BAR_C2_FULL, ph, 8);
        tc_fence_after();
        float e[16], o[16];
        uint4 w0, w1;
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        tmem_ld16(lane_addr + Cfg::TM_C2 + 0 * 64, e);
        tmem_ld16(lane_addr + Cfg::TM_C2 + 1 * 64, o);
        tmem_ld_wait();
        pool16(e, o, &re[0], &ro[0], bias2, w0, w1);
        uint32_t me = mbits_e, mo = mbits_o;
        float* catg = nullptr;
        if constexpr (TRAIN) {
          // flatten order of tools/models.py:141: feature = channel * P + pooled position (P = 25, or 4 at W = 11)
          catg = ta.cat + p * int64_t(G::CatDim) + (chalf * 32) * Cfg::P + pos;
          if (writer) {
#pragma unroll
            for (int j = 0; j < 16; ++j) catg[j * Cfg::P] = pooled[j];
          }
        } else {
          if (writer) { __stcs(d4, w0); __stcs(d4 + 1, w1); }
        }
        tmem_ld16(lane_addr + Cfg::TM_C2 + 0 * 64 + 16, e);
        tmem_ld16(lane_addr + Cfg::TM_C2 + 1 * 64 + 16, o);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(bars + 8 * BAR_C2_EMPTY);
        pool16(e, o, &re[2], &ro[2], bias2 + 16, w0, w1);
        if constexpr (TRAIN) {
          if (writer) {
#pragma unroll
            for (int j = 0; j < 16; ++j) catg[(16 + j) * Cfg::P] = pooled[j];
          }
          if (valid) {   // m2 [sample][y][x][half], rows y = 2i, 2i+1 of the H2 x H2 conv2 output
            uint32_t* mg = ta.m2 + (p * G::TPos2 + (2 * i) * Cfg::H2 + x) * 2 + chalf;
            mg[0] = me | (mbits_e << 16);
            mg[2 * Cfg::H2] = mo | (mbits_o << 16);
          }
        } else {
          if (writer) { __stcs(d4 + 2, w0); __stcs(d4 + 3, w1); }
        }
      }
      // A2 is rewritten by the next patch's conv1 epilogue: all residual reads must be done
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
    }
  }

  // ---------------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem, Cfg::TM_COLS);
  }
}

}  // namespace cmlpl

using namespace cmlpl;

static int launch_patch_cnn(const void* f0pad, int cols, int w, int band_rows, const void* packed, void* p2,
                            cudaStream_t stream) {
  CMLPL_CHECK_ARG(f0pad && packed && p2, "patch_cnn: null pointer");
  CMLPL_CHECK_ARG(w == 20 || w == 11, "patch_cnn: w=%d unsupported (20 = the reference's BaseNet2, tools/models.py:127; "
                  "11 = the odd-window variant of BASELINE configs[4])", w);
  CMLPL_CHECK_ARG(cols > 0 && band_rows > 0, "patch_cnn: bad dims");
  CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(f0pad) % 16 == 0 && reinterpret_cast<uintptr_t>(p2) % 16 == 0 &&
                      reinterpret_cast<uintptr_t>(packed) % 16 == 0, "patch_cnn: buffers must be 16-byte aligned");
  const PackedLayout L = packed_layout(1, 1, w);   // conv offsets do not depend on B, C
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const int64_t npix = int64_t(band_rows) * cols;
  int64_t grid = sm_count();
  if (grid > npix) grid = npix;
  if (w == 11) {
    using Cfg = PatchCfg<11>;
    auto kern = patch_cnn_kernel<11, false>;
    CMLPL_MAX_DYN_SMEM(kern, Cfg::SMEM);
    kern<<<int(grid), kThreads, Cfg::SMEM, stream>>>(
        static_cast<const __half*>(f0pad), cols, band_rows, pk + L.w1, pk + L.w2,
        reinterpret_cast<const float*>(pk + L.b1), reinterpret_cast<const float*>(pk + L.b2),
        static_cast<__half*>(p2), TrainCnnArgs{});
  } else {
    using Cfg = PatchCfg<20>;
    auto kern = patch_cnn_kernel<20, false>;
    CMLPL_MAX_DYN_SMEM(kern, Cfg::SMEM);
    kern<<<int(grid), kThreads, Cfg::SMEM, stream>>>(
        static_cast<const __half*>(f0pad), cols, band_rows, pk + L.w1, pk + L.w2,
        reinterpret_cast<const float*>(pk + L.b1), reinterpret_cast<const float*>(pk + L.b2),
        static_cast<__half*>(p2), TrainCnnArgs{});
  }
  CMLPL_CHECK_LAUNCH("patch_cnn");
  return CMLPL_OK;
}

namespace cmlpl {
int launch_train_cnn(const TrainCnnArgs& ta, int w, cudaStream_t st) {
  int grid = sm_count() & ~1;                       // split evenly between the two nets
  if (grid > 2 * ta.nb) grid = 2 * ta.nb;
  if (w == 11) {
    auto kern = patch_cnn_kernel<11, true>;
    CMLPL_MAX_DYN_SMEM(kern, PatchCfg<11>::SMEM);
    kern<<<grid, kThreads, PatchCfg<11>::SMEM, st>>>(nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, ta);
  } else {
    auto kern = patch_cnn_kernel<20, true>;
    CMLPL_MAX_DYN_SMEM(kern, PatchCfg<20>::SMEM);
    kern<<<grid, kThreads, PatchCfg<20>::SMEM, st>>>(nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, ta);
  }
  CMLPL_CHECK_LAUNCH("train_cnn");
  return CMLPL_OK;
}
}  // namespace cmlpl

extern "C" int cmlpl_patch_cnn_f16(const void* f0pad, int cols, int w, int band_rows, const void* packed, void* p2,
                                   cmlpl_stream_t stream) {
  return launch_patch_cnn(f0pad, cols, w, band_rows, packed, p2, static_cast<cudaStream_t>(stream));
}
