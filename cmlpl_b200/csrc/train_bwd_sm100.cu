// Fused training step, backward trunk (train.py:267,271 through tools/models.py:132-140): data gradients, weight
// gradients and bias gradients of conv2, conv1 and conv0 on tcgen05 (fp16 operands, fp32 accumulate in TMEM).
//
// One persistent CTA owns a slice of ONE net's samples and keeps that net's 3x3 weights in shared memory.  A sample's
// upstream gradient dz (after the pool / ReLU backward) and its saved input activation live in shared memory as
// zero-bordered chunk planes [8 chunks][(H+2)x(H+2) entries][8 channels]; that single layout is
//   * the K-major A operand of the DATA gradient (K = output channels; a 3x3 tap is a start-address offset, the
//     weights [tap][ci-chunk][co][8 ci] are read as an MN-major B operand, i.e. transposed for free):
//         dact[pos][ci] = sum_{tap,co} dz[pos - off(tap)][co] * W[co][ci][tap]            M=128 N=64 K=16 per MMA
//   * the MN-major A operand (dz) and MN-major B operand (activation, shifted by the tap) of the WEIGHT gradient,
//     whose K dimension runs over positions:
//         dW[co][ci][tap] = sum_pos dz[pos][co] * act[pos + off(tap)][ci]                 M=64 N=64 K=16 per MMA
//     accumulated in TMEM over all samples of the CTA (rows r of an M=64 accumulator sit in lanes r%16 + 32*(r/16);
//     taps 5..8 and the bias gradient use lanes +16 of the same columns) and added to the fp32 gradient once
//   * the bias gradient, as one more N=8 MMA per K-step against a plane of ones.
// Gradient operands are multiplied by a power of two S (grad_scale) so they sit in fp16's normal range; S is undone on
// the fp32 results.  (Layout facts verified on hardware by scripts/micro/mn_major_probe.cu.)
// H = 10 / 20 are conv2 / conv1 of the w = 20 net, H = 5 / 11 those of the w = 11 net.  Odd maps are pooled with floor
// semantics (avg_pool2d): the last row / column gets no upstream gradient, but stays a conv output whose data gradient
// (from its neighbours' taps) and residual fan-out are formed like any other position's.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "train_common.cuh"
#include "train_kernels.cuh"

namespace cmlpl {

__host__ __device__ constexpr uint32_t idesc_f16_major(int m, int n, int a_mn, int b_mn) {
  return (1u << 4) | (uint32_t(a_mn) << 15) | (uint32_t(b_mn) << 16) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}

template <int H>
struct BwdCfg {
  static constexpr int PW = H + 2;                       // padded row width (entries)
  static constexpr int E0 = PW + 1;                      // entry of position (0, 0)
  static constexpr int LEN = (H - 1) * PW + H;           // entries from (0,0) to (H-1,H-1)
  static constexpr int NT = (LEN + 127) / 128;           // 128-row tiles of the data gradient
  static constexpr int KS = (LEN + 15) / 16;             // K-steps of the weight gradient
  static constexpr int ENT = (E0 + NT * 128 + PW + 1 + 7) / 8 * 8;
  static constexpr int CH = ENT * 16;                    // bytes per chunk plane
  static constexpr int NPOS = H * H;
  static constexpr int WBYTES = 9 * 8 * 64 * 16;
  static constexpr int S_DZ = 0;
  static constexpr int S_ACT = 8 * CH;
  static constexpr int S_W = 16 * CH;
  static constexpr int S_ONES = S_W + WBYTES;
  static constexpr int S_BAR = S_ONES + 256;
  static constexpr int S_TMEM = S_BAR + 64;
  static constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
  static_assert(E0 + KS * 16 + PW + 1 <= ENT, "weight-gradient reads stay inside the planes");
};

enum { BB_IN_FULL = 0, BB_W_DONE, BB_D_FULL0, BB_D_FULL1, BB_D_EMPTY0, BB_D_EMPTY1 };
constexpr int kBwdWorkers = 256, kBwdThreads = kBwdWorkers + 32;
// TMEM columns: data-gradient slots 0..127; weight gradient 128 + tap*64 (taps 0..4, lanes +0) and
// 128 + (tap-5)*64 (taps 5..8, lanes +16); bias gradient 384..391 at lanes +16
__device__ __forceinline__ uint32_t wg_taddr(uint32_t tmem, int tap) {
  return tap < 5 ? tmem + 128 + tap * 64 : tmem + (16u << 16) + 128 + (tap - 5) * 64;
}

template <int H>
__global__ void __launch_bounds__(kBwdThreads, 1)
train_conv_bwd_kernel(ConvBwdArgs a) {
  using C = BwdCfg<H>;
  constexpr bool kConv2 = H == 10 || H == 5;             // conv2 of the window W = 20 / 11; otherwise conv1, H = W
  constexpr int W = H == 5 ? 11 : H == 10 ? 20 : H;
  using G = TrainGeom<W>;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + C::S_BAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + C::S_TMEM);
  const int cpn = int(gridDim.x >> 1);
  const int net = int(blockIdx.x) / cpn, cta = int(blockIdx.x) - net * cpn;
  const int per = (a.nb + cpn - 1) / cpn;
  const int k_begin = min(cta * per, a.nb), k_end = min(k_begin + per, a.nb);
  const int nsamp = k_end - k_begin;
  const int s0 = net * a.nb + k_begin;                   // first global sample of this CTA

  // ---------------------------------------------------------------- prologue
  {
    uint4* z = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < 16 * C::CH / 16; i += kBwdThreads) z[i] = make_uint4(0, 0, 0, 0);
    // fp16 [tap][ci chunk][co][8 ci], packed by train_conv0_kernel this step
    const uint4* wg = reinterpret_cast<const uint4*>(a.wpack[net]);
    uint4* sw = reinterpret_cast<uint4*>(smem + C::S_W);
    for (int i = tid; i < C::WBYTES / 16; i += kBwdThreads) sw[i] = __ldg(wg + i);
    if (tid < 128) reinterpret_cast<__half*>(smem + C::S_ONES)[tid] = __float2half_rn(1.f);
  }
  if (tid == 0) {
    mbar_init(bars + 8 * BB_IN_FULL, kBwdWorkers);
    mbar_init(bars + 8 * BB_W_DONE, 1);
    mbar_init(bars + 8 * BB_D_FULL0, 1);
    mbar_init(bars + 8 * BB_D_FULL1, 1);
    mbar_init(bars + 8 * BB_D_EMPTY0, kBwdWorkers);
    mbar_init(bars + 8 * BB_D_EMPTY1, kBwdWorkers);
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(sbase + C::S_TMEM, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const float S = grad_scale(a.prm->grad_amax), invS = 1.f / S;

  if (warp == 8) {
    // ================================================================ MMA issuer
    constexpr uint32_t kIdD = idesc_f16_major(128, 64, 0, 1);   // data gradient: A K-major, B MN-major
    constexpr uint32_t kIdW = idesc_f16_major(64, 64, 1, 1);    // weight gradient: both MN-major
    constexpr uint32_t kIdB = idesc_f16_major(64, 8, 1, 1);     // bias gradient
    uint32_t use[2] = {0, 0};
    for (int k = 0; k < nsamp; ++k) {
      mbar_wait(bars + 8 * BB_IN_FULL, k & 1, 50);
      tc_fence_after();
#pragma unroll 1
      for (int t = 0; t < C::NT; ++t) {
        const int slot = t & 1;
        mbar_wait(bars + 8 * (BB_D_EMPTY0 + slot), (use[slot] & 1) ^ 1, 51);
        ++use[slot];
        tc_fence_after();
        if (lane == 0) {
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            const int off = -(tap / 3 - 1) * C::PW - (tap % 3 - 1);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_f16(tmem + slot * 64,
                       make_desc(sbase + C::S_DZ + (C::E0 + t * 128 + off) * 16 + ks * 2 * C::CH, C::CH, 128),
                       make_desc(sbase + C::S_W + tap * 8192 + ks * 256, 128, 1024), kIdD, (tap | ks) != 0 ? 1u : 0u);
          }
          umma_commit(bars + 8 * (BB_D_FULL0 + slot));
        }
        __syncwarp();
      }
      if (lane == 0) {
#pragma unroll 1
        for (int ks = 0; ks < C::KS; ++ks) {
          const uint32_t acc = (k | ks) != 0 ? 1u : 0u;
          const uint64_t da = make_desc(sbase + C::S_DZ + (C::E0 + ks * 16) * 16, 128, C::CH);
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            const int off = (tap / 3 - 1) * C::PW + (tap % 3 - 1);
            umma_f16(wg_taddr(tmem, tap), da, make_desc(sbase + C::S_ACT + (C::E0 + ks * 16 + off) * 16, 128, C::CH),
                     kIdW, acc);
          }
          umma_f16(tmem + (16u << 16) + 384, da, make_desc(sbase + C::S_ONES, 128, 128), kIdB, acc);
        }
        umma_commit(bars + 8 * BB_W_DONE);
      }
      __syncwarp();
    }
  } else {
    // ================================================================ workers: fill the planes, drain the data gradient
    const int q4 = warp & 3, chalf = warp >> 2;
    const uint32_t lane_addr = tmem + (uint32_t(q4 * 32) << 16) + chalf * 32;
    uint32_t use[2] = {0, 0};
    for (int k = 0; k < nsamp; ++k) {
      const int64_t s = s0 + k;
      if (k > 0) {
        mbar_wait(bars + 8 * BB_W_DONE, (k - 1) & 1, 52);              // every MMA of the previous sample has read the planes
        named_bar_sync(1, kBwdWorkers);                                // ... and every worker its residual entries
      }
      if constexpr (kConv2) {
        // dz2 = dL/dp2 / 4 * [a2 > 0] (pool + ReLU backward, tools/models.py:139-140), scaled, and the p1 planes.
        // Odd H: the floor pool drops the last row / column, where dz2 = 0.
        constexpr int NP = G::NP2, P = NP * NP;
        const float* dc = a.dcat + s * G::CatDim;
        const uint32_t* m2 = a.m2 + s * (G::TPos2 * 2);
        const unsigned char* pg = reinterpret_cast<const unsigned char*>(a.act) + s * G::Act2Bytes;
        const float q = 0.25f * S;
        for (int i = tid; i < 8 * G::TPos2; i += kBwdWorkers) {
          const int chunk = i / G::TPos2, pos = i - chunk * G::TPos2;
          const int y = pos / H, x = pos - y * H;
          const int ent = (y + 1) * C::PW + x + 1;
          cp_async16(sbase + C::S_ACT + chunk * C::CH + ent * 16, pg + (chunk * G::TPos2 + pos) * 16);
          const bool kept = H % 2 == 0 || (y < 2 * NP && x < 2 * NP);
          const uint32_t bits = kept ? m2[pos * 2 + (chunk >> 2)] >> ((chunk & 3) * 8) : 0u;
          const float* d = dc + (chunk * 8) * P + (y >> 1) * NP + (x >> 1);
          __half2 h[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float v0 = (bits >> (2 * j)) & 1u ? __ldg(d + (2 * j) * P) * q : 0.f;
            const float v1 = (bits >> (2 * j + 1)) & 1u ? __ldg(d + (2 * j + 1) * P) * q : 0.f;
            h[j] = __floats2half2_rn(v0, v1);
          }
          *reinterpret_cast<uint4*>(smem + C::S_DZ + chunk * C::CH + ent * 16) = *reinterpret_cast<uint4*>(h);
        }
        if constexpr (W % 2 == 1) {
          // conv1's last row / column feed no pooling window: dz1 there is 0 (written here, read by conv1's backward)
          unsigned char* zg = reinterpret_cast<unsigned char*>(a.dz_out) + s * G::ActBytes;
          for (int i = tid; i < 8 * (2 * W - 1); i += kBwdWorkers) {
            const int chunk = i / (2 * W - 1), k = i - chunk * (2 * W - 1);
            const int y = k < W ? W - 1 : k - W, x = k < W ? k : W - 1;
            *reinterpret_cast<uint4*>(zg + (chunk * G::TPos + y * W + x) * 16) = make_uint4(0, 0, 0, 0);
          }
        }
      } else {
        const unsigned char* zg = reinterpret_cast<const unsigned char*>(a.dz_in) + s * G::ActBytes;
        const unsigned char* ag = reinterpret_cast<const unsigned char*>(a.act) + s * G::ActBytes;
        for (int i = tid; i < 8 * G::TPos; i += kBwdWorkers) {
          const int chunk = i / G::TPos, pos = i - chunk * G::TPos;
          const int y = pos / H, x = pos - y * H;
          const int ent = (y + 1) * C::PW + x + 1;
          cp_async16(sbase + C::S_DZ + chunk * C::CH + ent * 16, zg + (chunk * G::TPos + pos) * 16);
          cp_async16(sbase + C::S_ACT + chunk * C::CH + ent * 16, ag + (chunk * G::TPos + pos) * 16);
        }
      }
      cp_async_wait_all();
      fence_proxy_async();
      mbar_arrive(bars + 8 * BB_IN_FULL);
      mbar_wait(bars + 8 * BB_IN_FULL, k & 1, 55);       // the residual entries read below were written by other workers
#pragma unroll 1
      for (int t = 0; t < C::NT; ++t) {
        const int slot = t & 1;
        const int ent = C::E0 + t * 128 + q4 * 32 + lane;
        const int y = ent / C::PW - 1, x = ent - (y + 1) * C::PW - 1;
        const bool valid = x >= 0 && x < H && y < H;
        // the residual branch (models.py:135,139: x + x_res) hands dz straight through: same entry of the dz planes
        uint4 rz[4];
#pragma unroll
        for (int c = 0; c < 4; ++c)
          rz[c] = valid ? *reinterpret_cast<const uint4*>(smem + C::S_DZ + (chalf * 4 + c) * C::CH + ent * 16)
                        : make_uint4(0, 0, 0, 0);
        mbar_wait(bars + 8 * (BB_D_FULL0 + slot), use[slot] & 1, 53);
        ++use[slot];
        tc_fence_after();
        float v[32];
        tmem_ld16(lane_addr + slot * 64, v);
        tmem_ld16(lane_addr + slot * 64 + 16, v + 16);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(bars + 8 * (BB_D_EMPTY0 + slot));
        const __half2* rh = reinterpret_cast<const __half2*>(rz);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 f = __half22float2(rh[j]);
          v[2 * j] += f.x; v[2 * j + 1] += f.y;
        }
        if (!valid) continue;
        if constexpr (kConv2) {
          // dL/dp1 (scaled) -> pool backward to the four W x W positions, ReLU mask of a1 -> dz1 (scaled)
          unsigned char* og = reinterpret_cast<unsigned char*>(a.dz_out) + s * G::ActBytes + (chalf * 4) * (G::TPos * 16);
          const uint32_t* m1 = a.m1 + s * (G::TPos * 2) + chalf;
#pragma unroll
          for (int ab = 0; ab < 4; ++ab) {
            const int pos = (2 * y + (ab >> 1)) * W + 2 * x + (ab & 1);
            const uint32_t bits = m1[pos * 2];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              __half2 h[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int b = c * 8 + 2 * j;
                h[j] = __floats2half2_rn((bits >> b) & 1u ? v[b] * 0.25f : 0.f, (bits >> (b + 1)) & 1u ? v[b + 1] * 0.25f : 0.f);
              }
              *reinterpret_cast<uint4*>(og + c * (G::TPos * 16) + pos * 16) = *reinterpret_cast<uint4*>(h);
            }
          }
        } else {
          unsigned char* og = reinterpret_cast<unsigned char*>(a.dz_out) + s * G::ActBytes + (chalf * 4) * (G::TPos * 16) +
                              (y * H + x) * 16;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            __half2 h[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) h[j] = __floats2half2_rn(v[c * 8 + 2 * j], v[c * 8 + 2 * j + 1]);
            *reinterpret_cast<uint4*>(og + c * (G::TPos * 16)) = *reinterpret_cast<uint4*>(h);
          }
        }
      }
    }
    // ---------------------------------------------------------------- weight / bias gradient of this CTA's samples
    if (nsamp > 0) {
      mbar_wait(bars + 8 * BB_W_DONE, (nsamp - 1) & 1, 54);
      tc_fence_after();
      // staged as [tap][co][ci]: a thread's 32 accumulator columns are 32 consecutive ci -> eight 16-byte vector reds
      const int set = lane >> 4, co = q4 * 16 + (lane & 15);
      float* gs = a.g_stage[net] + co * 64 + chalf * 32;
#pragma unroll 1
      for (int j = 0; j < 5; ++j) {
        float v[32];
        tmem_ld16(lane_addr + 128 + j * 64, v);
        tmem_ld16(lane_addr + 128 + j * 64 + 16, v + 16);
        tmem_ld_wait();
        const int tap = set * 5 + j;
        if (tap < 9) {
#pragma unroll
          for (int c = 0; c < 32; c += 4)
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(gs + tap * 4096 + c), "f"(v[c] * invS),
                         "f"(v[c + 1] * invS), "f"(v[c + 2] * invS), "f"(v[c + 3] * invS) : "memory");
        } else if (tap == 9 && chalf == 0) {
          atomicAdd(a.g_b[net] + co, v[0] * invS);
        }
      }
    }
  }
  // ---------------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 8) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

template <int H>
static int launch_conv_bwd_h(const ConvBwdArgs& a, int grid, cudaStream_t st) {
  auto kern = train_conv_bwd_kernel<H>;
  CMLPL_MAX_DYN_SMEM(kern, BwdCfg<H>::SMEM);
  kern<<<grid, kBwdThreads, BwdCfg<H>::SMEM, st>>>(a);
  return CMLPL_OK;
}

// H = 10 / 20: conv2 / conv1 of the w = 20 net; H = 5 / 11: of the w = 11 net
int launch_train_conv_bwd(int H, const ConvBwdArgs& a, cudaStream_t st) {
  int grid = sm_count() & ~1;
  if (grid > 2 * a.nb) grid = 2 * a.nb;
  int rc;
  switch (H) {
    case 10: rc = launch_conv_bwd_h<10>(a, grid, st); break;
    case 20: rc = launch_conv_bwd_h<20>(a, grid, st); break;
    case 5: rc = launch_conv_bwd_h<5>(a, grid, st); break;
    case 11: rc = launch_conv_bwd_h<11>(a, grid, st); break;
    default: CMLPL_CHECK_ARG(false, "train_conv_bwd: H=%d unsupported", H);
  }
  if (rc != CMLPL_OK) return rc;
  CMLPL_CHECK_LAUNCH("train_conv_bwd");
  return CMLPL_OK;
}

// ============================================================================ conv0 weight gradient
// dW0[co][ci] = sum_{sample,pos} da0[pos][co] * x16[pos][ci], db0 = sum da0: both operands are unpadded chunk planes
// in HBM, so a sample is 2 x 8 bulk copies of its chunk planes into a two-stage ring; one M=64 N=64 and one N=8 (ones)
// MMA per K-step of 16 positions (25 at W = 20).  At W = 11 the 121 positions take 8 K-steps: a staged plane is padded
// to 128 positions whose zero tail (never written by the copies) adds nothing.
template <int W>
struct C0bCfg {
  using G = TrainGeom<W>;
  static constexpr int KS = (G::TPos + 15) / 16;        // K-steps per sample
  static constexpr int GCH = G::TPos * 16;              // chunk plane in HBM (bytes)
  static constexpr int PCH = KS * 256;                  // chunk plane in shared memory
  static constexpr int STAGE = 2 * 8 * PCH;             // da0 planes, then x16 planes
  static constexpr int S_ONES = 2 * STAGE;
  static constexpr int S_BAR = S_ONES + 256;
  static constexpr int S_TMEM = S_BAR + 64;
  static constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
};
enum { C0B_FULL0 = 0, C0B_FULL1, C0B_EMPTY0, C0B_EMPTY1, C0B_DONE };

template <int W>
__global__ void __launch_bounds__(128, 1)
train_conv0_bwd_kernel(Conv0BwdArgs a) {
  using Cfg = C0bCfg<W>;
  constexpr int STAGE = Cfg::STAGE, PCH = Cfg::PCH, GCH = Cfg::GCH, S_ONES = Cfg::S_ONES, S_BAR = Cfg::S_BAR,
                S_TMEM = Cfg::S_TMEM;
  enum { B_FULL0 = C0B_FULL0, B_FULL1 = C0B_FULL1, B_EMPTY0 = C0B_EMPTY0, B_EMPTY1 = C0B_EMPTY1, B_DONE = C0B_DONE };
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + S_BAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);
  const int cpn = int(gridDim.x >> 1);
  const int net = int(blockIdx.x) / cpn, cta = int(blockIdx.x) - net * cpn;
  const int per = (a.nb + cpn - 1) / cpn;
  const int k_begin = min(cta * per, a.nb), k_end = min(k_begin + per, a.nb);
  const int nsamp = k_end - k_begin;
  const int64_t s0 = int64_t(net) * a.nb + k_begin;
  reinterpret_cast<__half*>(smem + S_ONES)[tid] = __float2half_rn(1.f);
  if constexpr (PCH > GCH) {
    for (int i = tid; i < 2 * 2 * 8 * (PCH - GCH) / 16; i += 128) {     // zero tails of every staged plane
      const int plane = i / ((PCH - GCH) / 16), j = i - plane * ((PCH - GCH) / 16);
      reinterpret_cast<uint4*>(smem + plane * PCH + GCH)[j] = make_uint4(0, 0, 0, 0);
    }
  }
  // the 3x3 weight gradients train_conv_bwd_kernel staged as [net][conv][tap][co][ci] -> torch's [co][ci][3][3]
  for (int i = blockIdx.x * 128 + tid; i < 4 * 36864; i += int(gridDim.x) * 128) {
    const int t4 = i / 36864, j = i - t4 * 36864;                   // j = (tap * 64 + co) * 64 + ci, coalesced read
    const int tap = j >> 12, co = (j >> 6) & 63, ci = j & 63;
    a.g_w3[t4 >> 1][t4 & 1][(co * 64 + ci) * 9 + tap] = __ldg(a.gstage + i);
  }
  if (tid == 0) {
    for (int i = 0; i < 5; ++i) mbar_init(bars + 8 * i, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(sbase + S_TMEM, 128);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const float invS = 1.f / grad_scale(a.prm->grad_amax);
  if (warp == 1 && lane == 0) {
    // producer
    for (int k = 0; k < nsamp; ++k) {
      const int st = k & 1;
      mbar_wait(bars + 8 * (B_EMPTY0 + st), ((k >> 1) & 1) ^ 1, 60);
      const uint32_t full = bars + 8 * (B_FULL0 + st);
      mbar_arrive_expect_tx(full, 2 * 8 * GCH);
      const unsigned char* g0 = reinterpret_cast<const unsigned char*>(a.da0) + (s0 + k) * (8 * GCH);
      const unsigned char* g1 = reinterpret_cast<const unsigned char*>(a.x16) + (s0 + k) * (8 * GCH);
      for (int c = 0; c < 8; ++c) {
        bulk_g2s(sbase + st * STAGE + c * PCH, g0 + c * GCH, GCH, full);
        bulk_g2s(sbase + st * STAGE + 8 * PCH + c * PCH, g1 + c * GCH, GCH, full);
      }
    }
  } else if (warp == 2 && lane == 0) {
    // MMA issuer
    constexpr uint32_t kIdW = idesc_f16_major(64, 64, 1, 1), kIdB = idesc_f16_major(64, 8, 1, 1);
    for (int k = 0; k < nsamp; ++k) {
      const int st = k & 1;
      mbar_wait(bars + 8 * (B_FULL0 + st), (k >> 1) & 1, 61);
      tc_fence_after();
#pragma unroll 1
      for (int ks = 0; ks < Cfg::KS; ++ks) {
        const uint32_t acc = (k | ks) != 0 ? 1u : 0u;
        const uint64_t da = make_desc(sbase + st * STAGE + ks * 256, 128, PCH);
        umma_f16(tmem, da, make_desc(sbase + st * STAGE + 8 * PCH + ks * 256, 128, PCH), kIdW, acc);
        umma_f16(tmem + 64, da, make_desc(sbase + S_ONES, 128, 128), kIdB, acc);
      }
      umma_commit(bars + 8 * (B_EMPTY0 + st));
    }
    umma_commit(bars + 8 * B_DONE);
  }
  __syncwarp();
  if (nsamp > 0) {
    mbar_wait(bars + 8 * B_DONE, 0, 62);
    tc_fence_after();
    float v[64], b[8];
    const uint32_t la = tmem + (uint32_t(warp * 32) << 16);
    tmem_ld16(la, v); tmem_ld16(la + 16, v + 16); tmem_ld16(la + 32, v + 32); tmem_ld16(la + 48, v + 48);
    tmem_ld8(la + 64, b);
    tmem_ld_wait();
    if (lane < 16) {
      const int co = warp * 16 + lane;
#pragma unroll
      for (int ci = 0; ci < 60; ++ci) atomicAdd(a.g_w[net] + co * 60 + ci, v[ci] * invS);
      atomicAdd(a.g_b[net] + co, b[0] * invS);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem, 128); }
}

int launch_train_conv0_bwd(const Conv0BwdArgs& a, int w, cudaStream_t st) {
  int grid = sm_count() & ~1;
  if (grid > 2 * a.nb) grid = 2 * a.nb;
  if (w == 11) {
    auto kern = train_conv0_bwd_kernel<11>;
    CMLPL_MAX_DYN_SMEM(kern, C0bCfg<11>::SMEM);
    kern<<<grid, 128, C0bCfg<11>::SMEM, st>>>(a);
  } else {
    auto kern = train_conv0_bwd_kernel<20>;
    CMLPL_MAX_DYN_SMEM(kern, C0bCfg<20>::SMEM);
    kern<<<grid, 128, C0bCfg<20>::SMEM, st>>>(a);
  }
  CMLPL_CHECK_LAUNCH("train_conv0_bwd");
  return CMLPL_OK;
}

}  // namespace cmlpl
