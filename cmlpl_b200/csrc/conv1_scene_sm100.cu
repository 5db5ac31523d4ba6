// Scene-level conv1 + pool1 with exact compute sharing (SURVEY section 7 / 8-f3, conv1 part).
//
// The reference applies conv1 (3x3, zero padding at the PATCH border, tools/models.py:104,134) to
// every pixel's 20x20 window separately, but a window position's output only depends on (a) its
// 3x3 neighbourhood in the scene and (b) which taps the patch border cuts off: rows y=0 / 1..18 / 19
// drop dy=0 / nothing / dy=2 and likewise for columns.  So conv1 (+bias, +residual, ReLU,
// models.py:133-135) is evaluated ONCE per scene position in 3x3 = 9 border-class variants
//     G[a][b][p] = relu(b1 + F0[p] + sum_{dy in S_a, dx in S_b} W1[dy,dx] . F0[p + (dy-1, dx-1)])
//     S_top/left = {1,2},  S_mid = {0,1,2},  S_bot/right = {0,1}
// and the patch of pixel (r,c) reads G[a(y)][b(x)] at scene position (r+y, c+x): identical math up to
// fp32 summation order, ~15x fewer conv1 FLOPs.  The 2x2 average pools (models.py:136) are formed for
// every top-left position in the 9 pooled border classes
//     PM[A][B][pr,pc] = 1/4 sum_{u,v in {0,1}} G[a(A,u)][b(B,v)][pr+u, pc+v]
//     a(top,0)=top a(top,1)=mid   a(mid,.)=mid   a(bot,0)=mid a(bot,1)=bot     (pooled row 0 / 1..8 / 9)
// and likewise b(B,v) for columns.
//
// conv1_pool_kernel does both in ONE kernel -- the fp32 variants G (2.3 KB per scene position) never touch
// HBM.  It is a persistent, warp-specialised tcgen05 implicit GEMM over 4x30-position tiles (M=128 rows =
// 4 rows x 32 columns incl. one halo column each side), taps = A-descriptor offsets in a row-major
// zero-haloed shared-memory tile loaded by TMA:
//   * the tensor core produces the nine single-tap-column sums  T[dy][dx] = sum_ci W1[dy,dx] . F0[p+(dy-1,dx-1)]
//     separately (N = 32 channels at a time: sub-stage (h, dy) = T[dy][0..2] in 96 TMEM columns, ring of 5), so
//     that all three column classes  R[dy][left|mid|right] = T1+T2 | T0+T1+T2 | T0+T1  are formed in the
//     epilogue from one TMEM read (36 MMAs per 32 channels), and the row classes from them as
//     top = R1+R2, mid = R0+R1+R2, bot = R0+R1;
//   * a tile's 4 conv rows give 3 pooled rows and its 30 conv columns 29 pooled columns: the vertical 2x2
//     partner (ty+1, tx) lives in another warp (TMEM lane quarter) and comes through a double-buffered
//     shared-memory exchange, the horizontal partner (tx+1) through a warp shuffle;
//   * pooled cells go straight to the parity planes pmq (f16, chunk-planar), 8 channels = one 16-byte chunk
//     per thread and pass.
//   V[A][b]  = G[a0(A)][b](y,x) + G[a1(A)][b](y+1,x)                 (a0,a1 = top,mid | mid,mid | mid,bot)
//   PM[A][B] = 1/4 (V[A][b0(B)](x) + V[A][b1(B)](x+1))               (b0,b1 = left,mid | mid,mid | mid,right)
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "tma.cuh"

namespace cmlpl {

namespace c1p {
constexpr int TH = 4, TP = 32, OH = 3, OW = 29;      // conv rows, row pitch; pooled rows / columns per tile
constexpr int CH = (TH + 2) * TP * 16;               // 3 072: one chunk plane of the conv0 tile, dense (written by TMA)
constexpr int ABYTES = 8 * CH;
constexpr int WBYTES = 3 * 8 * 192 * 16;
constexpr int kEpi = 256, kThreads = kEpi + 64;      // warps 0-7 epilogue, warp 8 loader (one thread, TMA), warp 9 MMA issuer
constexpr int kLoadWarp = kEpi / 32, kMmaWarp = kLoadWarp + 1;
constexpr int XBYTES = 12 * kEpi * 16;               // exchange: 12 float4 (G[mid|bot][3 b][8 ch]) per epilogue thread
constexpr int S_W = 0, S_A = WBYTES, S_X = S_A + 2 * ABYTES, S_BIAS = S_X + 2 * XBYTES, S_BAR = S_BIAS + 256,
              S_TMEM = S_BAR + 128;
constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
constexpr int NSUB = 5, SUBCOLS = 96;
constexpr int kWLbo = 192 * 16, kWDx = 8 * kWLbo;
enum { A_FULL0 = 0, A_FULL1, A_EMPTY0, A_EMPTY1, S_FULL0 = 4, S_EMPTY0 = 4 + NSUB, W_FULL = 4 + 2 * NSUB };
static_assert(SMEM <= 232448, "conv1_pool: shared memory over the 227 KB limit");
static_assert(W_FULL < 16, "conv1_pool: barrier area too small");
static_assert(S_A % 128 == 0 && ABYTES % 128 == 0, "conv1_pool: TMA destinations must be 128-byte aligned");
}  // namespace c1p

// f0: f16 chunk-planar [8][PR][PC][8];  pmq f16 [9 = A*3+B][4 planes][8 chunks][PR2][PC2][8]
__global__ void __launch_bounds__(c1p::kThreads, 1)
conv1_pool_kernel(const __grid_constant__ CUtensorMap tm_f0, int PR, int PC, int PR2, int PC2, int ncls /* pooled classes per direction stored: 3, or 2 (top, mid) for 11x11 windows */,
                  const unsigned char* __restrict__ w1p, const float* __restrict__ b1g, __half* __restrict__ pmq) {
  using namespace c1p;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + S_BAR;
  float* sbias = reinterpret_cast<float*>(smem + S_BIAS);
  const int tiles_c = (2 * PC2 + OW - 1) / OW, tiles_r = (2 * PR2 + OH - 1) / OH;
  const int ntiles = tiles_r * tiles_c;
  const int64_t psz = int64_t(PR2) * PC2;

  {
    uint4* z = reinterpret_cast<uint4*>(smem + S_A);
    for (int i = tid; i < 2 * ABYTES / 16; i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (tid < 64) sbias[tid] = b1g[tid];
  if (tid == 0) {
    mbar_init(bars + 8 * W_FULL, 1);
    fence_barrier_init();
    bulk_weights_g2s(sbase + S_W, w1p, WBYTES, bars + 8 * W_FULL);
    mbar_init(bars + 8 * A_FULL0, 1); mbar_init(bars + 8 * A_FULL1, 1);
    mbar_init(bars + 8 * A_EMPTY0, 1 + kEpi); mbar_init(bars + 8 * A_EMPTY1, 1 + kEpi);
    for (int s = 0; s < NSUB; ++s) { mbar_init(bars + 8 * (S_FULL0 + s), 1); mbar_init(bars + 8 * (S_EMPTY0 + s), kEpi); }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(sbase + S_TMEM, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);

  if (warp == kLoadWarp) {
    // ================================================================ loader: one TMA box per tile ((TH+2) x TP entries, zero outside the map)
    if (lane == 0) {
      tma_prefetch_desc(&tm_f0);
      uint32_t j = 0;
      [[maybe_unused]] uint32_t ntr = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
        const uint32_t buf = j & 1, ph = (j >> 1) & 1;
        const int tr = t / tiles_c, tc = t - tr * tiles_c;
        mbar_wait(bars + 8 * (A_EMPTY0 + buf), ph ^ 1, 81);
        CMLPL_TR(4, ntr, j);
        mbar_arrive_expect_tx(bars + 8 * (A_FULL0 + buf), ABYTES);
        tma_load_tile(sbase + S_A + buf * ABYTES, &tm_f0, tc * OW - 1, tr * OH - 1, 0, bars + 8 * (A_FULL0 + buf));
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer
    if (tmem != 0) { printf("conv1_pool: unexpected TMEM base %u\n", tmem); __trap(); }
    constexpr uint64_t kHi = (uint64_t(128 >> 4) | (uint64_t(1) << 14)) << 32;
    constexpr uint32_t kI32 = make_idesc_f16(128, 32);
    const uint32_t w_lo = ((sbase + S_W) >> 4) | (uint32_t(kWLbo >> 4) << 16);
    uint32_t j = 0, slot = 0, sph = 0;
    [[maybe_unused]] uint32_t ntr = 0;
    mbar_wait(bars + 8 * W_FULL, 0, 80);                       // weights have landed
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
      const uint32_t buf = j & 1, ph = (j >> 1) & 1;
      // MMA row m of tap (dy,dx) reads tile entry m + dy*TP + dx - 1: descriptors start 16 B before the tile
      const uint32_t a_lo = ((sbase + S_A + buf * ABYTES - 16) >> 4) | (uint32_t(CH >> 4) << 16);
      mbar_wait(bars + 8 * (A_FULL0 + buf), ph, 82);
#pragma unroll 1
      for (int hd = 0; hd < 6; ++hd) {                         // sub-stage = (channel half h, tap row dy)
        const int h = hd / 3, dy = hd - h * 3;
        if (lane == 0) CMLPL_TR(0, ntr, (j * 6 + hd) * 4);
        mbar_wait(bars + 8 * (S_EMPTY0 + slot), sph ^ 1, 83);
        tc_fence_after();
        if (lane == 0) CMLPL_TR(0, ntr, (j * 6 + hd) * 4 + 1);
        if (elect_one_sync()) {
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            const uint32_t d = slot * SUBCOLS + dx * 32;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t a = a_lo + uint32_t(dy * TP + dx) + uint32_t(ks * 2 * CH / 16);
              const uint32_t bb = w_lo + uint32_t((dx * kWDx + ks * 2 * kWLbo) / 16) + uint32_t((2 - dy) * 64 + h * 32);
              umma_f16(d, kHi | uint64_t(a), kHi | uint64_t(bb), kI32, ks ? 1u : 0u);
            }
          }
          umma_commit(bars + 8 * (S_FULL0 + slot));
          if (hd == 5) umma_commit(bars + 8 * (A_EMPTY0 + buf));
        }
        __syncwarp();
        if (lane == 0) CMLPL_TR(0, ntr, (j * 6 + hd) * 4 + 2);
        if (++slot == NSUB) { slot = 0; sph ^= 1; }
      }
    }
  } else {
    // ================================================================ epilogue (warps 0-7)
    const int ty = warp & 3, tx = lane, chsel = warp >> 2;
    const uint32_t lane_addr = uint32_t(ty * 32) << 16;
    const int nb = ty < 3 ? tid + 32 : tid;                   // exchange slot of the position one row below
    uint32_t j = 0, slot = 0, sph = 0, xpar = 0;
    [[maybe_unused]] uint32_t ntr = 0;
    const bool tracer = (warp == 0 || warp == 4) && lane == 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
      const uint32_t buf = j & 1;
      const int tr = t / tiles_c, tc = t - tr * tiles_c;
      const int pr = tr * OH + ty, pc = tc * OW + tx - 1;
      const bool inplane = ty < OH && tx >= 1 && tx <= OW && (pr >> 1) < PR2 && (pc >> 1) < PC2;
      const bool cell = inplane && pr < PR - 1 && pc < PC - 1;
      const int64_t opos = inplane ? (int64_t((pr & 1) * 2 + (pc & 1)) * 8 * psz + int64_t(pr >> 1) * PC2 + (pc >> 1)) : 0;
      mbar_wait(bars + 8 * (A_FULL0 + buf), (j >> 1) & 1, 84);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        uint32_t sl[3];
        if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2) * 8);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          sl[k] = slot;
          mbar_wait(bars + 8 * (S_FULL0 + slot), sph, 85);
          if (++slot == NSUB) { slot = 0; sph ^= 1; }
        }
        tc_fence_after();
        if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2) * 8 + 1);
#pragma unroll 1
        for (int pp = 0; pp < 2; ++pp, xpar ^= 1) {
          const int chunk = h * 4 + pp * 2 + chsel;
          const uint32_t col = uint32_t(pp * 16 + chsel * 8);
          typedef unsigned long long f2;                       // two packed fp32 channels (FADD2 / FMUL2)
          f2 T[3][3][4];
#pragma unroll
          for (int dy = 0; dy < 3; ++dy)
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) tmem_ld8_x2(lane_addr + sl[dy] * SUBCOLS + dx * 32 + col, T[dy][dx]);
          tmem_ld_wait();
          if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2 + pp) * 8 + 2);
          if (pp == 1) {
            tc_fence_before();
#pragma unroll
            for (int k = 0; k < 3; ++k) mbar_arrive(bars + 8 * (S_EMPTY0 + sl[k]));
          }
          {
            // bias + residual (centre entry of the A tile) go into the centre tap, which every border class keeps
            const uint4 rv = *reinterpret_cast<const uint4*>(smem + S_A + buf * ABYTES + chunk * CH + ((ty + 1) * TP + tx) * 16);
            const __half2* hr = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = __half22float2(hr[e]);
              T[1][1][e] = f2_add(T[1][1][e], f2_pack(f.x + sbias[chunk * 8 + 2 * e], f.y + sbias[chunk * 8 + 2 * e + 1]));
            }
          }
          // G[a][b] = relu(b1 + F0 + sum of the taps the (row class a, column class b) border keeps)
          f2 G[3][3][4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            f2 R[3][3];
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
              const f2 s12 = f2_add(T[dy][1][c], T[dy][2][c]);
              R[dy][0] = s12; R[dy][1] = f2_add(T[dy][0][c], s12); R[dy][2] = f2_add(T[dy][0][c], T[dy][1][c]);
            }
#pragma unroll
            for (int b = 0; b < 3; ++b) {
              const f2 top = f2_add(R[1][b], R[2][b]);
              G[0][b][c] = f2_relu(top);
              G[1][b][c] = f2_relu(f2_add(R[0][b], top));
              G[2][b][c] = f2_relu(f2_add(R[0][b], R[1][b]));
            }
          }
          // vertical partner through shared memory: this thread publishes its mid / bot variants
          ulonglong2* xb = reinterpret_cast<ulonglong2*>(smem + S_X + xpar * XBYTES);
#pragma unroll
          for (int a = 1; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b)
#pragma unroll
              for (int q = 0; q < 2; ++q)
                xb[(((a - 1) * 3 + b) * 2 + q) * kEpi + tid] = make_ulonglong2(G[a][b][2 * q], G[a][b][2 * q + 1]);
          if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2 + pp) * 8 + 3);
          named_bar_sync(1, kEpi);
          if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2 + pp) * 8 + 4);
          f2 V[3][3][4];                                       // [A][b]
#pragma unroll
          for (int b = 0; b < 3; ++b)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const ulonglong2 m = xb[((0 * 3 + b) * 2 + q) * kEpi + nb];
              const ulonglong2 o = xb[((1 * 3 + b) * 2 + q) * kEpi + nb];
              V[0][b][2 * q] = f2_add(G[0][b][2 * q], m.x); V[0][b][2 * q + 1] = f2_add(G[0][b][2 * q + 1], m.y);
              V[1][b][2 * q] = f2_add(G[1][b][2 * q], m.x); V[1][b][2 * q + 1] = f2_add(G[1][b][2 * q + 1], m.y);
              V[2][b][2 * q] = f2_add(G[1][b][2 * q], o.x); V[2][b][2 * q + 1] = f2_add(G[1][b][2 * q + 1], o.y);
            }
          // horizontal partner (tx+1) by shuffle, scale (0 for plane cells without a pooled value), round, store
          const f2 sc = f2_pack(cell ? 0.25f : 0.f, cell ? 0.25f : 0.f);
#pragma unroll
          for (int A = 0; A < 3; ++A) {
            __half2 o0[4], o1[4], o2[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const f2 n1 = f2_shfl_down1(V[A][1][e]), n2 = f2_shfl_down1(V[A][2][e]);
              float lo, hi;
              f2_unpack(f2_mul(f2_add(V[A][0][e], n1), sc), lo, hi); o0[e] = __floats2half2_rn(lo, hi);
              f2_unpack(f2_mul(f2_add(V[A][1][e], n1), sc), lo, hi); o1[e] = __floats2half2_rn(lo, hi);
              f2_unpack(f2_mul(f2_add(V[A][1][e], n2), sc), lo, hi); o2[e] = __floats2half2_rn(lo, hi);
            }
            if (inplane && A < ncls) {
              __half* dst = pmq + (int64_t(A * 3) * 32 * psz + opos + int64_t(chunk) * psz) * 8;
              *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<uint4*>(o0);
              *reinterpret_cast<uint4*>(dst + int64_t(32) * psz * 8) = *reinterpret_cast<uint4*>(o1);
              if (ncls > 2) *reinterpret_cast<uint4*>(dst + int64_t(64) * psz * 8) = *reinterpret_cast<uint4*>(o2);
            }
          }
          if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2 + pp) * 8 + 5);
        }
      }
      mbar_arrive(bars + 8 * (A_EMPTY0 + buf));               // residual reads (and the MMAs, by their commit) done with A
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

}  // namespace cmlpl

using namespace cmlpl;

CMLPL_TRACE_EXPORT(cmlpl_debug_c1p_trace)

// conv1 variants + pooling fused (conv1_pool_kernel): f0pad -> pooled parity planes, no fp32 scratch
extern "C" int cmlpl_conv1_pool_planes_f16(const void* f0pad, int cols, int w, int band_rows, const void* packed,
                                           void* pmq, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(f0pad && packed && pmq, "conv1_pool_planes: null pointer");
  CMLPL_CHECK_ARG((w == 20 || w == 11) && cols > 0 && band_rows > 0, "conv1_pool_planes: bad dims (w must be 20 or 11)");
  const int PR = band_rows + w - 1, PC = cols + w - 1, PR2 = (PR + 1) / 2, PC2 = (PC + 1) / 2;
  const PackedLayout L = packed_layout(1, 1, w);
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  CMLPL_MAX_DYN_SMEM(conv1_pool_kernel, c1p::SMEM);
  const int ntiles = ((2 * PR2 + c1p::OH - 1) / c1p::OH) * ((2 * PC2 + c1p::OW - 1) / c1p::OW);
  int grid = sm_count(); if (grid > ntiles) grid = ntiles;
  CUtensorMap tm_f0;
  const int trc = make_scene_tmap(&tm_f0, f0pad, 1, PR, PC, c1p::TH + 2, c1p::TP);
  if (trc != CMLPL_OK) return trc;
  conv1_pool_kernel<<<grid, c1p::kThreads, c1p::SMEM, static_cast<cudaStream_t>(stream)>>>(
      tm_f0, PR, PC, PR2, PC2, w == 11 ? 2 : 3, pk + L.w1, reinterpret_cast<const float*>(pk + L.b1), static_cast<__half*>(pmq));
  CMLPL_CHECK_LAUNCH("conv1_pool");
  return CMLPL_OK;
}
