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
// zero-haloed shared-memory tile of 7 rows loaded by TMA:
//   * the tensor core produces, per 32-channel half and tap column dx, four accumulators over two FRAMES of the
//     same 4x32 lanes: frame 0 holds conv rows y0..y0+3 (one per TMEM lane quarter), frame 1 rows y0+1..y0+4,
//     the same lanes one row down (its A rows are frame 0's plus one tile row).  A row offset s of the A tile
//     feeds frame 0 tap dy = s and frame 1 tap dy = s-1, so
//         U  = frame 0 taps dy 1+2 | D = frame 1 taps dy 0+1   (s = 1, 2: one N = 64 MMA each, B = [W1;W0] / [W2;W1])
//         T0 = frame 0 tap  dy 0   | T2 = frame 1 tap  dy 2    (s = 0 / 3: one N = 32 MMA each)
//     (48 MMAs in 384 TMEM columns per half).  The epilogue forms the column classes
//     R[left|mid|right] = R1+R2 | R0+R1+R2 | R0+R1 of each, and the row classes  top = U, mid = T0+U  (frame 0)
//     and  mid = D+T2, bot = D  (frame 1) from one TMEM read;
//   * a tile emits 4 pooled rows x 29 pooled columns: the vertical 2x2 partner of frame 0's row is frame 1's row
//     in the SAME lane, the horizontal partner (tx+1) comes through a warp shuffle -- no exchange between warps;
//   * pooled cells go straight to the parity planes pmq (f16, chunk-planar), 8 channels = one 16-byte chunk
//     per thread and pass.
//   V[A][b]  = G[a0(A)][b](y,x) + G[a1(A)][b](y+1,x)                 (a0,a1 = top,mid | mid,mid | mid,bot)
//   PM[A][B] = 1/4 (V[A][b0(B)](x) + V[A][b1(B)](x+1))               (b0,b1 = left,mid | mid,mid | mid,right)
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "tma.cuh"

namespace cmlpl {

namespace c1p {
constexpr int TH = 4, TP = 32, OH = 4, OW = 29;      // conv rows per frame, row pitch; pooled rows / columns per tile
constexpr int AR = TH + 3;                           // 7 A-tile rows: frame 1 sits one row below frame 0, +1 halo row each side
constexpr int CH = AR * TP * 16;                     // 3 584: one chunk plane of the conv0 tile, dense (written by TMA)
constexpr int ABYTES = 8 * CH, NBUF = 3;
constexpr int WBYTES = 3 * 8 * 192 * 16;
constexpr int kEpi = 256, kThreads = kEpi + 64;      // warps 0-7 epilogue, warp 8 loader (one thread, TMA), warp 9 MMA issuer
constexpr int kLoadWarp = kEpi / 32, kMmaWarp = kLoadWarp + 1;
constexpr int S_W = 0, S_A = WBYTES, S_BIAS = S_A + NBUF * ABYTES, S_BAR = S_BIAS + 256, S_TMEM = S_BAR + 128;
constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
// TMEM columns of one channel half, per tap column dx (at dx * 128): [U | D] 0..63, T0 64..95, T2 96..127
constexpr int HALFCOLS = 384, C_UD = 0, C_T0 = 64, C_T2 = 96;
// weights in shared memory: [3 dx][8 kc][2 h][W2h W1h W0h: 96 rows][16 B], so [W2h;W1h] and [W1h;W0h] are contiguous
// N = 64 operands.  In HBM (the packed layout patch_cnn_kernel shares) a (dx, kc) block is [(2-dy)*64 + n][16 B].
constexpr int kWLbo = 192 * 16, kWDx = 8 * kWLbo;
enum { A_FULL0 = 0, A_EMPTY0 = NBUF, S_FULL = 2 * NBUF, S_EMPTY, W_FULL };
static_assert(SMEM <= 232448, "conv1_pool: shared memory over the 227 KB limit");
static_assert(W_FULL < 16, "conv1_pool: barrier area too small");
static_assert(S_A % 128 == 0 && ABYTES % 128 == 0, "conv1_pool: TMA destinations must be 128-byte aligned");
static_assert(HALFCOLS <= 512, "conv1_pool: a channel half must fit tensor memory");
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
  // Tiles run from the bottom of the band up, so the planes written last -- still in L2 when the kernel ends -- are the
  // top rows, which conv2_scene_kernel reads first.

  {
    uint4* z = reinterpret_cast<uint4*>(smem + S_A);
    for (int i = tid; i < NBUF * ABYTES / 16; i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (tid < 64) sbias[tid] = b1g[tid];
  if (tid == 0) {
    mbar_init(bars + 8 * W_FULL, 1);
    fence_barrier_init();
    // 144 bulk copies of 512 B (32 rows of one (dx, kc, dy, h)) permute the weights into the half-interleaved order
    mbar_arrive_expect_tx(bars + 8 * W_FULL, WBYTES);
#pragma unroll 1
    for (int i = 0; i < 3 * 8 * 6; ++i) {
      const int blk = i / 6, dy = (i % 6) >> 1, h = i & 1;
      bulk_g2s(sbase + S_W + (blk * 192 + h * 96 + (2 - dy) * 32) * 16, w1p + (blk * 192 + (2 - dy) * 64 + h * 32) * 16,
               512, bars + 8 * W_FULL);
    }
    for (int b = 0; b < NBUF; ++b) { mbar_init(bars + 8 * (A_FULL0 + b), 1); mbar_init(bars + 8 * (A_EMPTY0 + b), 1 + kEpi); }
    mbar_init(bars + 8 * S_FULL, 1); mbar_init(bars + 8 * S_EMPTY, kEpi);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(sbase + S_TMEM, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);

  if (warp == kLoadWarp) {
    // ================================================================ loader: one TMA box per tile (AR x TP entries, zero outside the map)
    if (lane == 0) {
      tma_prefetch_desc(&tm_f0);
      uint32_t j = 0, buf = 0, ph = 0;
      [[maybe_unused]] uint32_t ntr = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
        const int u = ntiles - 1 - t, tr = u / tiles_c, tc = u - tr * tiles_c;   // bottom tile rows first (see above)
        mbar_wait(bars + 8 * (A_EMPTY0 + buf), ph ^ 1, 81);
        CMLPL_TR(4, ntr, j);
        mbar_arrive_expect_tx(bars + 8 * (A_FULL0 + buf), ABYTES);
        tma_load_tile(sbase + S_A + buf * ABYTES, &tm_f0, tc * OW - 1, tr * OH - 1, 0, bars + 8 * (A_FULL0 + buf));
        if (++buf == NBUF) { buf = 0; ph ^= 1; }
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer
    if (tmem != 0) { printf("conv1_pool: unexpected TMEM base %u\n", tmem); __trap(); }
    constexpr uint64_t kHi = (uint64_t(128 >> 4) | (uint64_t(1) << 14)) << 32;
    constexpr uint32_t kI32 = make_idesc_f16(128, 32), kI64 = make_idesc_f16(128, 64);
    const uint32_t w_lo = ((sbase + S_W) >> 4) | (uint32_t(kWLbo >> 4) << 16);
    uint32_t j = 0, buf = 0, ph = 0, sph = 0;
    [[maybe_unused]] uint32_t ntr = 0;
    mbar_wait(bars + 8 * W_FULL, 0, 80);                       // weights have landed
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
      // MMA row m at A row offset s, tap column dx reads tile entry m + s*TP + dx - 1: descriptors start 16 B before the tile
      const uint32_t a_lo = ((sbase + S_A + buf * ABYTES - 16) >> 4) | (uint32_t(CH >> 4) << 16);
      mbar_wait(bars + 8 * (A_FULL0 + buf), ph, 82);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {                            // one channel half = one TMEM slot of 384 columns
        if (lane == 0) CMLPL_TR(0, ntr, (j * 2 + h) * 4);
        mbar_wait(bars + 8 * S_EMPTY, sph ^ 1, 83);
        tc_fence_after();
        if (lane == 0) CMLPL_TR(0, ntr, (j * 2 + h) * 4 + 1);
        if (elect_one_sync()) {
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            const uint32_t d = dx * 128;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t a = a_lo + uint32_t(dx) + uint32_t(ks * 2 * CH / 16);
              const uint32_t bb = w_lo + uint32_t((dx * kWDx + ks * 2 * kWLbo) / 16) + uint32_t(h * 96);
              const uint32_t acc = ks ? 1u : 0u;
              umma_f16(d + C_UD, kHi | uint64_t(a + 1 * TP), kHi | uint64_t(bb + 32), kI64, acc);   // [U|D] += [W1;W0]
              umma_f16(d + C_UD, kHi | uint64_t(a + 2 * TP), kHi | uint64_t(bb), kI64, 1u);         // [U|D] += [W2;W1]
              umma_f16(d + C_T0, kHi | uint64_t(a), kHi | uint64_t(bb + 64), kI32, acc);            // T0 += W0
              umma_f16(d + C_T2, kHi | uint64_t(a + 3 * TP), kHi | uint64_t(bb), kI32, acc);        // T2 += W2
            }
          }
          umma_commit(bars + 8 * S_FULL);
          if (h == 1) umma_commit(bars + 8 * (A_EMPTY0 + buf));
        }
        __syncwarp();
        if (lane == 0) CMLPL_TR(0, ntr, (j * 2 + h) * 4 + 2);
        sph ^= 1;
      }
      if (++buf == NBUF) { buf = 0; ph ^= 1; }
    }
  } else {
    // ================================================================ epilogue (warps 0-7, each on its own lane quarter)
    const int ty = warp & 3, tx = lane, chsel = warp >> 2;
    const uint32_t lane_addr = uint32_t(ty * 32) << 16;
    uint32_t j = 0, buf = 0, ph = 0, sph = 0;
    [[maybe_unused]] uint32_t ntr = 0;
    const bool tracer = (warp == 0 || warp == 4) && lane == 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
      const int u = ntiles - 1 - t, tr = u / tiles_c, tc = u - tr * tiles_c;   // bottom tile rows first (see above)
      const int pr = tr * OH + ty, pc = tc * OW + tx - 1;
      const bool inplane = tx >= 1 && tx <= OW && (pr >> 1) < PR2 && (pc >> 1) < PC2;
      const bool cell = inplane && pr < PR - 1 && pc < PC - 1;
      const int64_t opos = inplane ? (int64_t((pr & 1) * 2 + (pc & 1)) * 8 * psz + int64_t(pr >> 1) * PC2 + (pc >> 1)) : 0;
      const unsigned char* abuf = smem + S_A + buf * ABYTES;
      mbar_wait(bars + 8 * (A_FULL0 + buf), ph, 84);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2) * 8);
        mbar_wait(bars + 8 * S_FULL, sph, 85);
        sph ^= 1;
        tc_fence_after();
        if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2) * 8 + 1);
#pragma unroll 1
        for (int pp = 0; pp < 2; ++pp) {
          const int chunk = h * 4 + pp * 2 + chsel;
          const uint32_t col = uint32_t(pp * 16 + chsel * 8);
          typedef unsigned long long f2;                       // two packed fp32 channels (FADD2 / FMUL2)
          f2 U[3][4], D[3][4], T0[3][4], T2[3][4];
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            const uint32_t ta = lane_addr + dx * 128 + col;
            tmem_ld8_x2(ta + C_UD, U[dx]);
            tmem_ld8_x2(ta + C_UD + 32, D[dx]);
            tmem_ld8_x2(ta + C_T0, T0[dx]);
            tmem_ld8_x2(ta + C_T2, T2[dx]);
          }
          tmem_ld_wait();
          if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2 + pp) * 8 + 2);
          if (pp == 1) {                                       // the MMAs of the next half may overwrite the slot
            tc_fence_before();
            mbar_arrive(bars + 8 * S_EMPTY);
          }
          {
            // bias + residual (centre entry of the A tile, frame 0 row ty+1 / frame 1 row ty+2) go into the centre
            // tap, which every border class keeps
            const uint4 r0 = *reinterpret_cast<const uint4*>(abuf + chunk * CH + ((ty + 1) * TP + tx) * 16);
            const uint4 r1 = *reinterpret_cast<const uint4*>(abuf + chunk * CH + ((ty + 2) * TP + tx) * 16);
            const __half2* h0 = reinterpret_cast<const __half2*>(&r0);
            const __half2* h1 = reinterpret_cast<const __half2*>(&r1);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float b0 = sbias[chunk * 8 + 2 * e], b1 = sbias[chunk * 8 + 2 * e + 1];
              const float2 f = __half22float2(h0[e]), g = __half22float2(h1[e]);
              U[1][e] = f2_add(U[1][e], f2_pack(f.x + b0, f.y + b1));
              D[1][e] = f2_add(D[1][e], f2_pack(g.x + b0, g.y + b1));
            }
          }
          // G[a][b] = relu(b1 + F0 + sum of the taps the (row class a, column class b) border keeps), and the
          // vertical pool  V[A][b] = G0[a0(A)][b] + G1[a1(A)][b]  in the same lane
          f2 V[3][3][4];                                       // [A][b]
#pragma unroll
          for (int c = 0; c < 4; ++c) {
#pragma unroll
            for (int b = 0; b < 3; ++b) {
              // column class b of a tap-column triple: left = 1+2, mid = 0+1+2, right = 0+1
              auto cls = [&](const f2 (&X)[3][4]) {
                return b == 0 ? f2_add(X[1][c], X[2][c])
                              : b == 1 ? f2_add(X[0][c], f2_add(X[1][c], X[2][c])) : f2_add(X[0][c], X[1][c]);
              };
              const f2 u = cls(U), d = cls(D);
              const f2 g0top = f2_relu(u), g0mid = f2_relu(f2_add(cls(T0), u));
              const f2 g1mid = f2_relu(f2_add(cls(T2), d)), g1bot = f2_relu(d);
              V[0][b][c] = f2_add(g0top, g1mid);
              V[1][b][c] = f2_add(g0mid, g1mid);
              V[2][b][c] = f2_add(g0mid, g1bot);
            }
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
          if (tracer) CMLPL_TR(1 + chsel, ntr, (j * 4 + h * 2 + pp) * 8 + 3);
        }
      }
      mbar_arrive(bars + 8 * (A_EMPTY0 + buf));               // residual reads (and the MMAs, by their commit) done with A
      if (++buf == NBUF) { buf = 0; ph ^= 1; }
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
  const int trc = make_scene_tmap(&tm_f0, f0pad, 1, PR, PC, c1p::AR, c1p::TP);
  if (trc != CMLPL_OK) return trc;
  conv1_pool_kernel<<<grid, c1p::kThreads, c1p::SMEM, static_cast<cudaStream_t>(stream)>>>(
      tm_f0, PR, PC, PR2, PC2, w == 11 ? 2 : 3, pk + L.w1, reinterpret_cast<const float*>(pk + L.b1), static_cast<__half*>(pmq));
  CMLPL_CHECK_LAUNCH("conv1_pool");
  return CMLPL_OK;
}
