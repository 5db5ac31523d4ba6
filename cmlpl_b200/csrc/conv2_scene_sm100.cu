// Scene-level conv2 + pool + classifier with exact compute sharing (SURVEY section 7 / 8-f3, second half).
//
// After conv1_pool_kernel (conv1_scene_sm100.cu) the pooled conv1 window of pixel (r,c) is  PM[A(i)][B(j)][r+2i, c+2j]  (i,j = 0..9,
// A/B = top/mid/bot border class of the pooled row/column).  Everything downstream of it
// (tools/models.py:137-150: conv2 3x3 with zero padding at the PATCH border, +residual, ReLU, 2x2
// average pool, the conv columns of the classifier) again depends only on the scene position and on
// which border the patch cuts, so it is evaluated ONCE per scene position instead of once per pixel:
//
//   * positions (r+2i, c+2j) keep the parity of (r,c): the padded map splits into 4 PARITY PLANES
//     (y' = pr>>1, x' = pc>>1) on which conv2 is a plain 3x3 convolution and the pool a 2x2 window;
//   * conv2 output row i of a patch has row class rho(i) in {0: i=0, 1: i=1, 2: i=2..7, 3: i=8, 4: i=9}
//     (which taps the border drops AND which PM row class each remaining tap reads); same for columns:
//       Y[rho][kap][y',x'] = relu(b2 + PM[A(rho)][B(kap)][y',x']
//                                 + sum_{di in S(rho), dj in S(kap)} W2[di,dj] . PM[A(rho,di)][B(kap,dj)][y'+di, x'+dj])
//     -> conv2_scene_kernel: 25 variants per position, 169 tap products instead of 900 per pixel;
//   * pool + classifier are linear after the ReLU:  logit_conv(r,c) = sum_{I,J} L[I][J][r'+2I, c'+2J] with
//       L[I][J][y',x'] = sum_{u,v in {0,1}} (Wc[I,J]/4) . Y[rho(2I+u)][kap(2J+v)][y'+u, x'+v]
//     The border halves of that 2x2 pool pair two DIFFERENT variants at neighbouring positions (rho 0 with rho 1 one row
//     down, rho 3 with rho 4, and the same for kap), so conv2_scene_kernel's epilogue adds them before anything is
//     stored (the partner sits in the same TMEM lane because the accumulator frames are shifted accordingly) and writes
//     9 half-pooled maps  YP[Al][Be]  (Al, Be = border / middle / border) instead of 25 variants: 1 152 B per position
//     through HBM instead of 3 200;
//     -> pool2_cls_kernel: the remaining pool of the middle classes is accumulating tcgen05.mma whose A descriptors are
//        shifted by (u,v) inside the tile; 25 maps of 16 class partials per position;
//   * the head (head_sm100.cu) adds the 25 gathered partials of a pixel to its spectral logits.
//
// Identical math up to fp32 summation order; per PaviaU scene conv2 executes 0.32 TFLOP instead of 1.53.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "tma.cuh"

namespace cmlpl {

// =================================================================================================
// conv2_scene_kernel: persistent, warp-specialised tcgen05 implicit GEMM over 4x30-position tiles of a
// parity plane (M = 128 rows = 4 rows x 32 columns incl. one halo column each side; taps = A-descriptor
// offsets in zero-haloed row-major tiles).  Per tile the nine PM variant tiles are loaded once by TMA (one
// 24 KB box each, zero fill outside the plane), as three "slabs" of 3 row classes x one column class:
//     slab X <- left, slab M <- mid   : column classes kap = 0, 1
//                        (mid only)    : kap = 2
//     slab X <- right                  : kap = 3, 4
// ROW-TAP FUSION.  The five row classes rho = 0..4 of a column class are the conv2 output rows i = 0,1,4,8,9 of a
// patch, and output row i reads pooled rows i-1, i, i+1: consecutive classes share input rows.  The accumulator
// of class rho is kept in a frame shifted DOWN by rho rows (its row (ty,tx) is plane position (Y0+ty+rho, .)),
// so tap dy of class rho and tap dy-1 of class rho+1 read the SAME shared-memory rows of the same PM row-class
// tile; with the accumulators of rho = 0..4 in adjacent 64-column TMEM blocks and the weights stacked per dx as
// 192 rows [W(dy=2); W(dy=1); W(dy=0)], the 13 row taps of a (kap, dx) become five MMAs:
//     PA  N=128 [rho0|rho1]      <- PM top  (tile rows +1)  x [W1;W0]
//     T1  N=192 [rho0|rho1|rho2] <- PM mid  (tile rows +2)  x [W2;W1;W0]
//     T2  N=192 [rho1|rho2|rho3] <- PM mid  (tile rows +3)
//     T3  N=192 [rho2|rho3|rho4] <- PM mid  (tile rows +4)
//     PB  N=128 [rho3|rho4]      <- PM bot  (tile rows +5)  x [W2;W1]
// i.e. 416 tensor-core cycles instead of 13 x 64 = 832 (a tcgen05.mma of M=128,K=16 costs ~64 cycles up to N=128
// and 96 at N=192).  Issued group by group over all dx, the accumulators complete in the order rho0, rho1, rho2,
// rho3+rho4, so the epilogue (bias + residual + ReLU -> fp16) of one class overlaps the MMAs of the next groups
// and the single 320-column accumulator set is reused by the next column class as its blocks drain.  Rows
// y < rho of class rho are never produced -- no pixel reads them (pooled row i >= rho for that class).
// HALF POOL IN THE EPILOGUE.  The frames put Y[rho0](y) and Y[rho1](y+1) -- the two rows of pooled cell I = 0 -- in the
// same TMEM lane, likewise rho3 / rho4 (I = 4), so an epilogue thread adds them in registers.  Columns work the same way
// in time: the frame of kap = 0 is shifted one entry LEFT and that of kap = 4 one entry RIGHT (an A-descriptor offset;
// the taps the patch border cuts off are exactly the ones that would leave the tile), the row-pooled result of kap = 0
// (kap = 3) is parked as fp32 in the 192 TMEM columns the accumulators leave free (tcgen05.st) and added when
// kap = 1 (kap = 4) drains.  Per position the kernel stores 9 maps  YP[Al*3+Be]  (Al: rho {0+1 | 2 | 3+4}, Be alike),
// each the AVERAGE of its pre-pooled partners; the classifier block weights carry the matching factor (pack.cu).
namespace c2s {
constexpr int TH = 4, TP = 32, TW = 30;
constexpr int CH = (TH + 2) * TP * 16;               // 3 072: one chunk plane of a tile, dense (written by TMA)
constexpr int TBYTES = 8 * CH;                       // 24 576: one PM variant tile (6 rows)
constexpr int WBYTES = 3 * 8 * 192 * 16;             // 73 728
constexpr int S_W = 0, S_T = WBYTES, S_BIAS = S_T + 6 * TBYTES, S_BAR = S_BIAS + 256, S_TMEM = S_BAR + 256;
constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
constexpr int kEpi = 256, kThreads = kEpi + 64;      // warps 0-7 epilogue, warp 8 loader (one thread, TMA), warp 9 MMA issuer
constexpr int kLoadWarp = kEpi / 32, kMmaWarp = kLoadWarp + 1;
constexpr int kWLbo = 192 * 16, kWDx = 8 * kWLbo;
// one full / empty mbarrier per resident class tile (slab X or M x row class a), so the next tile's loads start as each
// tile is released (top tiles after the PA group of the last column class that reads them, ...) instead of after the
// whole slab; DF/DE: accumulator block of row class rho full / drained
enum { XF0 = 0, MF0 = 3, XE0 = 6, ME0 = 9, DF0 = 12, DE0 = 17, W_FULL = 22 };
constexpr int kPark = 320;                           // first TMEM column of the three parked 64-column items
static_assert(SMEM <= 232448, "conv2_scene: shared memory over the 227 KB limit");
static_assert(S_T % 128 == 0 && TBYTES % 128 == 0, "conv2_scene: TMA destinations must be 128-byte aligned");
// first tile row (relative to Y0 - 1) held by the tile of PM row class a: top rows +1.., mid +2.., bot +5..
__host__ __device__ constexpr int tile_r0(int a) { return a == 0 ? 1 : (a == 1 ? 2 : 5); }

// group G (0 = PA, 1..3 = T1..T3, 4 = PB) of column class KAP: every dx tap x 4 k-steps.  t_lo = low descriptor word of
// tile 0 minus 16 B (MMA row m of tap dx reads entry m + dx - 1), w_lo = weight block of dx = 0.  All offsets immediate.
// W11 (11x11 windows): only the row classes rho = 0, 1, 2 exist, so T2 feeds [rho1|rho2] (N=128), T3 [rho2] (N=64), no PB.
template <int KAP, int G, bool W11 = false>
__device__ __forceinline__ void issue_group(uint32_t t_lo, uint32_t w_lo) {
  constexpr uint64_t kHi = (uint64_t(128 >> 4) | (uint64_t(1) << 14)) << 32;   // SBO = 128 B, version 1
  constexpr int a = G == 0 ? 0 : (G == 4 ? 2 : 1);
  constexpr int o = G == 0 ? 1 : (G == 4 ? 5 : G + 1);
  constexpr int d = G == 0 ? 0 : (G == 4 ? 192 : (G - 1) * 64);
  constexpr int N = W11 ? (G == 1 ? 192 : (G == 3 ? 64 : 128)) : ((G == 0 || G == 4) ? 128 : 192);
  constexpr int brow = G == 0 ? 64 : 0;
  constexpr int dx_first = rep_of(KAP) == 0 ? 1 : 0;
  constexpr int xs = KAP == 0 ? -1 : (KAP == 4 ? 1 : 0);          // frame shift of the border column classes (entries)
#pragma unroll
  for (int dx = 0; dx < 3; ++dx) {
    const int j2 = rep_of(KAP) + dx - 1;
    if (j2 < 0 || j2 > 9) continue;
    const int tile = (cls_of(j2) == 1 ? 3 : 0) + a;               // slab M holds the mid column class
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t aa = t_lo + uint32_t((tile * TBYTES + ((o - tile_r0(a)) * TP + dx + xs) * 16 + ks * 2 * CH) / 16);
      const uint32_t bb = w_lo + uint32_t((dx * kWDx + ks * 2 * kWLbo) / 16) + uint32_t(brow);
      const bool first = dx == dx_first && ks == 0;
      if (first && G >= 1 && G <= (W11 ? 1 : 3)) {
        // the group's third accumulator starts here (overwrite); the other two already hold earlier groups
        umma_f16(uint32_t(d), kHi | uint64_t(aa), kHi | uint64_t(bb), make_idesc_f16(128, 128), 1u);
        umma_f16(uint32_t(d + 128), kHi | uint64_t(aa), kHi | uint64_t(bb + 128), make_idesc_f16(128, 64), 0u);
      } else {
        umma_f16(uint32_t(d), kHi | uint64_t(aa), kHi | uint64_t(bb), make_idesc_f16(128, N), (first && G == 0) ? 0u : 1u);
      }
    }
  }
}
}  // namespace c2s

// pmq f16 [9][4][8][PR2][PC2][8];  yq f16 [9 = Al*3+Be half-pooled maps][4][8][PR2][PC2][8]
// W11: the instantiation for 11x11 windows -- column / row classes 0, 1, 2 only (64 of the 169 tap products), top and
// mid-row tiles of the left and mid column classes only (4 of the 9 class tiles), maps Al, Be in {0, 1} written.
template <bool W11>
__global__ void __launch_bounds__(c2s::kThreads, 1)
conv2_scene_kernel(const __grid_constant__ CUtensorMap tm_pm, const __half* __restrict__ pmq, int PR2, int PC2,
                   const unsigned char* __restrict__ w2p, const float* __restrict__ b2g, __half* __restrict__ yq) {
  using namespace c2s;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + S_BAR;
  float* sbias = reinterpret_cast<float*>(smem + S_BIAS);
  const int tiles_c = (PC2 + TW - 1) / TW, tiles_r = (PR2 + TH - 1) / TH;
  const int tiles_p = tiles_r * tiles_c, ntiles = 4 * tiles_p;
  const int64_t psz = int64_t(PR2) * PC2;

  {
    uint4* z = reinterpret_cast<uint4*>(smem + S_T);
    for (int i = tid; i < 6 * TBYTES / 16; i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (tid < 64) sbias[tid] = b2g[tid];
  if (tid == 0) {
    mbar_init(bars + 8 * W_FULL, 1);
    fence_barrier_init();
    bulk_weights_g2s(sbase + S_W, w2p, WBYTES, bars + 8 * W_FULL);
    for (int a = 0; a < 3; ++a) {
      mbar_init(bars + 8 * (XF0 + a), 1); mbar_init(bars + 8 * (MF0 + a), 1);
      // released by the MMA commit after the last group that reads this class tile (the epilogue takes its residuals
      // from global memory, so nothing else reads the tiles)
      mbar_init(bars + 8 * (XE0 + a), 1); mbar_init(bars + 8 * (ME0 + a), 1);
    }
    for (int s = 0; s < 5; ++s) { mbar_init(bars + 8 * (DF0 + s), 1); mbar_init(bars + 8 * (DE0 + s), kEpi); }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(sbase + S_TMEM, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);

  if (warp == kLoadWarp) {
    // ================================================================ loader: one thread, three TMA boxes per slab
    if (lane == 0) {
      tma_prefetch_desc(&tm_pm);
      uint32_t fx[3] = {0, 0, 0}, fm[3] = {0, 0, 0};           // fills of each class tile of slab X / slab M so far
      [[maybe_unused]] uint32_t ntr = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int pl = t / tiles_p, tt = t - pl * tiles_p;
        const int tr = tt / tiles_c, tc = tt - tr * tiles_c;
        const int y0 = tr * TH - 1, x0 = tc * TW - 1;          // borders zero-filled; tile of row class a starts at row y0 + tile_r0(a)
        // left and mid tiles interleaved in the order the MMA groups need them (top, mid, bottom), then the right tiles
#pragma unroll
        for (int i = 0; i < (W11 ? 4 : 9); ++i) {
          const int a = i < 6 ? i >> 1 : i - 6;
          const int slab = i < 6 ? (i & 1) : 0, bcls = i < 6 ? (i & 1) : 2;
          const uint32_t k = slab ? fm[a] : fx[a];
          const uint32_t full = bars + 8 * ((slab ? MF0 : XF0) + a);
          mbar_wait(bars + 8 * ((slab ? ME0 : XE0) + a), (k & 1) ^ 1, 61);
          mbar_arrive_expect_tx(full, TBYTES);
          CMLPL_TR(3, ntr, uint32_t(i));
          tma_load_tile(sbase + S_T + (slab * 3 + a) * TBYTES, &tm_pm, x0, y0 + tile_r0(a), (a * 3 + bcls) * 4 + pl, full);
          if (slab) ++fm[a]; else ++fx[a];
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer
    if (tmem != 0) { printf("conv2_scene: unexpected TMEM base %u\n", tmem); __trap(); }
    const uint32_t t_lo = ((sbase + S_T - 16) >> 4) | (uint32_t(CH >> 4) << 16);
    const uint32_t w_lo = ((sbase + S_W) >> 4) | (uint32_t(kWLbo >> 4) << 16);
    uint32_t cx[3] = {0, 0, 0}, cm[3] = {0, 0, 0}, kc = 0;     // class-tile fills consumed, column-class stages issued
    [[maybe_unused]] uint32_t ntr = 0;
#define C2S_GROUP(KAP, G, ...)                                                       \
    do {                                                                             \
      tc_fence_after();                                                              \
      if (lane == 0) CMLPL_TR(0, ntr, KAP * 16 + G * 2);                               \
      if (elect_one_sync()) { issue_group<KAP, G>(t_lo, w_lo); __VA_ARGS__; }        \
      __syncwarp();                                                                  \
      if (lane == 0) CMLPL_TR(0, ntr, KAP * 16 + G * 2 + 1);                           \
    } while (0)
    // WX / WM: this column class is the first to read a fresh fill of slab X / M (wait per class tile, just before the
    // first group that reads it); RX / RM: it is the last to read the resident fill (release per class tile)
#define C2S_FILL(A, WX, WM)                                                          \
    do {                                                                             \
      if (WX) { mbar_wait(bars + 8 * (XF0 + A), cx[A] & 1, 62); ++cx[A]; }           \
      if (WM) { mbar_wait(bars + 8 * (MF0 + A), cm[A] & 1, 62); ++cm[A]; }           \
    } while (0)
#define C2S_REL(A, RX, RM) ((RX) ? umma_commit(bars + 8 * (XE0 + A)) : (void)0, (RM) ? umma_commit(bars + 8 * (ME0 + A)) : (void)0)
#define C2S_COLUMN(KAP, WX, WM, RX, RM)                                              \
    do {                                                                             \
      const uint32_t ep = (kc & 1) ^ 1;                                              \
      C2S_FILL(0, WX, WM);                                                           \
      mbar_wait(bars + 8 * (DE0 + 0), ep, 63); mbar_wait(bars + 8 * (DE0 + 1), ep, 63);                       \
      C2S_GROUP(KAP, 0, C2S_REL(0, RX, RM));                                         \
      C2S_FILL(1, WX, WM);                                                           \
      mbar_wait(bars + 8 * (DE0 + 2), ep, 63);                                       \
      C2S_GROUP(KAP, 1, umma_commit(bars + 8 * (DF0 + 0)));                          \
      mbar_wait(bars + 8 * (DE0 + 3), ep, 63);                                       \
      C2S_GROUP(KAP, 2, umma_commit(bars + 8 * (DF0 + 1)));                          \
      mbar_wait(bars + 8 * (DE0 + 4), ep, 63);                                       \
      C2S_GROUP(KAP, 3, (umma_commit(bars + 8 * (DF0 + 2)), C2S_REL(1, RX, RM)));    \
      C2S_FILL(2, WX, WM);                                                           \
      C2S_GROUP(KAP, 4, (umma_commit(bars + 8 * (DF0 + 3)), umma_commit(bars + 8 * (DF0 + 4)), C2S_REL(2, RX, RM)));   \
      ++kc;                                                                          \
    } while (0)
    // Column classes whose class tiles are resident (or landed long ago) issue their five groups in two runs, PA + T1 and
    // T2 + T3 + PB: every barrier poll between two groups is a few hundred cycles in which the issue queue runs dry.
#define C2S_COLUMN2(KAP, WX, RX, RM)                                                 \
    do {                                                                             \
      const uint32_t ep = (kc & 1) ^ 1;                                              \
      if (WX) { C2S_FILL(0, true, false); C2S_FILL(1, true, false); C2S_FILL(2, true, false); }              \
      mbar_wait(bars + 8 * (DE0 + 0), ep, 63); mbar_wait(bars + 8 * (DE0 + 1), ep, 63); mbar_wait(bars + 8 * (DE0 + 2), ep, 63);   \
      tc_fence_after();                                                              \
      if (lane == 0) CMLPL_TR(0, ntr, KAP * 16 + 0);                                 \
      if (elect_one_sync()) {                                                        \
        issue_group<KAP, 0>(t_lo, w_lo); C2S_REL(0, RX, RM);                         \
        issue_group<KAP, 1>(t_lo, w_lo); umma_commit(bars + 8 * (DF0 + 0));          \
      }                                                                              \
      __syncwarp();                                                                  \
      if (lane == 0) CMLPL_TR(0, ntr, KAP * 16 + 3);                                 \
      mbar_wait(bars + 8 * (DE0 + 3), ep, 63); mbar_wait(bars + 8 * (DE0 + 4), ep, 63);                       \
      tc_fence_after();                                                              \
      if (lane == 0) CMLPL_TR(0, ntr, KAP * 16 + 4);                                 \
      if (elect_one_sync()) {                                                        \
        issue_group<KAP, 2>(t_lo, w_lo); umma_commit(bars + 8 * (DF0 + 1));          \
        issue_group<KAP, 3>(t_lo, w_lo); umma_commit(bars + 8 * (DF0 + 2)); C2S_REL(1, RX, RM);              \
        issue_group<KAP, 4>(t_lo, w_lo); umma_commit(bars + 8 * (DF0 + 3)); umma_commit(bars + 8 * (DF0 + 4)); C2S_REL(2, RX, RM);   \
      }                                                                              \
      __syncwarp();                                                                  \
      if (lane == 0) CMLPL_TR(0, ntr, KAP * 16 + 9);                                 \
      ++kc;                                                                          \
    } while (0)
    // 11x11 windows: three column classes, groups PA, T1, T2 (two accumulators), T3 (one); top and mid-row tiles only
#define C2S_GROUP11(KAP, G, ...)                                                     \
    do {                                                                             \
      tc_fence_after();                                                              \
      if (elect_one_sync()) { issue_group<KAP, G, true>(t_lo, w_lo); __VA_ARGS__; }  \
      __syncwarp();                                                                  \
    } while (0)
#define C2S_COLUMN11(KAP, WX, WM, RX, RM)                                            \
    do {                                                                             \
      const uint32_t ep = (kc & 1) ^ 1;                                              \
      C2S_FILL(0, WX, WM);                                                           \
      mbar_wait(bars + 8 * (DE0 + 0), ep, 63); mbar_wait(bars + 8 * (DE0 + 1), ep, 63);                       \
      C2S_GROUP11(KAP, 0, C2S_REL(0, RX, RM));                                       \
      C2S_FILL(1, WX, WM);                                                           \
      mbar_wait(bars + 8 * (DE0 + 2), ep, 63);                                       \
      C2S_GROUP11(KAP, 1, (umma_commit(bars + 8 * (DF0 + 0)), (void)0));             \
      C2S_GROUP11(KAP, 2, (umma_commit(bars + 8 * (DF0 + 1)), (void)0));             \
      C2S_GROUP11(KAP, 3, (umma_commit(bars + 8 * (DF0 + 2)), C2S_REL(1, RX, RM)));  \
      ++kc;                                                                          \
    } while (0)
    mbar_wait(bars + 8 * c2s::W_FULL, 0, 60);                  // weights have landed
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      if constexpr (W11) {
        C2S_COLUMN11(0, true, true, false, false);             // left + mid arrive
        C2S_COLUMN11(1, false, false, true, false);            // last reader of the left tiles
        C2S_COLUMN11(2, false, false, false, true);            // last reader of the mid tiles
      } else {
        C2S_COLUMN(0, true, true, false, false);               // left + mid arrive: group by group, as the tiles land
        C2S_COLUMN2(1, false, true, false);                    // last reader of the left tiles
        C2S_COLUMN2(2, false, false, false);
        C2S_COLUMN2(3, true, false, false);                    // right tiles (loaded during the first two classes)
        C2S_COLUMN2(4, false, true, true);                     // last reader of the right and mid tiles
      }
    }
#undef C2S_COLUMN11
#undef C2S_GROUP11
#undef C2S_COLUMN2
#undef C2S_COLUMN
#undef C2S_REL
#undef C2S_FILL
#undef C2S_GROUP
  } else {
    // ================================================================ epilogue (warps 0-7)
    // Work items = (column class kap, row item it): it 0 = rho 0 + rho 1, it 1 = rho 2, it 2 = rho 3 + rho 4.  A thread owns
    // one position (TMEM lane) and 32 of its 64 channels: warps 0-3 take channels 0..31 of every item, warps 4-7 channels
    // 32..63, so an accumulator block is back with the MMA issuer one TMEM load after it completes.
    const int L = (warp & 3) * 32 + lane, hf = warp >> 2;
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const int ty = L >> 5, tx = L & 31;
    const float* bb = sbias + hf * 32;
    const int64_t cstep = psz * 8;                             // halves between the chunk planes of one map
    [[maybe_unused]] uint32_t ntr = 0;
    uint32_t kc = 0;                                           // column-class stage (phase of the DF barriers)
#pragma unroll 1
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const int pl = t / tiles_p, tt = t - pl * tiles_p, tr = tt / tiles_c, tc = tt - tr * tiles_c;
      const int yb = tr * TH + ty, xb = tc * TW + tx - 1;      // plane position of this lane in an unshifted frame
      const __half* pm_t = pmq + (int64_t(pl) * 8 + hf * 4) * cstep;
      __half* yq_t = yq + (int64_t(pl) * 8 + hf * 4) * cstep;
#pragma unroll 1
      for (int kap = 0; kap < (W11 ? 3 : 5); ++kap, ++kc) {
        const int xs = kap == 0 ? -1 : (kap == 4 ? 1 : 0);     // frame shift of this column class (entries)
        const int bcl = kap == 0 ? 0 : (kap == 4 ? 2 : 1);     // PM column class of the centre tap
        const int Be = kap <= 1 ? 0 : (kap == 2 ? 1 : 2);
        const bool park = kap == 0 || kap == 3, unpark = kap == 1 || kap == 4;
        // pooled cell column = the LEFT column of the pair: kap 1 holds column x+1 of the cell whose column x kap 0 parked
        const int xo = xb + xs, x = xb - (kap == 1 ? 1 : 0);
        const bool xok = xo >= 0 && xo < PC2, xval = tx >= 1 && tx <= TW && x >= 0 && x < PC2;
#pragma unroll
        for (int it = 0; it < (W11 ? 2 : 3); ++it) {
          constexpr int kRho0[3] = {0, 2, 3};
          const int rho0 = kRho0[it], nrho = it == 1 ? 1 : 2;
          // residual of row class rho = centre cell PM[A(rho)][B(kap)] at the variant's own position.  It is read from
          // GLOBAL memory (L2: the loader has just pulled the same tiles) rather than from the class tiles in shared
          // memory, and before the accumulator wait: the load latency disappears behind the MMAs and the tiles are free
          // for the next loads as soon as the MMAs have read them.
          uint4 res[2][4];
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            if (p < nrho) {
              const int rho = rho0 + p, a = cls_of(rep_of(rho));
              const int yo = yb + rho;
              const bool rok = xok && yo < PR2;                // outside the plane the tile holds TMA zero fill
              const uint4* rg = reinterpret_cast<const uint4*>(
                  pm_t + int64_t((a * 3 + bcl) * 32) * cstep + (rok ? int64_t(yo) * PC2 + xo : 0) * 8);
#pragma unroll
              for (int k = 0; k < 4; ++k) res[p][k] = rok ? __ldg(rg + int64_t(k) * psz) : make_uint4(0, 0, 0, 0);
            }
          }
          tmem_st_wait();                                      // a value parked by the previous item has landed by now
          if ((warp & 3) == 0 && lane == 0) CMLPL_TR(1 + hf, ntr, uint32_t(kap * 3 + it) * 4);
          mbar_wait(bars + 8 * (DF0 + rho0), kc & 1, 64);
          if (nrho == 2) mbar_wait(bars + 8 * (DF0 + rho0 + 1), kc & 1, 64);
          tc_fence_after();
          if ((warp & 3) == 0 && lane == 0) CMLPL_TR(1 + hf, ntr, uint32_t(kap * 3 + it) * 4 + 1);
          float v[2][32], s[32];
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            if (p < nrho) {
              tmem_ld16(lane_addr + uint32_t((rho0 + p) * 64 + hf * 32), v[p]);
              tmem_ld16(lane_addr + uint32_t((rho0 + p) * 64 + hf * 32 + 16), v[p] + 16);
            }
          }
          // column pairs: kap 0 (kap 3) parks its row-pooled 32 channels in this thread's own scratch columns; the same
          // thread picks them up when kap 1 (kap 4) has drained -- program order, no barrier
          const uint32_t pcol = lane_addr + uint32_t(kPark + it * 64 + hf * 32);
          if (unpark) { tmem_ld16(pcol, s); tmem_ld16(pcol + 16, s + 16); }
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive(bars + 8 * (DE0 + rho0));
          if (nrho == 2) mbar_arrive(bars + 8 * (DE0 + rho0 + 1));
          float acc[32];
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            if (p < nrho) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const __half2* hr = reinterpret_cast<const __half2*>(&res[p][k]);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 f = __half22float2(hr[e]);
                  const float y0 = fmaxf(v[p][k * 8 + 2 * e] + (f.x + bb[k * 8 + 2 * e]), 0.f);
                  const float y1 = fmaxf(v[p][k * 8 + 2 * e + 1] + (f.y + bb[k * 8 + 2 * e + 1]), 0.f);
                  if (p == 0) { acc[k * 8 + 2 * e] = y0; acc[k * 8 + 2 * e + 1] = y1; }
                  else { acc[k * 8 + 2 * e] = (acc[k * 8 + 2 * e] + y0) * 0.5f; acc[k * 8 + 2 * e + 1] = (acc[k * 8 + 2 * e + 1] + y1) * 0.5f; }
                }
              }
            }
          }
          if (park) {
            tmem_st16(pcol, acc);
            tmem_st16(pcol + 16, acc + 16);
          } else {
            if (unpark) {
#pragma unroll
              for (int c = 0; c < 32; ++c) acc[c] = (acc[c] + s[c]) * 0.5f;
            }
            const int y = yb + rho0;                           // the item's frame lives rho0 rows further down
            if (xval && y < PR2) {
              __half* dst = yq_t + int64_t((it * 3 + Be) * 32) * cstep + (int64_t(y) * PC2 + x) * 8;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                __half2 h[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) h[e] = __floats2half2_rn(acc[k * 8 + 2 * e], acc[k * 8 + 2 * e + 1]);
                *reinterpret_cast<uint4*>(dst + int64_t(k) * cstep) = *reinterpret_cast<uint4*>(h);
              }
            }
          }
          if ((warp & 3) == 0 && lane == 0) CMLPL_TR(1 + hf, ntr, uint32_t(kap * 3 + it) * 4 + 2);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// =================================================================================================
// pool2_cls_kernel:  M[I][y',x'][cls] = sum_J L[I][J][y', x'+2J],
//                    L[I][J][y',x'][cls] = sum_{u,v} (Wc[I,J]/4) . Y[rho(2I+u)][kap(2J+v)][y'+u, x'+v]
// A pixel's conv logits are sum_{I,J} L[I][J][r'+2I, c'+2J]; the sum over J is taken here, so that 5 row maps leave the
// kernel instead of 25 cell maps and the head gathers 5 vectors per pixel.  Inputs are the 9 half-pooled maps YP[Al][Be]
// of conv2_scene_kernel (border classes already averaged over their two variants, the middle class per position).  For a
// pooled row class Al and a pooled column J the tile of YP[Al][Be(J)] is loaded with its origin 2J columns to the right
// (the column shift of the J-sum is a TMA coordinate), the remaining 2x2 pool of the middle classes is an A-descriptor
// offset (u,v) inside the tile, and the maps I of the row class share the operand: (Al==1 ? 2 : 1) x (Be==1 ? 2 : 1)
// shifts x 4 k-steps tcgen05.mma with M = 128 positions, N = NC classes x (1 or 3) maps, all J accumulating into the
// same TMEM columns.  The block weights carry 1/4, 1/2 or 1 (pack.cu).  Two accumulator stages: the MMAs of the next
// tile run under the read-out of this one.
// NC = class width: 16 for <= 16 classes; 32 for 17-32, whose 100 KB of weights leave room for 6 ring slots, and whose two
// accumulator stages of 5 maps x 32 columns need 512 TMEM columns.
namespace p2c {
constexpr int TH = 4, TP = 32, TW = 31;              // outputs valid for tx = 0..30 (tx+1 must be in the tile)
constexpr int CH = (TH + 1) * TP * 16;               // 2 560: one chunk plane of a tile, dense (written by TMA)
constexpr int TBYTES = 8 * CH;                       // 20 480: one map tile
constexpr int kEpi = 256, kThreads = kEpi + 64;      // warps 0-7 epilogue, warp 8 loader, warp 9 MMA issuer
constexpr int kLoadWarp = kEpi / 32, kMmaWarp = kLoadWarp + 1;
template <int NC>
struct Plan {
  static constexpr int NSLOT = NC == 16 ? 8 : 6;     // ring of map tiles (164 / 123 KB in flight per SM)
  static constexpr int WBYTES = 25 * NC * 128;       // 25 maps x NC classes x 64 channels, f16
  static constexpr int TCOLS = NC == 16 ? 256 : 512; // TMEM allocation; accumulator stage st at column st * TCOLS / 2
  static constexpr int S_W = 0, S_T = WBYTES, S_BAR = S_T + NSLOT * TBYTES + 128, S_TMEM = S_BAR + 256;   // +128: shifted A rows of the last slot
  static constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
  enum { F0 = 0, E0 = NSLOT, DFULL0 = 2 * NSLOT, DEMPTY0 = 2 * NSLOT + 2, W_FULL = 2 * NSLOT + 4 };
  static_assert(SMEM <= 232448, "pool2_cls: shared memory over the 227 KB limit");
  static_assert(S_T % 128 == 0 && TBYTES % 128 == 0, "pool2_cls: TMA destinations must be 128-byte aligned");
  static_assert(2 * 5 * NC <= TCOLS && 5 * NC <= TCOLS / 2, "pool2_cls: two accumulator stages of 5 maps must fit TMEM");
};
static_assert(Plan<16>::SMEM <= 232448 && Plan<16>::NSLOT == 8, "pool2_cls<16>: 8-slot ring within 227 KB");
static_assert(Plan<32>::SMEM <= 232448 && Plan<32>::NSLOT == 6, "pool2_cls<32>: 6-slot ring within 227 KB");
}  // namespace p2c

// yq f16 [9][4][8][PR2][PC2][8];  wcq f16 per block (Al,Be) [8 kchunks][N rows = ((J-J0)*nI + I-I0)*NC + cls][8];
// lmap f32 [4 planes][5 = I][NC/4 class quads][PR2][PC2][4]
// Every map tile ((TH+1) rows x 32 entries x 8 chunks, 20 KB) is ONE cp.async.bulk.tensor (TMA, 4-D tile mode, zero
// fill outside the plane) into a ring of NSLOT slots, each with its own full / empty mbarrier, so a single loader thread
// runs up to NSLOT tiles ahead of the MMAs; 15 loads per output tile (the three middle columns re-read their map at
// three origins, from L2).
template <int NC>
__global__ void __launch_bounds__(p2c::kThreads, 1)
pool2_cls_kernel(const __grid_constant__ CUtensorMap tm_y, int PR2, int PC2, int nq, int ncell /* pooled cells per side: 5 (w = 20) or 2 (w = 11) */,
                 const unsigned char* __restrict__ wcq, float* __restrict__ lmap) {
  using namespace p2c;
  using P = Plan<NC>;
  constexpr int NSLOT = P::NSLOT, WBYTES = P::WBYTES, TCOLS = P::TCOLS, S_W = P::S_W, S_T = P::S_T, S_BAR = P::S_BAR,
                S_TMEM = P::S_TMEM;
  constexpr int F0 = P::F0, E0 = P::E0, DFULL0 = P::DFULL0, DEMPTY0 = P::DEMPTY0, W_FULL = P::W_FULL;
  constexpr int NQ = NC / 4;                           // class quads per lmap entry
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + S_BAR;
  const int tiles_c = (PC2 + TW - 1) / TW, tiles_r = (PR2 + TH - 1) / TH;
  const int tiles_p = tiles_r * tiles_c, ntiles = 4 * tiles_p;
  const int64_t psz = int64_t(PR2) * PC2;
  // Tiles run in the reverse of conv2_scene_kernel's order (last parity plane, bottom rows first): the maps conv2 wrote
  // last are still in L2 when this kernel starts, and it reads them before they are evicted.
  // w = 11: pooled cells I, J in {0, 1} only -> row classes Al = 0, 1 and pooled columns J = 0, 1 (the weights of every
  // other cell are zero in wcq, their maps are neither loaded nor multiplied)
  const int nAl = ncell >= 5 ? 3 : 2, nJ = ncell >= 5 ? 5 : 2;

  {
    uint4* z = reinterpret_cast<uint4*>(smem + S_T);
    for (int i = tid; i < (NSLOT * TBYTES + 128) / 16; i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (tid == 0) {
    mbar_init(bars + 8 * W_FULL, 1);
    fence_barrier_init();
    bulk_weights_g2s(sbase + S_W, wcq, WBYTES, bars + 8 * W_FULL);
    for (int s = 0; s < NSLOT; ++s) { mbar_init(bars + 8 * (F0 + s), 1); mbar_init(bars + 8 * (E0 + s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(bars + 8 * (DFULL0 + s), 1); mbar_init(bars + 8 * (DEMPTY0 + s), kEpi); }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(sbase + S_TMEM, TCOLS);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);

  if (warp == kLoadWarp) {
    // ================================================================ loader: one TMA per (row class, pooled column)
    if (lane == 0) {
      tma_prefetch_desc(&tm_y);
      uint32_t slot = 0, ph = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int u = ntiles - 1 - t, pl = u / tiles_p, tt = u - pl * tiles_p;   // last plane, bottom rows first (see above)
        const int tr = tt / tiles_c, tc = tt - tr * tiles_c;
#pragma unroll 1
        for (int q = 0; q < 15; ++q) {
          const int Al = q / 5, J = q - Al * 5, Be = J == 0 ? 0 : (J == 4 ? 2 : 1);
          if (Al >= nAl || J >= nJ) continue;
          mbar_wait(bars + 8 * (E0 + slot), ph ^ 1, 71);
          mbar_arrive_expect_tx(bars + 8 * (F0 + slot), TBYTES);
          tma_load_tile(sbase + S_T + slot * TBYTES, &tm_y, tc * TW + 2 * J, tr * TH, (Al * 3 + Be) * 4 + pl, bars + 8 * (F0 + slot));
          if (++slot == NSLOT) { slot = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer
    constexpr uint64_t kHi = (uint64_t(128 >> 4) | (uint64_t(1) << 14)) << 32;
    uint32_t slot = 0, ph = 0, tj = 0;
    mbar_wait(bars + 8 * W_FULL, 0, 70);                       // weights have landed
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++tj) {
      const uint32_t st = tj & 1;
      mbar_wait(bars + 8 * (DEMPTY0 + st), ((tj >> 1) & 1) ^ 1, 72);   // this stage's previous tile has been read out
      tc_fence_after();
#pragma unroll
      for (int Al = 0; Al < 3; ++Al) {
        const int nI = blk_n(Al), N = nI * NC, nu = Al == 1 ? 2 : 1;
        const uint32_t idesc = make_idesc_f16(128, N);
        const uint32_t dcol = tmem + st * (TCOLS / 2) + uint32_t(blk_first(Al) * NC);
        if (Al >= nAl) continue;
#pragma unroll
        for (int J = 0; J < 5; ++J) {
          if (J >= nJ) continue;
          const int Be = J == 0 ? 0 : (J == 4 ? 2 : 1), nv = Be == 1 ? 2 : 1;
          const int Nb = nI * blk_n(Be) * NC;                  // rows of the block (Al, Be): its k-chunk stride
          const uint32_t w_lo = ((sbase + S_W + blk_start(Al * 3 + Be) * NC * 128 + (J - blk_first(Be)) * N * 16) >> 4) |
                                (uint32_t((Nb * 16) >> 4) << 16);
          mbar_wait(bars + 8 * (F0 + slot), ph, 73);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t t_lo = ((sbase + S_T + slot * TBYTES) >> 4) | (uint32_t(CH >> 4) << 16);
#pragma unroll
            for (int u = 0; u < nu; ++u) {
#pragma unroll
              for (int v = 0; v < nv; ++v) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                  const uint32_t a = t_lo + uint32_t(((u * TP + v) * 16 + ks * 2 * CH) / 16);
                  const uint32_t bw = w_lo + uint32_t((ks * 2 * Nb * 16) / 16);
                  umma_f16(dcol, kHi | uint64_t(a), kHi | uint64_t(bw), idesc, (J | u | v | ks) ? 1u : 0u);
                }
              }
            }
            umma_commit(bars + 8 * (E0 + slot));
            if (Al == nAl - 1 && J == nJ - 1) umma_commit(bars + 8 * (DFULL0 + st));
          }
          __syncwarp();
          if (++slot == NSLOT) { slot = 0; ph ^= 1; }
        }
      }
    }
  } else {
    // ================================================================ epilogue (warps 0-7): warps 0-3 read out I = 0..2, warps 4-7 I = 3, 4
    const int L = (warp & 3) * 32 + lane, half = warp >> 2;
    const uint32_t lane_addr = tmem + (uint32_t((warp & 3) * 32) << 16);
    const int ty = L >> 5, tx = L & 31;
    const int m0 = half ? 3 : 0, m1 = half ? 5 : 3;
    uint32_t tj = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++tj) {
      const int u = ntiles - 1 - t, pl = u / tiles_p, tt = u - pl * tiles_p;   // last plane, bottom rows first (see above)
      const int tr = tt / tiles_c, tc = tt - tr * tiles_c;
      const int y = tr * TH + ty, x = tc * TW + tx;
      const bool valid = tx < TW && y < PR2 && x < PC2;
      const uint32_t st = tj & 1;
      // lmap f32 [4 planes][5 maps][NC/4 class quads][PR2][PC2][4]: a warp's store of one (map, quad) is 512 contiguous bytes
      float4* dst = reinterpret_cast<float4*>(lmap) + int64_t(pl) * 5 * NQ * psz + (valid ? int64_t(y) * PC2 + x : 0);
      mbar_wait(bars + 8 * (DFULL0 + st), (tj >> 1) & 1, 74);
      tc_fence_after();
      float v[3][NC];
#pragma unroll
      for (int m = 0; m < 3; ++m) {
        if (m0 + m < m1) {
#pragma unroll
          for (int h = 0; h < NC / 16; ++h)
            tmem_ld16(lane_addr + st * (TCOLS / 2) + uint32_t((m0 + m) * NC + h * 16), v[m] + h * 16);
        }
      }
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bars + 8 * (DEMPTY0 + st));
      if (valid) {
#pragma unroll
        for (int m = 0; m < 3; ++m) {
          if (m0 + m < m1 && m0 + m < ncell) {
#pragma unroll
            for (int q = 0; q < NQ; ++q)                        // class quads beyond the real classes are never read (head_sum_kernel)
              if (q < nq) dst[int64_t((m0 + m) * NQ + q) * psz] = make_float4(v[m][4 * q], v[m][4 * q + 1], v[m][4 * q + 2], v[m][4 * q + 3]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) { tc_fence_after(); tmem_dealloc(tmem, TCOLS); }
}

}  // namespace cmlpl

using namespace cmlpl;

CMLPL_TRACE_EXPORT(cmlpl_debug_c2s_trace)

extern "C" int cmlpl_conv2_scene_f16(const void* pmq, int cols, int w, int band_rows, const void* packed, void* yq,
                                     cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(pmq && packed && yq, "conv2_scene: null pointer");
  CMLPL_CHECK_ARG((w == 20 || w == 11) && cols > 0 && band_rows > 0, "conv2_scene: bad dims (w must be 20 or 11)");
  const int PR2 = (band_rows + w) / 2, PC2 = (cols + w) / 2;
  const PackedLayout L = packed_layout(1, 1, w);
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const int ntiles = 4 * ((PR2 + c2s::TH - 1) / c2s::TH) * ((PC2 + c2s::TW - 1) / c2s::TW);
  int grid = sm_count(); if (grid > ntiles) grid = ntiles;
  CUtensorMap tm_pm;
  const int trc = make_scene_tmap(&tm_pm, pmq, 36, PR2, PC2, c2s::TH + 2, c2s::TP);
  if (trc != CMLPL_OK) return trc;
  if (w == 11) {
    CMLPL_MAX_DYN_SMEM(conv2_scene_kernel<true>, c2s::SMEM);
    conv2_scene_kernel<true><<<grid, c2s::kThreads, c2s::SMEM, static_cast<cudaStream_t>(stream)>>>(
        tm_pm, static_cast<const __half*>(pmq), PR2, PC2, pk + L.w2, reinterpret_cast<const float*>(pk + L.b2),
        static_cast<__half*>(yq));
  } else {
    CMLPL_MAX_DYN_SMEM(conv2_scene_kernel<false>, c2s::SMEM);
    conv2_scene_kernel<false><<<grid, c2s::kThreads, c2s::SMEM, static_cast<cudaStream_t>(stream)>>>(
        tm_pm, static_cast<const __half*>(pmq), PR2, PC2, pk + L.w2, reinterpret_cast<const float*>(pk + L.b2),
        static_cast<__half*>(yq));
  }
  CMLPL_CHECK_LAUNCH("conv2_scene");
  return CMLPL_OK;
}

extern "C" int cmlpl_pool2_cls_f16(const void* yq, int cols, int w, int band_rows, int num_features, int num_classes,
                                   const void* packed, float* lmap, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(yq && packed && lmap, "pool2_cls: null pointer");
  CMLPL_CHECK_ARG((w == 20 || w == 11) && cols > 0 && band_rows > 0 && num_classes > 0 && num_classes <= 32,
                  "pool2_cls: bad dims (w must be 20 or 11, <= 32 classes)");
  const int PR2 = (band_rows + w) / 2, PC2 = (cols + w) / 2;
  const PackedLayout L = packed_layout(num_features, num_classes, w);
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const int ntiles = 4 * ((PR2 + p2c::TH - 1) / p2c::TH) * ((PC2 + p2c::TW - 1) / p2c::TW);
  int grid = sm_count(); if (grid > ntiles) grid = ntiles;
  CUtensorMap tm_y;
  const int trc = make_scene_tmap(&tm_y, yq, 36, PR2, PC2, p2c::TH + 1, p2c::TP);
  if (trc != CMLPL_OK) return trc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int nq = (num_classes + 3) / 4, ncell = w == 20 ? 5 : 2;
  if (L.nc == 16) {
    CMLPL_MAX_DYN_SMEM(pool2_cls_kernel<16>, p2c::Plan<16>::SMEM);
    pool2_cls_kernel<16><<<grid, p2c::kThreads, p2c::Plan<16>::SMEM, s>>>(tm_y, PR2, PC2, nq, ncell, pk + L.wcq, lmap);
  } else {
    CMLPL_MAX_DYN_SMEM(pool2_cls_kernel<32>, p2c::Plan<32>::SMEM);
    pool2_cls_kernel<32><<<grid, p2c::kThreads, p2c::Plan<32>::SMEM, s>>>(tm_y, PR2, PC2, nq, ncell, pk + L.wcq, lmap);
  }
  CMLPL_CHECK_LAUNCH("pool2_cls");
  return CMLPL_OK;
}
