// Similarity GEMMs of the losses on tcgen05:  S = A . B^T  with A [M, K], B [N, K] fp32 row-major (K contiguous), K = 1024-d
// unit-norm features (train.py:213,217,246,257; tools/models.py:27).  Operands are rounded to fp16 on the way into
// shared memory (the loaders write the UMMA no-swizzle K-major tiles directly), fp32 accumulation in TMEM.
//
// Two epilogues:
//   STORE  the 128 x 128 tile is written to C (pseudo-label graph logits G; the standalone loss entry points)
//   BANK   flash-style streaming memory-bank smoothing (train.py:213-215): the tile never leaves the SM -- every row
//          accumulates  sum_j exp(S_rj / T)  and  sum_j exp(S_rj / T) * queue_probs[j, c]  over the tile's 128 bank rows
//          and writes C+1 partial sums; loss_rows_kernel adds the partials of the bank tiles.  |S| <= 1 for unit-norm
//          features, so the plain exponential needs no running maximum.  The [rows, queue] logits are never materialised.
// grid (tiles, problems); 9 warps: 0-7 load + convert during the K loop and run the epilogue, 8 issues the MMAs.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "train_common.cuh"
#include "train_head.cuh"

namespace cmlpl {

namespace sim {
constexpr int KB = 64;                                  // K per stage
constexpr int OPB = 128 * KB * 2;                       // one operand tile of a stage: 16 384 B
constexpr int STAGES = 2;
constexpr int S_A = 0, S_B = STAGES * OPB, S_QP = 2 * STAGES * OPB, S_BAR = S_QP + 128 * 32 * 4, S_TMEM = S_BAR + 64;
constexpr int SMEM = (S_TMEM + 16 + 127) / 128 * 128;
constexpr int kWorkers = 256, kThreads = kWorkers + 32;
enum { FULL0 = 0, EMPTY0 = 2, DONE = 4 };
}  // namespace sim

__global__ void __launch_bounds__(sim::kThreads)
sim_tc_kernel(SimBatch sb) {
  using namespace sim;
  const SimProb& p = sb.p[blockIdx.y];
  if (p.enable && *p.enable == 0) return;
  const int tiles_n = (p.N + 127) / 128, tiles_m = (p.M + 127) / 128;
  if (int(blockIdx.x) >= tiles_n * tiles_m) return;
  const int m0 = (blockIdx.x / tiles_n) * 128, n0 = (blockIdx.x % tiles_n) * 128;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + S_BAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + S_TMEM);
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bars + 8 * (FULL0 + s), kWorkers); mbar_init(bars + 8 * (EMPTY0 + s), 1); }
    mbar_init(bars + 8 * DONE, 1);
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(sbase + S_TMEM, 128);
  if (p.mode == 1) {   // queue_probs rows of this bank tile, zero beyond N and in the class slots C..31 the epilogue reads
    float* qs = reinterpret_cast<float*>(smem + S_QP);
    for (int i = tid; i < 128 * 32; i += kThreads) {
      const int j = i >> 5, c = i & 31;
      qs[i] = (c < p.C && n0 + j < p.N) ? __ldg(p.qp + int64_t(n0 + j) * p.C + c) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int nkb = p.K / KB;

  if (warp == 8) {
    constexpr uint32_t kI = make_idesc_f16(128, 128);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % STAGES;
      mbar_wait(bars + 8 * (FULL0 + s), (kb / STAGES) & 1, 70);
      tc_fence_after();
      if (lane == 0) {
#pragma unroll
        for (int ks = 0; ks < KB / 16; ++ks)
          umma_f16(tmem, make_desc(sbase + S_A + s * OPB + ks * 2 * 2048, 2048, 128),
                   make_desc(sbase + S_B + s * OPB + ks * 2 * 2048, 2048, 128), kI, (kb | ks) != 0 ? 1u : 0u);
        umma_commit(bars + 8 * (EMPTY0 + s));
        if (kb == nkb - 1) umma_commit(bars + 8 * DONE);
      }
      __syncwarp();
    }
  } else {
    // ---- loaders: thread = (row, half of the 64-wide K block): 8 float4 -> four 16-byte chunks of 8 halves
    const int row = tid >> 1, kh = tid & 1;
    const bool a_ok = m0 + row < p.M, b_ok = n0 + row < p.N;
    const float* ga = p.A + int64_t(m0 + row) * p.lda + kh * 32;
    const float* gb = p.B + int64_t(n0 + row) * p.ldb + kh * 32;
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % STAGES;
      mbar_wait(bars + 8 * (EMPTY0 + s), ((kb / STAGES) & 1) ^ 1, 71);
      float4 va[8], vb[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        va[q] = a_ok ? __ldg(reinterpret_cast<const float4*>(ga + kb * KB) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        vb[q] = b_ok ? __ldg(reinterpret_cast<const float4*>(gb + kb * KB) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        __half2 h[4];
        h[0] = __floats2half2_rn(va[2 * c].x, va[2 * c].y); h[1] = __floats2half2_rn(va[2 * c].z, va[2 * c].w);
        h[2] = __floats2half2_rn(va[2 * c + 1].x, va[2 * c + 1].y); h[3] = __floats2half2_rn(va[2 * c + 1].z, va[2 * c + 1].w);
        *reinterpret_cast<uint4*>(smem + S_A + s * OPB + (kh * 4 + c) * 2048 + row * 16) = *reinterpret_cast<uint4*>(h);
        h[0] = __floats2half2_rn(vb[2 * c].x, vb[2 * c].y); h[1] = __floats2half2_rn(vb[2 * c].z, vb[2 * c].w);
        h[2] = __floats2half2_rn(vb[2 * c + 1].x, vb[2 * c + 1].y); h[3] = __floats2half2_rn(vb[2 * c + 1].z, vb[2 * c + 1].w);
        *reinterpret_cast<uint4*>(smem + S_B + s * OPB + (kh * 4 + c) * 2048 + row * 16) = *reinterpret_cast<uint4*>(h);
      }
      fence_proxy_async();
      mbar_arrive(bars + 8 * (FULL0 + s));
    }
    // ---- epilogue: warp w reads TMEM lanes (w&3)*32.. (tile rows) and the 64 columns of half w>>2
    mbar_wait(bars + 8 * DONE, 0, 72);
    tc_fence_after();
    const int q4 = warp & 3, chalf = warp >> 2;
    const int r = m0 + q4 * 32 + lane;
    const uint32_t taddr = tmem + (uint32_t(q4 * 32) << 16) + chalf * 64;
    if (p.mode == 0) {
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + c0, v);
        tmem_ld_wait();
        if (r < p.M) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int n = n0 + chalf * 64 + c0 + j;
            if (n < p.N) p.Cout[int64_t(r) * p.ldc + n] = v[j];
          }
        }
      }
    } else {
      const float invT = 1.f / sb.prm->temperature;
      const float* qs = reinterpret_cast<const float*>(smem + S_QP) + (chalf * 64) * 32;
      float asum = 0.f, acc[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) acc[c] = 0.f;
      float acc2[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) acc2[c] = 0.f;
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const bool in = n0 + chalf * 64 + c0 + j < p.N;
          const float w = in ? __expf(v[j] * invT) : 0.f;
          asum += w;
          const float4* q = reinterpret_cast<const float4*>(qs + (c0 + j) * 32);
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 t = q[c4];
            acc[4 * c4] = fmaf(w, t.x, acc[4 * c4]); acc[4 * c4 + 1] = fmaf(w, t.y, acc[4 * c4 + 1]);
            acc[4 * c4 + 2] = fmaf(w, t.z, acc[4 * c4 + 2]); acc[4 * c4 + 3] = fmaf(w, t.w, acc[4 * c4 + 3]);
          }
          if (p.C > 16) {
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) {
              const float4 t = q[4 + c4];
              acc2[4 * c4] = fmaf(w, t.x, acc2[4 * c4]); acc2[4 * c4 + 1] = fmaf(w, t.y, acc2[4 * c4 + 1]);
              acc2[4 * c4 + 2] = fmaf(w, t.z, acc2[4 * c4 + 2]); acc2[4 * c4 + 3] = fmaf(w, t.w, acc2[4 * c4 + 3]);
            }
          }
        }
      }
      if (r < p.M) {
        // part [2 * tiles_n][M][33]: 32 class sums + the exp sum, one entry per (bank tile, column half)
        float* o = p.part + ((int64_t((blockIdx.x % tiles_n) * 2 + chalf) * p.M) + r) * 33;
#pragma unroll
        for (int c = 0; c < 16; ++c) o[c] = acc[c];
        if (p.C > 16) {
#pragma unroll
          for (int c = 0; c < 16; ++c) o[16 + c] = acc2[c];
        }
        o[32] = asum;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) { tc_fence_after(); tmem_dealloc(tmem, 128); }
}

int launch_sim_tc(const SimBatch& sb, cudaStream_t st, const char* name) {
  int tiles = 0;
  for (int i = 0; i < sb.count; ++i) {
    const SimProb& p = sb.p[i];
    CMLPL_CHECK_ARG(p.K > 0 && p.K % sim::KB == 0 && p.lda % 4 == 0 && p.ldb % 4 == 0 &&
                        reinterpret_cast<uintptr_t>(p.A) % 16 == 0 && reinterpret_cast<uintptr_t>(p.B) % 16 == 0,
                    "%s: K must be a multiple of 64 and the operands 16-byte aligned rows", name);
    CMLPL_CHECK_ARG(p.mode == 0 || (p.C > 0 && p.C <= 32 && p.qp && p.part), "%s: bad bank epilogue arguments", name);
    const int t = ((p.N + 127) / 128) * ((p.M + 127) / 128);
    if (t > tiles) tiles = t;
  }
  if (tiles == 0) return CMLPL_OK;
  CMLPL_MAX_DYN_SMEM(sim_tc_kernel, sim::SMEM);
  sim_tc_kernel<<<dim3(tiles, sb.count), sim::kThreads, sim::SMEM, st>>>(sb);
  CMLPL_CHECK_LAUNCH(name);
  return CMLPL_OK;
}

}  // namespace cmlpl

// C = A . B^T on tcgen05 (fp16 operands, fp32 accumulate): the similarity matrices of the loss entry points in their
// tensor-core mode (cmlpl_set_loss_gemm_mode).
extern "C" int cmlpl_sim_nt_tc_f32(const float* A, const float* B, int M, int N, int K, float* C, cmlpl_stream_t stream) {
  using namespace cmlpl;
  CMLPL_CHECK_ARG(A && B && C && M > 0 && N > 0, "sim_nt_tc: bad args");
  SimBatch sb{};
  sb.count = 1;
  sb.p[0] = SimProb{A, B, K, K, M, N, K, 0, C, N, nullptr, nullptr, 0, nullptr};
  return launch_sim_tc(sb, static_cast<cudaStream_t>(stream), "sim_nt_tc");
}
