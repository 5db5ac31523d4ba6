// Fused training step: everything around the conv trunk, for BOTH BaseNet2 peers per launch (train.py:150-272).
//   multi_gemm_kernel   fp32 tiled GEMMs, several independent problems in one grid (spectral branch forward, the
//                       memory-bank / graph similarity matrices, the feature gradients, feat_spe's weight gradient)
//   head_fwd_kernel     dropout mask (injected or Philox) + classifier + L2-normalised spectral feature
//                       (tools/models.py:144-150, 87-90)
//   loss_rows_kernel    supervised CE on the labelled rows (train.py:191-194) and the memory-bank pseudo-label
//                       smoothing + adaptive threshold on the unlabelled rows (train.py:203-228)
//   loss_graph_kernel   pseudo-label-graph contrastive loss (train.py:243-265), masked soft CE cross supervision
//                       (train.py:239-242), and the memory-bank writes (train.py:223-235)
//   head_bwd_kernel     dL/dcat (dropout mask applied), ReLU / L2-norm backward of the spectral feature, max|dL/dcat|
//   head_wgrad_kernel   classifier weight / bias gradients and feat_spe's bias gradient (column reductions)
//   adam_all_kernel     torch.optim.Adam (train.py:131-132,268,272) over the 20 live tensors of both nets
// All fp32 (warp-per-row kernels with shuffle reductions): these are latency-bound at 128 + 128 rows.
#include "common.cuh"
#include "train_common.cuh"
#include "train_head.cuh"

namespace cmlpl {

// ============================================================================ multi-problem fp32 GEMM
// C[m][n] = act(alpha * sum_k A(m,k) B(k,n) + bias[n]);  64x64x16 tiles, 256 threads, 4x4 micro-tiles (packed FFMA2).
__global__ void __launch_bounds__(256)
multi_gemm_kernel(MultiGemm mg) {
  const GemmProb& p = mg.p[blockIdx.y];
  if (p.enable && *p.enable == 0) return;
  const int tiles_n = (p.N + 63) / 64, tiles_m = (p.M + 63) / 64;
  if (int(blockIdx.x) >= tiles_n * tiles_m) return;
  const int m0 = (blockIdx.x / tiles_n) * 64, n0 = (blockIdx.x % tiles_n) * 64;
  __shared__ float As[2][16][68];
  __shared__ float Bs[2][16][68];
  const int tid = threadIdx.x;
  // loader mapping per operand: the fastest thread index runs along the unit-stride dimension
  const bool a_kfast = p.a_cs == 1, b_kfast = p.b_rs == 1;
  int a_row[4], a_k[4], b_row[4], b_k[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    a_row[j] = a_kfast ? (tid >> 4) + 16 * j : (tid & 63);
    a_k[j] = a_kfast ? (tid & 15) : (tid >> 6) + 4 * j;
    b_row[j] = b_kfast ? (tid >> 4) + 16 * j : (tid & 63);
    b_k[j] = b_kfast ? (tid & 15) : (tid >> 6) + 4 * j;
  }
  const int tx = tid & 15, ty = tid >> 4;
  unsigned long long acc2[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc2[i][0] = acc2[i][1] = 0ull;
  float ra[4], rb[4];
  auto gload = [&](int k0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int am = m0 + a_row[j], ak = k0 + a_k[j], bn = n0 + b_row[j], bk = k0 + b_k[j];
      ra[j] = (am < p.M && ak < p.K) ? __ldg(p.A + am * p.a_rs + ak * p.a_cs) : 0.f;
      rb[j] = (bn < p.N && bk < p.K) ? __ldg(p.B + bk * p.b_rs + bn * p.b_cs) : 0.f;
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int j = 0; j < 4; ++j) { As[buf][a_k[j]][a_row[j]] = ra[j]; Bs[buf][b_k[j]][b_row[j]] = rb[j]; }
  };
  gload(0);
  sstore(0);
  __syncthreads();
  int buf = 0;
  for (int k0 = 0; k0 < p.K; k0 += 16) {
    const bool more = k0 + 16 < p.K;
    if (more) gload(k0 + 16);
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      const ulonglong2 b = *reinterpret_cast<const ulonglong2*>(&Bs[buf][k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        unsigned long long aa;
        asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(av[i]));
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][0]) : "l"(aa), "l"(b.x));
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][1]) : "l"(aa), "l"(b.y));
      }
    }
    if (more) { sstore(buf ^ 1); __syncthreads(); buf ^= 1; }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
    float v[4];
    asm("mov.b64 {%0, %1}, %2;" : "=f"(v[0]), "=f"(v[1]) : "l"(acc2[i][0]));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(v[2]), "=f"(v[3]) : "l"(acc2[i][1]));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= p.N) continue;
      float o = v[j] * p.alpha;
      if (p.bias) o += __ldg(p.bias + n);
      if (p.act == 1) o = fmaxf(o, 0.f);
      p.C[m * p.c_rs + n * p.c_cs] = o;
    }
  }
}

int launch_multi_gemm(const MultiGemm& mg, cudaStream_t st, const char* name) {
  int tiles = 0;
  for (int i = 0; i < mg.count; ++i) {
    const int t = ((mg.p[i].N + 63) / 64) * ((mg.p[i].M + 63) / 64);
    if (t > tiles) tiles = t;
  }
  if (tiles == 0) return CMLPL_OK;
  multi_gemm_kernel<<<dim3(tiles, mg.count), 256, 0, st>>>(mg);
  CMLPL_CHECK_LAUNCH(name);
  return CMLPL_OK;
}

// ============================================================================ classifier forward
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// block-wide sum of NV per-thread values (128 threads = 4 warps); the result is valid in every thread
template <int NV>
__device__ __forceinline__ void block_sum4(float (&v)[NV], float* red /* [4][NV] */) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  __syncthreads();                                   // red may still be read from a previous call
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) red[warp * NV + i] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = (red[i] + red[NV + i]) + (red[2 * NV + i] + red[3 * NV + i]);
}

// one CTA (4 warps) per row: 656 float4 groups of the 2624 features (320 of 1280 at W = 11) over 128 threads
template <int CMAX, int W>
__global__ void __launch_bounds__(128)
head_fwd_kernel(HeadArgs a) {
  constexpr int CAT = TrainGeom<W>::CatDim, CONV = TrainGeom<W>::ConvFeat;
  __shared__ float red[4 * (CMAX + 1)];
  const int s = blockIdx.x;
  const int tid = threadIdx.x;
  const int e = s / a.nb;
  const float* cat = a.cat + int64_t(s) * CAT;
  float* dm = a.dmask + int64_t(s) * CAT;
  const float* wc = a.wc[e];
  const float p = a.prm->dropout_p;
  const float keep_scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  const unsigned long long seed = a.prm->seed, offset = a.prm->offset;
  float acc[CMAX + 1];                                 // [CMAX] = sum of squares of the spectral features
#pragma unroll
  for (int c = 0; c <= CMAX; ++c) acc[c] = 0.f;
  for (int g = tid; g < CAT / 4; g += 128) {
    const float4 x = ld4(cat + 4 * g);
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
    if (a.drop_mask) {
      m = ld4(a.drop_mask + int64_t(s) * CAT + 4 * g);
    } else if (p > 0.f && a.training) {
      const uint4 u = philox_uniform4(seed, offset, PHILOX_DROP, uint32_t(s) * (CAT / 4) + uint32_t(g));
      const uint32_t thr = uint32_t(fminf(p, 1.f) * 4294967295.0f);
      m.x = u.x >= thr ? keep_scale : 0.f; m.y = u.y >= thr ? keep_scale : 0.f;
      m.z = u.z >= thr ? keep_scale : 0.f; m.w = u.w >= thr ? keep_scale : 0.f;
    }
    *reinterpret_cast<float4*>(dm + 4 * g) = m;
    const float4 xd = make_float4(x.x * m.x, x.y * m.y, x.z * m.z, x.w * m.w);
    if (4 * g >= CONV) acc[CMAX] += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < a.C) {
        const float4 w = ld4(wc + int64_t(c) * CAT + 4 * g);
        acc[c] += xd.x * w.x + xd.y * w.y + xd.z * w.z + xd.w * w.w;
      }
    }
  }
  block_sum4<CMAX + 1>(acc, red);
  const float nr = sqrtf(acc[CMAX]);                           // models.py:88: no epsilon
  if (tid == 0) a.norm[s] = nr;
  if (tid < a.C) {
    float v = 0.f;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) v = tid == c ? acc[c] : v;
    a.logits[int64_t(s) * a.C + tid] = v + a.bc[e][tid];
  }
  float* f = a.feat + int64_t(s) * kHid;
  for (int j = tid; j < kHid; j += 128) f[j] = cat[CONV + j] / nr;
}

int launch_head_fwd(const HeadArgs& a, int w, cudaStream_t st) {
  const int grid = 2 * a.nb;
  if (w == 11) {
    if (a.C <= 16) head_fwd_kernel<16, 11><<<grid, 128, 0, st>>>(a);
    else head_fwd_kernel<32, 11><<<grid, 128, 0, st>>>(a);
  } else {
    if (a.C <= 16) head_fwd_kernel<16, 20><<<grid, 128, 0, st>>>(a);
    else head_fwd_kernel<32, 20><<<grid, 128, 0, st>>>(a);
  }
  CMLPL_CHECK_LAUNCH("train_head_fwd");
  return CMLPL_OK;
}

// ============================================================================ losses
enum { H_LC = 0, H_TOTAL, H_CLS, H_CON, H_ACC, H_TOTAL1, H_CLS1, H_CON1, H_LC1 };

template <int CMAX>
__global__ void __launch_bounds__(256)
loss_rows_kernel(LossArgs a) {
  const int wi = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int C = a.C, nb = a.bs + a.btu;
  if (wi >= 2 * a.btu + 2 * a.bs) return;
  if (wi < 2 * a.btu) {
    // ---- unlabelled row r of target t: the peer's (net 1-t) prediction, smoothed with bank t (train.py:203-222)
    const int t = wi / a.btu, r = wi - t * a.btu, src = 1 - t;
    const float* zr = a.logits + (int64_t(src) * nb + a.bs + r) * C;
    float mx = -INFINITY;
    for (int c = 0; c < C; ++c) mx = fmaxf(mx, zr[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(zr[c] - mx);
    float p[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) p[c] = c < C ? expf(zr[c] - mx) / se : 0.f;
    float* po = a.probs_orig + (int64_t(t) * a.btu + r) * C;
    if (lane == 0)
      for (int c = 0; c < C; ++c) po[c] = p[c];
    if (a.prm->smooth) {
      // A = exp(f.Qf^T / T) row-normalised, probs = alpha*probs + (1-alpha) * A.Qp (train.py:213-215): the exp sums
      // were streamed out of the similarity tiles by sim_tc_kernel (one partial per bank tile and column half)
      const float alpha = a.prm->alpha;
      const int nparts = 2 * ((a.queue + 127) / 128);
      const float* part = a.S + (int64_t(t) * nparts * a.btu + r) * 33;
      float asum = 0.f, acc = 0.f;                           // lane c < C accumulates class c
      for (int q = 0; q < nparts; ++q) {
        const float* pq = part + int64_t(q) * a.btu * 33;
        asum += pq[32];
        if (lane < C) acc += pq[lane];
      }
      const float sm = acc / asum;
#pragma unroll
      for (int c = 0; c < CMAX; ++c)
        if (c < C) p[c] = alpha * p[c] + (1.f - alpha) * __shfl_sync(0xffffffffu, sm, c);
    }
    if (lane == 0) {
      float best = -INFINITY;
      float* pr = a.probs + (int64_t(t) * a.btu + r) * C;
      for (int c = 0; c < C; ++c) { pr[c] = p[c]; best = fmaxf(best, p[c]); }
      a.mask[t * a.btu + r] = best >= a.prm->adap_thr ? 1.f : 0.f;
    }
  } else {
    // ---- labelled row r of net e: supervised CE (train.py:191-192), accuracy of net 1 (train.py:194,278)
    const int q = wi - 2 * a.btu, e = q / a.bs, r = q - e * a.bs;
    const float* zr = a.logits + (int64_t(e) * nb + r) * C;
    float* dz = a.dlogits + (int64_t(e) * nb + r) * C;
    float mx = -INFINITY; int arg = 0;
    for (int c = 0; c < C; ++c)
      if (zr[c] > mx) { mx = zr[c]; arg = c; }               // first index on ties, like torch.max
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(zr[c] - mx);
    const float lse = mx + logf(se);
    const int y = int(a.labels[r]);
    const float g = 1.f / float(a.bs);
    if (lane < C) dz[lane] = g * (expf(zr[lane] - lse) - (lane == y ? 1.f : 0.f));
    if (C > 32 && lane == 0)
      for (int c = 32; c < C; ++c) dz[c] = g * (expf(zr[c] - lse) - (c == y ? 1.f : 0.f));
    if (lane == 0) {
      const float li = -(zr[y] - lse) * g;
      atomicAdd(a.hist + (e ? H_CLS1 : H_CLS), li);
      atomicAdd(a.hist + (e ? H_TOTAL1 : H_TOTAL), li);
      if (e == 1 && arg == y) atomicAdd(a.hist + H_ACC, g);
    }
  }
}

template <int CMAX>
__global__ void __launch_bounds__(256)
loss_graph_kernel(LossArgs a) {
  const int wi = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int C = a.C, n = a.btu, nb = a.bs + a.btu;
  if (wi >= a.btu + a.bs) return;
  if (wi >= a.btu) {
    // ---- memory-bank rows of the labelled samples: [feats_x ; onehot(Y)]  (train.py:223-235)
    const int r = wi - a.btu;
    const int y = int(a.labels[r]);
    for (int t = 0; t < 2; ++t) {
      const int row = a.prm->queue_ptr[t] + a.btu + r;
      if (row >= a.queue) continue;
      const float4* src = reinterpret_cast<const float4*>(a.feat + (int64_t(t) * nb + r) * kHid);
      float4* dst = reinterpret_cast<float4*>(a.queue_feats[t] + int64_t(row) * kHid);
      for (int j = lane; j < kHid / 4; j += 32) dst[j] = src[j];
      if (lane < C) a.queue_probs[t][int64_t(row) * C + lane] = lane == y ? 1.f : 0.f;
    }
    return;
  }
  const int i = wi;
  const float invT = 1.f / a.prm->temperature;
  // ---- pseudo-label graph contrastive loss, row i (train.py:246-265).  Q0 = probs1 . probs^T with the diagonal
  //      forced to 1 is formed on the fly (C <= 32 products per entry) instead of being stored.
  const float* g = a.G + int64_t(i) * n;
  float p1[CMAX];
#pragma unroll
  for (int c = 0; c < CMAX; ++c) p1[c] = c < C ? a.probs[(int64_t(n) + i) * C + c] : 0.f;
  auto q0_of = [&](int j) {
    if (j == i) return 1.f;
    const float* pj = a.probs + int64_t(j) * C;
    float q = 0.f;
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
      if (c < C) q = fmaf(p1[c], pj[c], q);
    return q;
  };
  float z = 0.f, qs = 0.f, qns = 0.f;
  for (int j = lane; j < n; j += 32) {
    z += expf(g[j] * invT);
    const float q0 = q0_of(j);
    if (q0 >= 0.8f) qs += q0;
    if (q0 <= 0.3f) qns += 1.f - q0;
  }
  z = warp_sum(z); qs = warp_sum(qs); qns = warp_sum(qns);
  const float inv_qs = 1.f / qs, inv_qns = 1.f / (qns + 1e-8f);
  float li = 0.f, w = 0.f;
  for (int j = lane; j < n; j += 32) {
    const float sp = expf(g[j] * invT) / z;
    const float q0 = q0_of(j);
    const float aa = q0 >= 0.8f ? q0 * inv_qs : 0.f;
    const float bb = q0 <= 0.3f ? (1.f - q0) * inv_qns : 0.f;
    li += -logf(sp) * aa + logf(sp + 1.f) * bb;
    w += -aa + bb * sp / (sp + 1.f);
  }
  li = warp_sum(li); w = warp_sum(w);
  {
    const float cf = 0.5f * invT / float(n);                 // 0.5 = weight of loss_contrast in total_loss (train.py:266)
    float* dg = a.dG + int64_t(i) * n;
    for (int j = lane; j < n; j += 32) {
      const float sp = expf(g[j] * invT) / z;
      const float q0 = q0_of(j);
      const float aa = q0 >= 0.8f ? q0 * inv_qs : 0.f;
      const float bb = q0 <= 0.3f ? (1.f - q0) * inv_qns : 0.f;
      dg[j] = cf * ((-aa + bb * sp / (sp + 1.f)) - sp * w);
    }
  }
  if (lane == 0) {
    const float L = li / float(n);
    atomicAdd(a.hist + H_LC, L); atomicAdd(a.hist + H_LC1, L);
    atomicAdd(a.hist + H_TOTAL, 0.5f * L); atomicAdd(a.hist + H_TOTAL1, 0.5f * L);
  }
  // ---- masked soft CE against the peer's smoothed pseudo-labels (train.py:239-242), weight 4 in total_loss
  for (int e = 0; e < 2; ++e) {
    const float* zr = a.logits + (int64_t(e) * nb + a.bs + i) * C;
    const float* pr = a.probs + (int64_t(e) * n + i) * C;
    float* dz = a.dlogits + (int64_t(e) * nb + a.bs + i) * C;
    const float m = a.mask[e * n + i];
    float mx = -INFINITY;
    for (int c = 0; c < C; ++c) mx = fmaxf(mx, zr[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(zr[c] - mx);
    const float lse = mx + logf(se);
    float tsum = 0.f, dot = 0.f;
    for (int c = 0; c < C; ++c) { tsum += pr[c]; dot += (zr[c] - lse) * pr[c]; }
    const float gsc = 4.f / float(n);
    for (int c = lane; c < C; c += 32) dz[c] = gsc * m * (expf(zr[c] - lse) * tsum - pr[c]);
    if (lane == 0) {
      const float l = -dot * m / float(n);
      atomicAdd(a.hist + (e ? H_CON1 : H_CON), l);
      atomicAdd(a.hist + (e ? H_TOTAL1 : H_TOTAL), 4.f * l);
    }
  }
  // ---- memory-bank rows of the unlabelled samples: [peer feature ; peer's unsmoothed probs] (train.py:223-235)
  for (int t = 0; t < 2; ++t) {
    const int row = a.prm->queue_ptr[t] + i;
    if (row >= a.queue) continue;
    const float4* src = reinterpret_cast<const float4*>(a.feat + (int64_t(1 - t) * nb + a.bs + i) * kHid);
    float4* dst = reinterpret_cast<float4*>(a.queue_feats[t] + int64_t(row) * kHid);
    for (int j = lane; j < kHid / 4; j += 32) dst[j] = src[j];
    if (lane < C) a.queue_probs[t][int64_t(row) * C + lane] = a.probs_orig[(int64_t(t) * n + i) * C + lane];
  }
}

int launch_loss_rows(const LossArgs& a, cudaStream_t st) {
  const int grid = (2 * a.btu + 2 * a.bs + 7) / 8;
  if (a.C <= 16) loss_rows_kernel<16><<<grid, 256, 0, st>>>(a);
  else loss_rows_kernel<32><<<grid, 256, 0, st>>>(a);
  CMLPL_CHECK_LAUNCH("train_loss_rows");
  return CMLPL_OK;
}
int launch_loss_graph(const LossArgs& a, cudaStream_t st) {
  const int grid = (a.btu + a.bs + 7) / 8;
  if (a.C <= 16) loss_graph_kernel<16><<<grid, 256, 0, st>>>(a);
  else loss_graph_kernel<32><<<grid, 256, 0, st>>>(a);
  CMLPL_CHECK_LAUNCH("train_loss_graph");
  return CMLPL_OK;
}

// ============================================================================ head backward
template <int CMAX, int W>
__global__ void __launch_bounds__(128)
head_bwd_kernel(HeadArgs a) {
  constexpr int CAT = TrainGeom<W>::CatDim, CONV = TrainGeom<W>::ConvFeat;
  __shared__ float red[4];
  const int s = blockIdx.x;
  const int tid = threadIdx.x;
  const int e = s / a.nb, r = s - e * a.nb;
  const float* wc = a.wc[e];
  const float* cat = a.cat + int64_t(s) * CAT;
  const float* dm = a.dmask + int64_t(s) * CAT;
  float* dcat = a.dcat + int64_t(s) * CAT;
  float dl[CMAX];
#pragma unroll
  for (int c = 0; c < CMAX; ++c) dl[c] = c < a.C ? a.dlogits[int64_t(s) * a.C + c] : 0.f;
  // L2-norm backward of the unlabelled rows' features (models.py:87-90; the labelled rows' features only feed the bank)
  const bool unl = r >= a.bs;
  const float* df = unl ? a.dfeat + (int64_t(e) * a.btu + (r - a.bs)) * kHid : nullptr;
  const float* ft = a.feat + int64_t(s) * kHid;
  float dot[1] = {0.f};
  if (unl)
    for (int j = tid; j < kHid; j += 128) dot[0] = fmaf(df[j], ft[j], dot[0]);
  block_sum4<1>(dot, red);
  const float inv_norm = 1.f / a.norm[s];
  float amax = 0.f;
  for (int g = tid; g < CAT / 4; g += 128) {
    float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < a.C) {
        const float4 w = ld4(wc + int64_t(c) * CAT + 4 * g);
        d.x = fmaf(dl[c], w.x, d.x); d.y = fmaf(dl[c], w.y, d.y); d.z = fmaf(dl[c], w.z, d.z); d.w = fmaf(dl[c], w.w, d.w);
      }
    }
    const float4 m = ld4(dm + 4 * g);
    d.x *= m.x; d.y *= m.y; d.z *= m.z; d.w *= m.w;
    if (4 * g < CONV) {
      *reinterpret_cast<float4*>(dcat + 4 * g) = d;
      amax = fmaxf(amax, fmaxf(fmaxf(fabsf(d.x), fabsf(d.y)), fmaxf(fabsf(d.z), fabsf(d.w))));
    } else {
      const int j = 4 * g - CONV;
      const float4 h = ld4(cat + 4 * g);
      if (unl) {
        const float4 f = ld4(ft + j), q = ld4(df + j);
        d.x += (q.x - f.x * dot[0]) * inv_norm; d.y += (q.y - f.y * dot[0]) * inv_norm;
        d.z += (q.z - f.z * dot[0]) * inv_norm; d.w += (q.w - f.w * dot[0]) * inv_norm;
      }
      float4 o;
      o.x = h.x > 0.f ? d.x : 0.f; o.y = h.y > 0.f ? d.y : 0.f; o.z = h.z > 0.f ? d.z : 0.f; o.w = h.w > 0.f ? d.w : 0.f;
      *reinterpret_cast<float4*>(a.dhp + int64_t(s) * kHid + j) = o;
    }
  }
  amax = warp_max(amax);
  if ((tid & 31) == 0 && amax > 0.f) atomicMax(reinterpret_cast<unsigned int*>(&a.prm_rw->grad_amax), __float_as_uint(amax));
}

int launch_head_bwd(const HeadArgs& a, int w, cudaStream_t st) {
  const int grid = 2 * a.nb;
  if (w == 11) {
    if (a.C <= 16) head_bwd_kernel<16, 11><<<grid, 128, 0, st>>>(a);
    else head_bwd_kernel<32, 11><<<grid, 128, 0, st>>>(a);
  } else {
    if (a.C <= 16) head_bwd_kernel<16, 20><<<grid, 128, 0, st>>>(a);
    else head_bwd_kernel<32, 20><<<grid, 128, 0, st>>>(a);
  }
  CMLPL_CHECK_LAUNCH("train_head_bwd");
  return CMLPL_OK;
}

// column reductions over the rows of one net: classifier weight gradient dWc[c][k] = sum_s dl[s][c] * cat[s][k] * mask[s][k],
// classifier bias gradient, feat_spe bias gradient dbs[j] = sum_s dhp[s][j].  grid (col blocks, net, row splits).
constexpr int kWgRows = 32;
template <int CMAX, int W>
__global__ void __launch_bounds__(256)
head_wgrad_kernel(HeadArgs a) {
  constexpr int CAT = TrainGeom<W>::CatDim;
  __shared__ float sdl[kWgRows][CMAX];
  const int e = blockIdx.y;
  const int r0 = blockIdx.z * kWgRows;
  const int rows = min(kWgRows, a.nb - r0);
  if (rows <= 0) return;
  const int64_t sb = int64_t(e) * a.nb + r0;
  for (int i = threadIdx.x; i < rows * CMAX; i += 256) {
    const int rr = i / CMAX, c = i - rr * CMAX;
    sdl[rr][c] = c < a.C ? a.dlogits[(sb + rr) * a.C + c] : 0.f;
  }
  __syncthreads();
  constexpr int kCatBlocks = (CAT + 255) / 256;
  if (int(blockIdx.x) < kCatBlocks) {
    const int k = blockIdx.x * 256 + threadIdx.x;
    if (k < CAT) {
      float acc[CMAX];
#pragma unroll
      for (int c = 0; c < CMAX; ++c) acc[c] = 0.f;
      for (int rr = 0; rr < rows; ++rr) {
        const float x = a.cat[(sb + rr) * CAT + k] * a.dmask[(sb + rr) * CAT + k];
#pragma unroll
        for (int c = 0; c < CMAX; ++c) acc[c] = fmaf(sdl[rr][c], x, acc[c]);
      }
#pragma unroll
      for (int c = 0; c < CMAX; ++c)
        if (c < a.C) atomicAdd(a.g_wc[e] + int64_t(c) * CAT + k, acc[c]);
    }
    if (blockIdx.x == 0 && threadIdx.x < a.C) {
      float b = 0.f;
      for (int rr = 0; rr < rows; ++rr) b += sdl[rr][threadIdx.x];
      atomicAdd(a.g_bc[e] + threadIdx.x, b);
    }
  } else {
    const int j = (blockIdx.x - kCatBlocks) * 256 + threadIdx.x;
    if (j < kHid) {
      float b = 0.f;
      for (int rr = 0; rr < rows; ++rr) b += a.dhp[(sb + rr) * kHid + j];
      atomicAdd(a.g_bs[e] + j, b);
    }
  }
}

int launch_head_wgrad(const HeadArgs& a, int w, cudaStream_t st) {
  const int cat = w == 11 ? TrainGeom<11>::CatDim : kCatDim;
  const dim3 grid((cat + 255) / 256 + kHid / 256, 2, (a.nb + kWgRows - 1) / kWgRows);
  if (w == 11) {
    if (a.C <= 16) head_wgrad_kernel<16, 11><<<grid, 256, 0, st>>>(a);
    else head_wgrad_kernel<32, 11><<<grid, 256, 0, st>>>(a);
  } else {
    if (a.C <= 16) head_wgrad_kernel<16, 20><<<grid, 256, 0, st>>>(a);
    else head_wgrad_kernel<32, 20><<<grid, 256, 0, st>>>(a);
  }
  CMLPL_CHECK_LAUNCH("train_head_wgrad");
  return CMLPL_OK;
}

// ============================================================================ Adam over every live tensor of both nets
__global__ void __launch_bounds__(256)
adam_all_kernel(AdamAll t) {
  const int ti = blockIdx.y;
  float* p = t.p[ti]; const float* g = t.g[ti]; float* m = t.m[ti]; float* v = t.v[ti];
  const int64_t n = t.n[ti];
  const cmlpl_train_params* prm = t.prm;
  const float b1 = prm->beta1, b2 = prm->beta2, eps = prm->eps;
  const float step_size = prm->lr / prm->bc1, bc2_sqrt = prm->bc2_sqrt;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const float gi = g[i];
    const float mi = m[i] + (gi - m[i]) * (1.f - b1);          // lerp form of torch's _single_tensor_adam
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = p[i] - step_size * (mi / denom);
  }
}

int launch_adam_all(const AdamAll& t, cudaStream_t st) {
  int64_t mx = 0;
  for (int i = 0; i < t.count; ++i) mx = t.n[i] > mx ? t.n[i] : mx;
  int gx = int((mx + 1023) / 1024);
  if (gx > 64) gx = 64;
  if (gx < 1) gx = 1;
  adam_all_kernel<<<dim3(gx, t.count), 256, 0, st>>>(t);
  CMLPL_CHECK_LAUNCH("train_adam");
  return CMLPL_OK;
}

}  // namespace cmlpl
