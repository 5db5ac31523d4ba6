// Loss kernels of the mutual-learning step (train.py:191-265) and NT-Xent (tools/models.py:14-39).
// fp32 throughout (parity bar rtol 1e-5).  Matrix products go through the tiled GEMM core; the
// per-row softmax / masking / normalisation logic is fused into one warp-per-row kernel per loss
// (warp-shuffle reductions), forward and gradient in the same pass.
#include "common.cuh"
#include "gemm_core.cuh"

namespace cmlpl {

// ---------------------------------------------------------------- cross entropy (hard / soft+mask)
// one thread per row (C <= 64 classes)
__global__ void ce_kernel(const float* __restrict__ z, const int64_t* __restrict__ labels, const float* __restrict__ probs,
                          const float* __restrict__ mask, int64_t rows, int C, float scale, float* __restrict__ loss,
                          float* __restrict__ dz) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  float li = 0.f;
  if (r < rows) {
    const float* zr = z + r * C;
    float mx = -INFINITY;
    for (int c = 0; c < C; ++c) mx = fmaxf(mx, zr[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(zr[c] - mx);
    const float lse = mx + logf(se);
    const float m = mask ? mask[r] : 1.f;
    const float g = scale / float(rows);
    if (labels) {
      const int y = int(labels[r]);
      const bool ok = y >= 0 && y < C;                       // e.g. ignore_index 255 with mask 0
      li = ok ? -(zr[y] - lse) * m : 0.f;
      if (dz)
        for (int c = 0; c < C; ++c) dz[r * C + c] = ok ? g * m * (expf(zr[c] - lse) - (c == y ? 1.f : 0.f)) : 0.f;
    } else {
      const float* pr = probs + r * C;
      float tsum = 0.f, dot = 0.f;
      for (int c = 0; c < C; ++c) { tsum += pr[c]; dot += (zr[c] - lse) * pr[c]; }
      li = -dot * m;
      if (dz)
        for (int c = 0; c < C; ++c) dz[r * C + c] = g * m * (expf(zr[c] - lse) * tsum - pr[c]);
    }
  }
  li = warp_sum(li);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = li;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(loss, v * scale / float(rows));
  }
}

// ---------------------------------------------------------------- softmax entropy (loss_helper.py:247-248)
// entropy_i = -sum_c p_ic * log(p_ic + eps),  p = softmax(z_i); one thread per row
__global__ void softmax_entropy_kernel(const float* __restrict__ z, int64_t rows, int C, float eps, float* __restrict__ ent) {
  const int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (r >= rows) return;
  const float* zr = z + r * C;
  float mx = -INFINITY;
  for (int c = 0; c < C; ++c) mx = fmaxf(mx, zr[c]);
  float se = 0.f;
  for (int c = 0; c < C; ++c) se += expf(zr[c] - mx);
  float e = 0.f;
  for (int c = 0; c < C; ++c) { const float p = expf(zr[c] - mx) / se; e -= p * logf(p + eps); }
  ent[r] = e;
}

// ---------------------------------------------------------------- softmax JS divergence (trian_CCT.py:76-84)
// loss = 0.5 * (kl_div(log_softmax(z), M, 'mean') + kl_div(log(t + 1e-5), M, 'mean')),  M = (softmax(z) + t) / 2,
// 'mean' = over all rows*C elements.  One thread per row; gradient w.r.t. z in the same pass (t is a constant):
//   f_k = 2 M log M - M log p - M log(t + eps);  g_k = df/dp_k = h_k - M_k/p_k,  h_k = log M + 1 - log(p)/2 - log(t + eps)/2
//   dz_j = p_j (g_j - sum_k g_k p_k) * cf = (p_j h_j - M_j - p_j sum_k (p_k h_k - M_k)) * cf,  cf = scale * 0.5 / (rows*C)
// The second form has no M/p: where the softmax underflows (a logit ~88 or more below the row's max) p is 0 or a
// denormal, and M/p would be inf or 0/0 and turn the whole row of dz into NaN.
__global__ void js_kernel(const float* __restrict__ z, const float* __restrict__ t, int64_t rows, int C, float scale,
                          float* __restrict__ loss, float* __restrict__ dz) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  float li = 0.f;
  if (r < rows) {
    const float* zr = z + r * C; const float* tr = t + r * C;
    float mx = -INFINITY;
    for (int c = 0; c < C; ++c) mx = fmaxf(mx, zr[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(zr[c] - mx);
    const float lse = mx + logf(se);
    float gp = 0.f;
    for (int c = 0; c < C; ++c) {
      const float lp = zr[c] - lse, p = expf(lp), tt = tr[c];
      const float M = 0.5f * (p + tt), lt = logf(tt + 1e-5f);
      const float lM = M > 0.f ? logf(M) : 0.f;                // xlogy: 0 * log 0 = 0 (F.kl_div)
      li += M * (lM - lp) + M * (lM - lt);
      gp += p * (lM + 1.f - 0.5f * lp - 0.5f * lt) - M;
    }
    if (dz) {
      const float cf = scale * 0.5f / (float(rows) * float(C));
      for (int c = 0; c < C; ++c) {
        const float lp = zr[c] - lse, p = expf(lp), tt = tr[c];
        const float M = 0.5f * (p + tt), lt = logf(tt + 1e-5f);
        const float lM = M > 0.f ? logf(M) : 0.f;
        dz[r * C + c] = cf * (p * (lM + 1.f - 0.5f * lp - 0.5f * lt) - M - p * gp);
      }
    }
  }
  li = warp_sum(li);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = li;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(loss, v * scale * 0.5f / (float(rows) * float(C)));
  }
}

// ---------------------------------------------------------------- memory-bank smoothing (train.py:203-222)
// one warp per row: probs_orig = softmax(z); A = exp(S/T) over the bank (S = f.Qf^T precomputed by the
// GEMM core, streamed once), probs = alpha*p + (1-alpha) * (A/sum A).Qp ; mask = max(probs) >= thr
template <int CMAX>
__global__ void bank_smooth_kernel(const float* __restrict__ z, const float* __restrict__ S, const float* __restrict__ qp,
                                   int64_t rows, int C, int64_t queue, float alpha, float invT, int smooth, float thr,
                                   float* __restrict__ probs_orig, float* __restrict__ probs, float* __restrict__ mask) {
  const int64_t r = blockIdx.x * int64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* zr = z + r * C;
  float mx = -INFINITY;
  for (int c = 0; c < C; ++c) mx = fmaxf(mx, zr[c]);
  float se = 0.f;
  for (int c = 0; c < C; ++c) se += expf(zr[c] - mx);
  float p[CMAX];
#pragma unroll
  for (int c = 0; c < CMAX; ++c) p[c] = c < C ? expf(zr[c] - mx) / se : 0.f;
  if (lane == 0 && probs_orig)
    for (int c = 0; c < C; ++c) probs_orig[r * C + c] = p[c];
  if (smooth) {
    float asum = 0.f, acc[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) acc[c] = 0.f;
    for (int64_t j = lane; j < queue; j += 32) {
      const float a = expf(S[r * queue + j] * invT);      // |f.q| <= 1 => plain exp is safe (train.py:213)
      asum += a;
#pragma unroll
      for (int c = 0; c < CMAX; ++c)
        if (c < C) acc[c] = fmaf(a, qp[j * C + c], acc[c]);
    }
    asum = warp_sum(asum);
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
      if (c < C) p[c] = alpha * p[c] + (1.f - alpha) * (warp_sum(acc[c]) / asum);
  }
  if (lane == 0) {
    float best = -INFINITY;
    for (int c = 0; c < C; ++c) { probs[r * C + c] = p[c]; best = fmaxf(best, p[c]); }
    mask[r] = best >= thr ? 1.f : 0.f;
  }
}

// ---------------------------------------------------------------- pseudo-label graph contrastive (train.py:246-265)
// one warp per row i of G = f_row.f_col^T (precomputed) and Q0 = p1.p^T (precomputed, diagonal forced to 1):
//   sp = softmax_j(G/T);  a = Q0[Q0>=0.8]/sum ;  b = (1-Q0)[Q0<=0.3]/(sum+1e-8)
//   L_i = -sum_j a log sp + sum_j b log(sp+1)
//   dL_i/dl_ik = (-a_ik + b_ik sp_ik/(sp_ik+1)) - sp_ik * sum_j(-a_ij + b_ij sp_ij/(sp_ij+1)),  l = G/T
__global__ void graph_contrast_kernel(const float* __restrict__ G, float* __restrict__ Q0, int64_t n, float invT,
                                      float scale, float* __restrict__ loss, float* __restrict__ dG) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= n) return;
  const int lane = threadIdx.x & 31;
  const float* g = G + i * n;
  float* q = Q0 + i * n;
  float z = 0.f, qs = 0.f, qns = 0.f;
  for (int64_t j = lane; j < n; j += 32) {
    z += expf(g[j] * invT);                                 // unit-norm features: |logit| <= 1/T
    const float q0 = (j == i) ? 1.f : q[j];                 // fill_diagonal_(1)  (train.py:250)
    if (q0 >= 0.8f) qs += q0;
    if (q0 <= 0.3f) qns += 1.f - q0;
  }
  z = warp_sum(z); qs = warp_sum(qs); qns = warp_sum(qns);
  const float inv_qs = 1.f / qs, inv_qns = 1.f / (qns + 1e-8f);
  float li = 0.f, w = 0.f;
  for (int64_t j = lane; j < n; j += 32) {
    const float sp = expf(g[j] * invT) / z;
    const float q0 = (j == i) ? 1.f : q[j];
    const float a = q0 >= 0.8f ? q0 * inv_qs : 0.f;
    const float b = q0 <= 0.3f ? (1.f - q0) * inv_qns : 0.f;
    li += -logf(sp) * a + logf(sp + 1.f) * b;
    w += -a + b * sp / (sp + 1.f);
  }
  li = warp_sum(li); w = warp_sum(w);
  if (dG) {
    const float c = scale * invT / float(n);
    for (int64_t j = lane; j < n; j += 32) {
      const float sp = expf(g[j] * invT) / z;
      const float q0 = (j == i) ? 1.f : q[j];
      const float a = q0 >= 0.8f ? q0 * inv_qs : 0.f;
      const float b = q0 <= 0.3f ? (1.f - q0) * inv_qns : 0.f;
      dG[i * n + j] = c * ((-a + b * sp / (sp + 1.f)) - sp * w);
    }
  }
  if (lane == 0) atomicAdd(loss, li * scale / float(n));
}

// ---------------------------------------------------------------- NT-Xent (models.py:22-39)
// one warp per row i of S = z.z^T (z unit rows, [2bs, 2bs]): loss_i = -pos_i/T + log sum_{k!=i} exp(S_ik/T)
//   dS_ik = (1/(2bs)) * ( softmax_{k!=i}(S_i/T)_k - [k == partner(i)] ) / T
__global__ void ntxent_kernel(const float* __restrict__ S, int64_t bs, float invT, float* __restrict__ loss,
                              float* __restrict__ dS) {
  const int64_t n = 2 * bs;
  const int64_t i = blockIdx.x * int64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= n) return;
  const int lane = threadIdx.x & 31;
  const float* s = S + i * n;
  const int64_t partner = i < bs ? i + bs : i - bs;
  float den = 0.f;
  for (int64_t k = lane; k < n; k += 32)
    if (k != i) den += expf(s[k] * invT);
  den = warp_sum(den);
  if (dS) {
    const float c = invT / float(n);
    for (int64_t k = lane; k < n; k += 32) {
      float v = (k != i) ? expf(s[k] * invT) / den : 0.f;
      if (k == partner) v -= 1.f;
      dS[i * n + k] = c * v;
    }
  }
  if (lane == 0) atomicAdd(loss, (-s[partner] * invT + logf(den)) / float(n));
}

// C = A + A^T (in place on a square matrix): dz needs (dS + dS^T).z
__global__ void symmetrize_kernel(float* __restrict__ A, int64_t n) {
  const int64_t t = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (t >= n * n) return;
  const int64_t i = t / n, j = t - i * n;
  if (i < j) { const float v = A[i * n + j] + A[j * n + i]; A[i * n + j] = v; A[j * n + i] = v; }
  else if (i == j) A[t] = 2.f * A[t];
}

// ---------------------------------------------------------------- fused multi-tensor Adam (torch.optim.Adam defaults)
struct AdamTable {
  float* p[16]; const float* g[16]; float* m[16]; float* v[16]; int64_t n[16];
  int count;
};
__global__ void adam_kernel(AdamTable t, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt) {
  const int ti = blockIdx.y;
  if (ti >= t.count || t.g[ti] == nullptr) return;
  float* p = t.p[ti]; const float* g = t.g[ti]; float* m = t.m[ti]; float* v = t.v[ti];
  const int64_t n = t.n[ti];
  const float step_size = lr / bc1;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const float gi = g[i];
    const float mi = m[i] + (gi - m[i]) * (1.f - b1);          // lerp form used by torch's _single_tensor_adam
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = p[i] - step_size * (mi / denom);
  }
}

}  // namespace cmlpl

using namespace cmlpl;

// Similarity matrices S = A . B^T (both operands [rows, K] with K contiguous) of the loss entry points: fp32 FFMA tiles by
// default (the 1e-5 parity path); mode 1 rounds the operands to fp16 and runs them on tcgen05 (cmlpl_sim_nt_tc_f32,
// |d| ~ 1e-4 on unit-norm features) -- at the config-3 stress size the CUDA-core GEMM dominates these calls.
static thread_local int g_loss_gemm_mode = 0;
extern "C" int cmlpl_set_loss_gemm_mode(int mode) {
  CMLPL_CHECK_ARG(mode == 0 || mode == 1, "set_loss_gemm_mode: 0 (fp32 CUDA cores) or 1 (tcgen05 fp16 operands)");
  g_loss_gemm_mode = mode;
  return CMLPL_OK;
}
static int sim_nt(const float* A, const float* B, int M, int N, int K, float* C, cudaStream_t s, const char* name) {
  if (g_loss_gemm_mode == 1 && K % 64 == 0 && reinterpret_cast<uintptr_t>(A) % 16 == 0 && reinterpret_cast<uintptr_t>(B) % 16 == 0)
    return cmlpl_sim_nt_tc_f32(A, B, M, N, K, C, s);
  return launch_gemm(M, N, K, 1, StridedA{A, K, 1}, StridedB{B, 1, K}, StridedC{C, N, 1, nullptr, 1.f, 0.f, 0}, s, name);
}

extern "C" int cmlpl_ce_fwd_bwd_f32(const float* logits, const int64_t* labels, const float* probs, const float* mask,
                                    int64_t rows, int C, float scale, float* loss, float* dlogits, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(logits && loss, "ce: null pointer");
  CMLPL_CHECK_ARG((labels != nullptr) != (probs != nullptr), "ce: pass exactly one of labels / probs");
  CMLPL_CHECK_ARG(rows >= 0 && C > 0 && C <= 4096, "ce: bad dims");
  if (rows == 0) return CMLPL_OK;
  ce_kernel<<<int((rows + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(logits, labels, probs, mask, rows, C,
                                                                                    scale, loss, dlogits);
  CMLPL_CHECK_LAUNCH("ce");
  return CMLPL_OK;
}

extern "C" int cmlpl_softmax_js_f32(const float* logits, const float* targets, int64_t rows, int C, float scale,
                                    float* loss, float* dlogits, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(logits && targets && loss, "softmax_js: null pointer");
  CMLPL_CHECK_ARG(rows >= 0 && C > 0 && C <= 4096, "softmax_js: bad dims");
  if (rows == 0) return CMLPL_OK;
  js_kernel<<<int((rows + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(logits, targets, rows, C, scale, loss, dlogits);
  CMLPL_CHECK_LAUNCH("softmax_js");
  return CMLPL_OK;
}

extern "C" int cmlpl_softmax_entropy_f32(const float* logits, int64_t rows, int C, float eps, float* entropy,
                                         cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(logits && entropy && rows >= 0 && C > 0, "softmax_entropy: bad args");
  if (rows == 0) return CMLPL_OK;
  softmax_entropy_kernel<<<int((rows + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(logits, rows, C, eps, entropy);
  CMLPL_CHECK_LAUNCH("softmax_entropy");
  return CMLPL_OK;
}

extern "C" int cmlpl_bank_smooth_f32(const float* logits, const float* feats, const float* queue_feats,
                                     const float* queue_probs, int64_t rows, int C, int dim, int64_t queue, float alpha,
                                     float T, int smooth, float thr, float* work, float* probs_orig, float* probs,
                                     float* mask, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(logits && probs && mask, "bank_smooth: null pointer");
  CMLPL_CHECK_ARG(rows >= 0 && C > 0 && C <= 32 && T > 0, "bank_smooth: bad dims (C=%d)", C);
  CMLPL_CHECK_ARG(!smooth || (feats && queue_feats && queue_probs && work && queue > 0 && dim > 0),
                  "bank_smooth: smoothing needs feats, bank and a [rows, queue] work buffer");
  if (rows == 0) return CMLPL_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (smooth) {   // S = feats . queue_feats^T   (train.py:213)
    int rc = sim_nt(feats, queue_feats, int(rows), int(queue), dim, work, s, "bank_sim");
    if (rc != CMLPL_OK) return rc;
  }
  const int grid = int((rows + 3) / 4);
  if (C <= 16)
    bank_smooth_kernel<16><<<grid, 128, 0, s>>>(logits, work, queue_probs, rows, C, queue, alpha, 1.f / T, smooth, thr,
                                                probs_orig, probs, mask);
  else
    bank_smooth_kernel<32><<<grid, 128, 0, s>>>(logits, work, queue_probs, rows, C, queue, alpha, 1.f / T, smooth, thr,
                                                probs_orig, probs, mask);
  CMLPL_CHECK_LAUNCH("bank_smooth");
  return CMLPL_OK;
}

extern "C" int cmlpl_graph_contrast_f32(const float* f_row, const float* f_col, const float* p1, const float* p,
                                        int64_t n, int dim, int C, float T, int grad_side, float scale, float* work,
                                        float* loss, float* dfeat, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(f_row && f_col && p1 && p && work && loss, "graph_contrast: null pointer");
  CMLPL_CHECK_ARG(n > 0 && dim > 0 && C > 0 && T > 0 && (grad_side == 0 || grad_side == 1), "graph_contrast: bad args");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* G = work; float* Q0 = work + n * n; float* dG = work + 2 * n * n;
  int rc = sim_nt(f_row, f_col, int(n), int(n), dim, G, s, "graph_sim");                  // train.py:246 / :257
  if (rc != CMLPL_OK) return rc;
  rc = launch_gemm(int(n), int(n), C, 1, StridedA{p1, C, 1}, StridedB{p, 1, C},
                   StridedC{Q0, n, 1, nullptr, 1.f, 0.f, 0}, s, "graph_q0");              // train.py:249
  if (rc != CMLPL_OK) return rc;
  graph_contrast_kernel<<<int((n + 3) / 4), 128, 0, s>>>(G, Q0, n, 1.f / T, scale, loss, dfeat ? dG : nullptr);
  CMLPL_CHECK_LAUNCH("graph_contrast");
  if (dfeat) {
    if (grad_side == 0)   // d f_row = dG . f_col
      rc = launch_gemm(int(n), dim, int(n), 1, StridedA{dG, n, 1}, StridedB{f_col, dim, 1},
                       StridedC{dfeat, dim, 1, nullptr, 1.f, 0.f, 0}, s, "graph_dfrow");
    else                  // d f_col = dG^T . f_row
      rc = launch_gemm(int(n), dim, int(n), 1, StridedA{dG, 1, n}, StridedB{f_row, dim, 1},
                       StridedC{dfeat, dim, 1, nullptr, 1.f, 0.f, 0}, s, "graph_dfcol");
  }
  return rc;
}

extern "C" int cmlpl_ntxent_f32(const float* z, int64_t bs, int dim, float T, float* work, float* loss, float* dz,
                                cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(z && work && loss, "ntxent: null pointer");
  CMLPL_CHECK_ARG(bs > 0 && dim > 0 && T > 0, "ntxent: bad args");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t n = 2 * bs;
  float* S = work; float* dS = work + n * n;
  int rc = sim_nt(z, z, int(n), int(n), dim, S, s, "ntxent_sim");                        // models.py:27 on unit rows
  if (rc != CMLPL_OK) return rc;
  ntxent_kernel<<<int((n + 3) / 4), 128, 0, s>>>(S, bs, 1.f / T, loss, dz ? dS : nullptr);
  CMLPL_CHECK_LAUNCH("ntxent");
  if (dz) {
    symmetrize_kernel<<<int((n * n + 255) / 256), 256, 0, s>>>(dS, n);
    CMLPL_CHECK_LAUNCH("ntxent_sym");
    rc = launch_gemm(int(n), dim, int(n), 1, StridedA{dS, n, 1}, StridedB{z, dim, 1},
                     StridedC{dz, dim, 1, nullptr, 1.f, 0.f, 0}, s, "ntxent_dz");
  }
  return rc;
}

extern "C" int cmlpl_adam_multi_f32(int n_tensors, float* const* p_host, const float* const* g_host, float* const* m_host,
                                    float* const* v_host, const int64_t* numel_host, float lr, float beta1, float beta2,
                                    float eps, int step, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(n_tensors >= 0 && p_host && g_host && m_host && v_host && numel_host, "adam: null table");
  CMLPL_CHECK_ARG(step >= 1, "adam: step must be >= 1");
  // bias corrections in double like torch's Python-side scalars (torch/optim/adam.py _single_tensor_adam)
  const float bc1 = float(1.0 - pow(double(beta1), double(step)));
  const float bc2_sqrt = float(sqrt(1.0 - pow(double(beta2), double(step))));
  for (int base = 0; base < n_tensors; base += 16) {
    AdamTable t;
    t.count = n_tensors - base < 16 ? n_tensors - base : 16;
    int64_t mx = 0;
    for (int i = 0; i < t.count; ++i) {
      t.p[i] = p_host[base + i]; t.g[i] = g_host[base + i]; t.m[i] = m_host[base + i]; t.v[i] = v_host[base + i];
      t.n[i] = numel_host[base + i];
      // an empty tensor may have null pointers (torch allocates nothing for it); the kernel never touches them
      CMLPL_CHECK_ARG(t.n[i] == 0 || (t.p[i] && t.m[i] && t.v[i] && t.n[i] > 0), "adam: null tensor %d", base + i);
      if (t.g[i] && t.n[i] > mx) mx = t.n[i];
    }
    if (mx == 0) continue;
    int gx = int((mx + 255) / 256); if (gx > 2 * sm_count()) gx = 2 * sm_count();
    adam_kernel<<<dim3(gx, t.count), 256, 0, static_cast<cudaStream_t>(stream)>>>(t, lr, beta1, beta2, eps, bc1, bc2_sqrt);
    CMLPL_CHECK_LAUNCH("adam");
  }
  return CMLPL_OK;
}
