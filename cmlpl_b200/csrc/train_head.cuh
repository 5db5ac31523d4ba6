// Argument blocks of train_head.cu (the non-convolutional kernels of the fused training step).
#pragma once
#include "common.cuh"

namespace cmlpl {

struct GemmProb {
  const float* A; int64_t a_rs, a_cs;      // A(m,k) = A[m*a_rs + k*a_cs]
  const float* B; int64_t b_rs, b_cs;      // B(k,n) = B[k*b_rs + n*b_cs]
  float* C; int64_t c_rs, c_cs;
  const float* bias;                       // per n, or nullptr
  const int* enable;                       // device flag: the problem is skipped when *enable == 0 (nullptr = always)
  int M, N, K;
  float alpha; int act;                    // act 1 = ReLU
};
struct MultiGemm { GemmProb p[4]; int count; };
int launch_multi_gemm(const MultiGemm& mg, cudaStream_t st, const char* name);

// S = A . B^T on tcgen05 (train_sim_sm100.cu).  mode 0: store the tile; mode 1: streaming bank-smoothing partials.
struct SimProb {
  const float* A; const float* B; int64_t lda, ldb;   // A [M, K], B [N, K], K contiguous
  int M, N, K, mode;
  float* Cout; int64_t ldc;                            // mode 0
  const float* qp; float* part; int C;                 // mode 1: queue_probs [N, C], part [2*ceil(N/128)][M][33]
  const int* enable;
};
struct SimBatch { SimProb p[4]; int count; const cmlpl_train_params* prm; };
int launch_sim_tc(const SimBatch& sb, cudaStream_t st, const char* name);

struct HeadArgs {
  const cmlpl_train_params* prm; cmlpl_train_params* prm_rw;
  int nb, bs, btu, C, training;
  const float* cat; float* dmask; const float* drop_mask;
  const float* wc[2]; const float* bc[2];
  float* logits; float* feat; float* norm;
  // backward
  const float* dlogits; const float* dfeat; float* dcat; float* dhp;
  float* g_wc[2]; float* g_bc[2]; float* g_bs[2];
};
// w = 20 or 11 selects the classifier input width (2624 / 1280; conv features 1600 / 256)
int launch_head_fwd(const HeadArgs& a, int w, cudaStream_t st);
int launch_head_bwd(const HeadArgs& a, int w, cudaStream_t st);
int launch_head_wgrad(const HeadArgs& a, int w, cudaStream_t st);

struct LossArgs {
  const cmlpl_train_params* prm;
  int bs, btu, C, queue;
  const float* logits; const float* feat; const int64_t* labels;
  const float* S;                  // bank-smoothing partials [2 banks][2*ceil(queue/128)][btu][33]
  const float* G; float* dG;
  float* queue_feats[2]; float* queue_probs[2];
  float* probs_orig; float* probs; float* mask;
  float* dlogits; float* hist;
};
int launch_loss_rows(const LossArgs& a, cudaStream_t st);
int launch_loss_graph(const LossArgs& a, cudaStream_t st);

struct AdamAll {
  float* p[2 * CMLPL_TRAIN_TENSORS]; const float* g[2 * CMLPL_TRAIN_TENSORS];
  float* m[2 * CMLPL_TRAIN_TENSORS]; float* v[2 * CMLPL_TRAIN_TENSORS];
  int64_t n[2 * CMLPL_TRAIN_TENSORS];
  int count;
  const cmlpl_train_params* prm;
};
int launch_adam_all(const AdamAll& t, cudaStream_t st);

}  // namespace cmlpl
