// Argument blocks and launchers of the fused training-step kernels (one translation unit each; train_step.cu strings
// them together behind cmlpl_train_step).
#pragma once
#include "common.cuh"

namespace cmlpl {

// Every trunk kernel exists for the window w = 20 and w = 11 (TrainGeom); the layouts below are written for w = 20,
// w = 11 packs the same regions at its own sizes (121 / 25 positions, cat width 1280).

// gather + noise + conv0 (train_fwd_sm100.cu)
struct Conv0Args {
  const float* cube; int scene_rows, cols;
  const int64_t* pix;              // [nb]
  const float* noise;              // [2][nb][60][w][w] or nullptr
  const float* w0[2]; const float* b0[2];
  const cmlpl_train_params* prm;
  __half* x16; __half* a0;         // [2*nb][8][400][8]
  int nb;
  // spectral input of the same sample: ynoisy[s] = spectra[row] + noise * sigma (train.py:158-182)
  const float* spectra; const int64_t* spec_row; const float* spec_noise; float* ynoisy; int bands;
  // block 0 also clears the per-step accumulators
  float* hist; cmlpl_train_params* prm_rw;
  // every CTA also converts a slice of the 3x3 weights to fp16 in the layouts the conv kernels read (wpack region)
  const float* w3[2][2];           // [net][conv1 | conv2] fp32 [64][64][3][3]
  unsigned char* wpack;
};
int launch_train_conv0(const Conv0Args& a, int w, cudaStream_t st);

// conv1 + pool + conv2 + pool (patch_cnn_sm100.cu, TRAIN instantiation)
struct TrainCnnArgs {
  const __half* a0;
  const unsigned char* wpack;      // fp16 packs written by train_conv0_kernel
  const float* b1[2]; const float* b2[2];
  __half* p1;                      // [2*nb][8][100][8]
  uint32_t* m1;                    // [2*nb][400][2]
  uint32_t* m2;                    // [2*nb][100][2]
  float* cat;                      // [2*nb][2624], first 1600 written here
  int nb;
};
int launch_train_cnn(const TrainCnnArgs& a, int w, cudaStream_t st);

// conv2 / conv1 backward: data gradient + weight gradient + bias gradient (train_bwd_sm100.cu)
struct ConvBwdArgs {
  const cmlpl_train_params* prm;
  const unsigned char* wpack[2];   // fp16 [tap][ci chunk][co][8 ci] of this conv, per net
  float* g_stage[2]; float* g_b[2];   // weight gradient staging [tap][co][ci] / bias gradient: accumulated into (zeroed by the caller)
  // H = 10 / 5 (conv2 of w = 20 / 11): dz2 is formed from dcat (dL/dcat, first 1600 / 256 columns), the ReLU mask
  //                 m2; activation = p1; the epilogue applies the pool backward + mask m1 and writes dz1
  // H = 20 / 11 (conv1): dz1 is read back; activation = a0; the epilogue writes da0
  const float* dcat; const uint32_t* m2; const uint32_t* m1;
  const __half* act;               // p1 or a0
  const __half* dz_in;             // dz1 (H = 20)
  __half* dz_out;                  // dz1 (H = 10) or da0 (H = 20)
  int nb;
};
int launch_train_conv_bwd(int H, const ConvBwdArgs& a, cudaStream_t st);

// conv0 weight gradient (train_bwd_sm100.cu)
struct Conv0BwdArgs {
  const cmlpl_train_params* prm;
  const __half* da0; const __half* x16;
  float* g_w[2]; float* g_b[2];
  int nb;
  // prologue: staged 3x3 weight gradients [net][conv][tap][co][ci] -> torch layout [co][ci][3][3]
  const float* gstage; float* g_w3[2][2];
};
int launch_train_conv0_bwd(const Conv0BwdArgs& a, int w, cudaStream_t st);

}  // namespace cmlpl
