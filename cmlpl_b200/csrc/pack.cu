// Repack the reference's BaseNet2 state_dict tensors (tools/models.py:102-127) into the
// layouts the scene-inference kernels read (PackedLayout in common.cuh).
#include "common.cuh"

namespace cmlpl {

struct PackArgs {
  const float *c0w, *c0b, *c1w, *c1b, *c2w, *c2b, *sw, *sb, *cw, *cb;
  int B, C, P;
  unsigned char* out;
  PackedLayout L;
};

__global__ void pack_kernel(PackArgs a) {
  const int seg = blockIdx.y;
  const int64_t t0 = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int64_t step = int64_t(gridDim.x) * blockDim.x;
  unsigned char* o = a.out;
  switch (seg) {
    case 0:
    case 1: {  // conv1 / conv2 -> f16 [dx][kc][192 rows = (2-dy)*64 + n][8]  (UMMA no-swizzle K-major B operand;
               // rows ordered W(dy=2), W(dy=1), W(dy=0) so that tap pairs are contiguous N=128 blocks)
      const float* w = seg == 0 ? a.c1w : a.c2w;
      __half* d = reinterpret_cast<__half*>(o + (seg == 0 ? a.L.w1 : a.L.w2));
      for (int64_t i = t0; i < 3 * 8 * 192 * 8; i += step) {
        const int e = int(i & 7); const int64_t q = i >> 3; const int r = int(q % 192); const int kc = int((q / 192) & 7);
        const int dx = int(q / (192 * 8));
        const int dy = 2 - r / 64, n = r % 64, ci = kc * 8 + e;
        d[i] = __float2half_rn(w[(int64_t(n) * 64 + ci) * 9 + dy * 3 + dx]);
      }
    } break;
    case 2: {  // biases
      float* b1 = reinterpret_cast<float*>(o + a.L.b1);
      float* b2 = reinterpret_cast<float*>(o + a.L.b2);
      float* b0 = reinterpret_cast<float*>(o + a.L.b0);
      float* bs = reinterpret_cast<float*>(o + a.L.bspe);
      float* bc = reinterpret_cast<float*>(o + a.L.bc);
      for (int64_t i = t0; i < 64; i += step) { b1[i] = a.c1b[i]; b2[i] = a.c2b[i]; b0[i] = a.c0b[i]; }
      for (int64_t i = t0; i < 1024; i += step) bs[i] = a.sb[i];
      for (int64_t i = t0; i < a.L.nc || i < a.C; i += step) bc[i] = i < a.C ? a.cb[i] : 0.f;
    } break;
    case 3: {  // conv0 -> f32 [ci][n]
      float* d = reinterpret_cast<float*>(o + a.L.w0);
      for (int64_t i = t0; i < 60 * 64; i += step) {
        const int n = int(i & 63), ci = int(i >> 6);
        d[i] = a.c0w[n * 60 + ci];
      }
    } break;
    case 4: {  // feat_spe weight, as is
      float* d = reinterpret_cast<float*>(o + a.L.wspe);
      for (int64_t i = t0; i < int64_t(1024) * a.B; i += step) d[i] = a.sw[i];
    } break;
    case 5: {  // classifier: conv part permuted (ch,pos)->(pos,ch); spectral part as is
      float* dc = reinterpret_cast<float*>(o + a.L.wc_conv);
      float* ds = reinterpret_cast<float*>(o + a.L.wc_spe);
      const int P = a.P, in_f = 64 * P + 1024;
      for (int64_t i = t0; i < int64_t(a.C) * P * 64; i += step) {
        const int ch = int(i & 63); const int64_t r = i >> 6; const int pos = int(r % P), cls = int(r / P);
        dc[i] = a.cw[int64_t(cls) * in_f + ch * P + pos];
      }
      for (int64_t i = t0; i < int64_t(a.C) * 1024; i += step) {
        const int j = int(i & 1023), cls = int(i >> 10);
        ds[i] = a.cw[int64_t(cls) * in_f + 64 * P + j];
      }
    } break;
    case 6: {  // feat_spe weight -> f16 [4][KC][256][8], zero for k >= B
      __half* d = reinterpret_cast<__half*>(o + a.L.w1s);
      const int KC = a.L.kc_spe_in;
      for (int64_t i = t0; i < int64_t(4) * KC * 256 * 8; i += step) {
        const int e = int(i & 7), r = int((i >> 3) & 255); const int64_t q = i >> 11; const int kc = int(q % KC), nt = int(q / KC);
        const int k = kc * 8 + e, nrow = nt * 256 + r;
        d[i] = __float2half_rn(k < a.B ? a.sw[int64_t(nrow) * a.B + k] : 0.f);
      }
    } break;
    case 7: {  // classifier -> f16 [(P*8 + 128)][NC][8]; K order = (pos, ch) then spectral j
      __half* d = reinterpret_cast<__half*>(o + a.L.wc16);
      const int P = a.P, in_f = 64 * P + 1024, kc_conv = P * 8, NC = a.L.nc;
      for (int64_t i = t0; i < int64_t(kc_conv + 128) * NC * 8; i += step) {
        const int e = int(i & 7), cls = int((i >> 3) % NC), kc = int((i >> 3) / NC);
        float v = 0.f;
        if (cls < a.C) {
          if (kc < kc_conv) { const int pos = kc >> 3, ch = (kc & 7) * 8 + e; v = a.cw[int64_t(cls) * in_f + ch * P + pos]; }
          else { const int j = (kc - kc_conv) * 8 + e; v = a.cw[int64_t(cls) * in_f + 64 * P + j]; }
        }
        d[i] = __float2half_rn(v);
      }
    } break;
    case 8: {  // dense-path classifier: per block [8 kc][N][8], row = ((J-J0)*nI + (I-I0))*NC + cls, value = Wc[cls][ch,I,J] / 4 for
               // the middle classes; a border class arrives averaged over its two variants (conv2_scene_kernel), so its factor
               // doubles per border direction
      // w = 20: 5x5 pooled cells.  w = 11: 2x2 cells (I, J in {0, 1}) at the same border classes, every other map zero
      if (a.P != 25 && a.P != 4) break;
      __half* d = reinterpret_cast<__half*>(o + a.L.wcq);
      const int pw = a.P == 25 ? 5 : 2;                         // pooled cells per side
      const int in_f = 64 * a.P + 1024, NC = a.L.nc;
      for (int64_t i = t0; i < int64_t(25) * NC * 64; i += step) {
        int b = 0;
        while (b < 8 && i >= int64_t(blk_start(b + 1)) * NC * 64) ++b;
        const int Al = b / 3, Be = b % 3, N = blk_n(Al) * blk_n(Be) * NC;
        const int64_t li = i - int64_t(blk_start(b)) * NC * 64;
        const int e = int(li & 7), row = int((li >> 3) % N), kc = int((li >> 3) / N);
        // rows J-major: the maps of one pooled column J (all I of the block) are one contiguous B operand
        const int nI = blk_n(Al), cls = row % NC, ch = kc * 8 + e;
        const int I = blk_first(Al) + (row / NC) % nI, J = blk_first(Be) + (row / NC) / nI;
        const float sc = 0.25f * (Al != 1 ? 2.f : 1.f) * (Be != 1 ? 2.f : 1.f);
        d[i] = __float2half_rn(cls < a.C && I < pw && J < pw ? sc * a.cw[int64_t(cls) * in_f + ch * a.P + I * pw + J] : 0.f);
      }
    } break;
  }
}

}  // namespace cmlpl

using namespace cmlpl;

extern "C" size_t cmlpl_packed_bytes(int num_features, int num_classes, int w) {
  if (num_features <= 0 || num_classes <= 0 || w < 4) return 0;
  return packed_layout(num_features, num_classes, w).total;
}

extern "C" int cmlpl_pack_basenet2(const float* conv0_w, const float* conv0_b, const float* conv1_w,
                                   const float* conv1_b, const float* conv2_w, const float* conv2_b,
                                   const float* spe_w, const float* spe_b, const float* cls_w,
                                   const float* cls_b, int num_features, int num_classes, int w,
                                   void* packed, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(conv0_w && conv0_b && conv1_w && conv1_b && conv2_w && conv2_b && spe_w && spe_b && cls_w &&
                      cls_b && packed, "pack_basenet2: null pointer");
  CMLPL_CHECK_ARG(num_features > 0 && num_classes > 0 && num_classes <= 64 && w >= 4,
                  "pack_basenet2: bad dims (B=%d C=%d w=%d)", num_features, num_classes, w);
  PackArgs a;
  a.c0w = conv0_w; a.c0b = conv0_b; a.c1w = conv1_w; a.c1b = conv1_b; a.c2w = conv2_w; a.c2b = conv2_b;
  a.sw = spe_w; a.sb = spe_b; a.cw = cls_w; a.cb = cls_b;
  a.B = num_features; a.C = num_classes;
  a.L = packed_layout(num_features, num_classes, w);
  a.P = a.L.conv_pos;
  a.out = static_cast<unsigned char*>(packed);
  pack_kernel<<<dim3(64, 9), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  CMLPL_CHECK_LAUNCH("pack_basenet2");
  return CMLPL_OK;
}
