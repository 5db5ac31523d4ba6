// Shared helpers for libcmlpl_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>

#include "../../include/cmlpl.h"

namespace cmlpl {

void set_error(const char* fmt, ...);

#define CMLPL_CHECK_ARG(cond, ...)                     \
  do {                                                 \
    if (!(cond)) {                                     \
      ::cmlpl::set_error(__VA_ARGS__);                 \
      return CMLPL_ERR_ARG;                            \
    }                                                  \
  } while (0)

#define CMLPL_CHECK_LAUNCH(name)                                                      \
  do {                                                                                \
    cudaError_t e__ = cudaGetLastError();                                             \
    if (e__ != cudaSuccess) {                                                         \
      ::cmlpl::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));    \
      return CMLPL_ERR_CUDA;                                                          \
    }                                                                                 \
  } while (0)

#define CMLPL_CUDA(call)                                                              \
  do {                                                                                \
    cudaError_t e__ = (call);                                                         \
    if (e__ != cudaSuccess) {                                                         \
      ::cmlpl::set_error("%s failed: %s", #call, cudaGetErrorString(e__));           \
      return CMLPL_ERR_CUDA;                                                          \
    }                                                                                 \
  } while (0)

// opt a kernel into `bytes` of dynamic shared memory; the attribute call is made once per (call site, device) and
// again only if a larger size is requested -- it costs microseconds of host time that a 1 ms step cannot hide
#define CMLPL_MAX_DYN_SMEM(kernel, bytes)                                                             \
  do {                                                                                                \
    static int set__[64];                                                                             \
    int dev__ = 0;                                                                                    \
    if (cudaGetDevice(&dev__) != cudaSuccess || dev__ < 0 || dev__ >= 64) dev__ = 0;                  \
    if (int(bytes) > set__[dev__]) {                                                                  \
      CMLPL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes))); \
      set__[dev__] = int(bytes);                                                                      \
    }                                                                                                 \
  } while (0)

// number of SMs of the current device (cached)
int sm_count();

// Fork / join inside one C call: kernels without a mutual dependency (the scene's spectral branch next to its conv tower;
// in the training step the spectral GEMM next to the conv trunk and the head weight gradients next to the conv backward
// chain) run on a side stream between a fork and a join event.  Works the same in eager mode and under stream capture
// (the events become graph edges).  One side stream and two event pairs per device, created together on first use and
// kept for the life of the process -- the only persistent resources the library owns.  A caller holds `mu` from its
// first fork to its last join, so host threads that drive the same device from several streams take turns (the
// launches are microseconds) and never enqueue onto a side stream that another thread's capture has forked.
struct SideStream {
  cudaStream_t s = nullptr;
  cudaEvent_t fork[2] = {nullptr, nullptr}, join[2] = {nullptr, nullptr};
  std::mutex mu;
};
// the current device's side stream, or nullptr if it cannot be created
SideStream* side_stream();

// Band-major raw slab (include/cmlpl.h: CMLPL_RAW_BIL / CMLPL_RAW_BSQ): the sample of slab row r, column c, band b is
// at r * rs + c + b * bs (BIL: rs = B * cols, bs = cols; BSQ: rs = cols, bs = slab_rows * cols).
struct BandMajor {
  int cols;
  int64_t rs, bs;
};

// The raw cube code (include/cmlpl.h): dtype = sample (CMLPL_RAW_U16 / F32 / I16) | interleave (CMLPL_RAW_BIP / BIL /
// BSQ).  Bytes per sample:
inline int raw_sample_bytes(int dtype) { return (dtype & 0x0f) == CMLPL_RAW_F32 ? 4 : 2; }
// Checks a code and the alignment of the pointer `what` to its samples; `fn` names the entry point.  No CUDA call.
inline int check_raw_code(const char* fn, const char* what, const void* p, int dtype) {
  CMLPL_CHECK_ARG((dtype & ~0xff) == 0, "%s: dtype 0x%x has bits outside sample (0x0f) and interleave (0xf0)", fn,
                  unsigned(dtype));
  CMLPL_CHECK_ARG((dtype & 0x0f) <= CMLPL_RAW_I16, "%s: unknown sample type %d (0 = uint16, 1 = float32, 2 = int16)", fn,
                  dtype & 0x0f);
  CMLPL_CHECK_ARG((dtype & 0xf0) <= CMLPL_RAW_BSQ, "%s: unknown interleave 0x%x (0x00 = BIP, 0x10 = BIL, 0x20 = BSQ)", fn,
                  unsigned(dtype & 0xf0));
  CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(p) % raw_sample_bytes(dtype) == 0, "%s: %s must be aligned to its %d-byte samples",
                  fn, what, raw_sample_bytes(dtype));
  return CMLPL_OK;
}
// Strides of a BIL / BSQ cube of B bands whose planes hold plane_rows rows of cols samples (BIP is not band-major)
inline BandMajor band_major(int dtype, int B, int64_t plane_rows, int cols) {
  return (dtype & 0xf0) == CMLPL_RAW_BSQ ? BandMajor{cols, int64_t(cols), plane_rows * cols}
                                         : BandMajor{cols, int64_t(B) * cols, int64_t(cols)};
}

// a1 index map (tools/hyper_tools.py:35-55 == symmetric padding): single reflection.
__host__ __device__ __forceinline__ int mirror_index(int o, int n) {
  return o < 0 ? -o - 1 : (o >= n ? 2 * n - 1 - o : o);
}

// window of pixel r: rows r+lo .. r+lo+w-1.  even w (ExtractPatches): lo=-w/2;
// odd w (ExtractPatches_for_base): lo=-(w-1)/2.   Both equal -(w/2) in integer division.
__host__ __device__ __forceinline__ int window_lo(int w) { return -(w / 2); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- class bookkeeping of the dense (scene-level) conv2 / pool / classifier path (conv2_scene_sm100.cu) ----
// pooled row/column index that represents conv2 class k (0: i=0, 1: i=1, 2: i=2..7, 3: i=8, 4: i=9) of a
// 10-wide pooled window, and the PM border class (top/mid/bot) of pooled index i
__host__ __device__ constexpr int rep_of(int k) { return k == 0 ? 0 : (k == 1 ? 1 : (k == 2 ? 4 : (k == 3 ? 8 : 9))); }
__host__ __device__ constexpr int cls_of(int i) { return i == 0 ? 0 : (i == 9 ? 2 : 1); }
// block b = Alpha*3 + Beta: number of I / J values, first map index, Y classes per (Alpha,u)
__host__ __device__ constexpr int blk_n(int cls) { return cls == 1 ? 3 : 1; }
__host__ __device__ constexpr int blk_first(int cls) { return cls == 0 ? 0 : (cls == 1 ? 1 : 4); }
__host__ __device__ constexpr int blk_start(int b) {
  return b == 0 ? 0 : b == 1 ? 1 : b == 2 ? 4 : b == 3 ? 5 : b == 4 ? 8 : b == 5 ? 17 : b == 6 ? 20 : b == 7 ? 21 : 24;
}

// ---- packed BaseNet2 weights (layout shared by pack.cu and the scene kernels) ----
// All offsets in bytes from the start of the packed buffer, 256-B aligned.
struct PackedLayout {
  size_t w1;      // f16 [3 dx][8 kchunks][192 rows = (2-dy)*64+n][8]   conv1, UMMA no-swizzle K-major B operand
  size_t w2;      // f16 same for conv2
  size_t b1;      // f32 [64]
  size_t b2;      // f32 [64]
  size_t w0;      // f32 [60][64]  conv0 weight transposed (ci-major) for the per-pixel map
  size_t b0;      // f32 [64]
  size_t wspe;    // f32 [1024][B]  (as in the state dict)
  size_t bspe;    // f32 [1024]
  size_t wc_conv; // f32 [C][P*64]   classifier columns of the conv features, permuted to (pos, ch)
  size_t wc_spe;  // f32 [C][1024]
  size_t bc;      // f32 [C] (padded to NC)
  size_t w1s;     // f16 [4 n-tiles][KC][256][8]  feat_spe weight, UMMA B operand tiles (K padded to 16)
  size_t wc16;    // f16 [(P*8 + 128) k-chunks][NC classes][8]  classifier over [conv(pos,ch) | spectral]
  size_t wcq;     // f16 per (Alpha,Beta) block [8 k-chunks][N = maps*NC rows = map*NC+cls][8]: 0.25 * conv classifier
                  //     columns of pooled cell (I,J), per border block (Al,Be), rows J-major (w = 20 only; pool2_cls_kernel)
  size_t total;
  int conv_pos;   // P = (w/4)^2 pooled positions
  int kc_spe_in;  // KC = ceil(B/16)*2: 16-byte K-chunks of the spectral input
  int nc;         // NC: class width of the tensor-core classifier blocks, 16 (C <= 16) or 32
};

__host__ __device__ inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// class width of the tensor-core classifier operands and of the dense path's partial maps: one MMA N of 16 up to 16
// classes, 32 beyond (C > 32 has no tensor-core classifier; its packed blocks hold the first 32 classes and go unread)
__host__ __device__ constexpr int class_width(int C) { return C <= 16 ? 16 : 32; }

__host__ __device__ inline PackedLayout packed_layout(int B, int C, int w) {
  PackedLayout L;
  int p = (w / 2) / 2;
  L.conv_pos = p * p;
  L.nc = class_width(C);
  size_t o = 0;
  L.w1 = o; o = align256(o + 9 * 8 * 64 * 8 * 2);
  L.w2 = o; o = align256(o + 9 * 8 * 64 * 8 * 2);
  L.b1 = o; o = align256(o + 64 * 4);
  L.b2 = o; o = align256(o + 64 * 4);
  L.w0 = o; o = align256(o + 60 * 64 * 4);
  L.b0 = o; o = align256(o + 64 * 4);
  L.wspe = o; o = align256(o + size_t(1024) * B * 4);
  L.bspe = o; o = align256(o + 1024 * 4);
  L.wc_conv = o; o = align256(o + size_t(C) * L.conv_pos * 64 * 4);
  L.wc_spe = o; o = align256(o + size_t(C) * 1024 * 4);
  L.bc = o; o = align256(o + size_t(C > L.nc ? C : L.nc) * 4);
  L.kc_spe_in = ((B + 15) / 16) * 2;
  L.w1s = o; o = align256(o + size_t(4) * L.kc_spe_in * 256 * 16);
  L.wc16 = o; o = align256(o + size_t(L.conv_pos * 8 + 128) * L.nc * 16);
  L.wcq = o; o = align256(o + size_t(25) * L.nc * 128);
  L.total = o;
  return L;
}

}  // namespace cmlpl
