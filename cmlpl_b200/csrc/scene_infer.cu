// Full-scene inference (tools/hyper_tools.py:416-437 test_whole) without materialised
// patches.  Stages (one launch each, all on the caller's stream):
//   1. conv0_map     conv0 (1x1, models.py:102,132) once per scene pixel -> mirrored,
//                    halo-padded fp16 map F0pad[8 chunks][(rows+w-1)][(cols+w-1)][8 channels]; a pixel's patch
//                    is then a plain w x w window of this map (hyper_tools.py:35-55,226-243)
//   2. spectral_head relu(feat_spe(x)) (models.py:142-143) and its classifier columns
//   3. conv1_pool    conv1 + residual + ReLU once per scene position in 9 patch-border classes and the
//                    pooled maps as parity planes (conv1_scene_sm100.cu); conv2_scene: conv2 + residual +
//                    ReLU once per position in 25 classes, border classes pooled in its epilogue; pool2_cls: rest of
//                    the avg-pool + conv columns of the classifier -> 25 class-partial maps (conv2_scene_sm100.cu)
//   4. head          spectral columns of the classifier (models.py:150) + the pixel's 25 gathered conv
//                    partials + bias, argmax (hyper_tools.py:426, first index wins ties)
//   (<= 32 classes and <= 224 bands; otherwise the all-per-pixel patch_cnn_sm100.cu kernel + CUDA-core classify instead,
//   on both entry points; the raw entry point's CUDA-core spectral head reads the raw band, z-scored on load)
// With a validity mask (cmlpl_scene_infer_raw_masked) a no-data pixel stands in as its band means wherever it is read:
// conv0's loaders and the spectral branch's operands z-score it to 0 (so F0 there is the folded bias), and the heads label
// it CMLPL_NODATA_LABEL.  Everything between conv0 and the heads is unchanged.
#include "common.cuh"
#include "gemm_core.cuh"

namespace cmlpl {

// ------------------------------------------------------------------ conv0 map
// tcgen05 kernel of conv0_sm100.cu: plain fp16 operands for the 60-channel PCA cube (z-scored, well conditioned); for
// the RAW cube both operands are split into fp16 hi + lo parts (3 MMAs per K-step), because folding the PCA projection
// into conv0 makes the contraction ill-conditioned in fp16 -- the noise components of the PCA are differences of band
// values ~10x larger than the result (measured: with single fp16 operands the B = 200 raw parity test misses the 1e-3
// logit bar).  PCA projection, both z-scores and conv0 are per-pixel affine maps, so they fold into one
// F0 = Wf . (x - mu) + bf with Wf = W0 . (U/s)^T [64 x B] (SURVEY 8-f1).  Output: mirrored halo baked in, chunk-planar fp16
// [8 chunks][prow_n][pcol_n][8].
// bm: a band-major raw slab (BIL / BSQ), or nullptr for pixel-major; valid: the raw slab's validity mask, or nullptr
template <typename T, bool kVec4, bool kSplit>
int launch_conv0_tc(const T* in, int K, int scene_rows, int cols, int slab_row0, int w, int band_row0, int prow_n, int pcol_n,
                    const float* wt, const float* bias, const float* mu, const float* inv_sigma, __half* f0pad,
                    const BandMajor* bm, const uint8_t* valid, cudaStream_t s);

// x16_tile(_raw) + spectral_logits_kernel (head_sm100.cu): x is the f32 z-scored spectra (dtype -1) or the raw cube's
// rows (dtype = the sample type CMLPL_RAW_U16 / F32 / I16, z-scored with mu / inv_sigma in the conversion; band-major
// through bm, else pixel-major; valid: the band's validity mask, or nullptr)
int launch_spectral_logits(const void* x, int dtype, const BandMajor* bm, int64_t n, int num_features, int num_classes,
                           int w, const float* mu, const float* inv_sigma, const uint8_t* valid, const void* packed,
                           void* x16, float* part, cmlpl_stream_t stream);
// head_sum_kernel (head_sm100.cu) behind cmlpl_head_sum_lmap; valid: the band's validity mask, or nullptr
int launch_head_sum(const float* part, const float* lmap, int cols, int band_rows, int num_features, int num_classes, int w,
                    const void* packed, const uint8_t* valid, uint8_t* labels, float* logits, cmlpl_stream_t stream);

// ------------------------------------------------------------------ classifier + argmax
// one warp per pixel; lanes stride over the K = P*64 pooled features in 8-half chunks.  valid (u8 [n] or nullptr):
// no-data pixels are labelled CMLPL_NODATA_LABEL
template <int CMAX>
__global__ void __launch_bounds__(256)
classify_kernel(const __half* __restrict__ p2, const float* __restrict__ spe, const float* __restrict__ part,
                int64_t part_stride, int part_width, int64_t n, int K, int C,
                const float* __restrict__ wc, const float* __restrict__ bc, const uint8_t* __restrict__ valid,
                uint8_t* __restrict__ labels, float* __restrict__ logits) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = blockIdx.x * int64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = int64_t(gridDim.x) * (blockDim.x >> 5);
  const int chunks = K >> 3;
  for (int64_t p = warp; p < n; p += nwarps) {
    float acc[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) acc[c] = 0.f;
    const uint4* src = reinterpret_cast<const uint4*>(p2 + p * K);
    for (int ch = lane; ch < chunks; ch += 32) {
      const uint4 raw = __ldcs(src + ch);
      const __half2* h = reinterpret_cast<const __half2*>(&raw);
      float x[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(h[j]); x[2 * j] = f.x; x[2 * j + 1] = f.y; }
#pragma unroll
      for (int c = 0; c < CMAX; ++c) {
        if (c < C) {
          const float4 wa = __ldg(reinterpret_cast<const float4*>(wc + int64_t(c) * K + ch * 8));
          const float4 wb = __ldg(reinterpret_cast<const float4*>(wc + int64_t(c) * K + ch * 8 + 4));
          float s = acc[c];
          s = fmaf(x[0], wa.x, s); s = fmaf(x[1], wa.y, s); s = fmaf(x[2], wa.z, s); s = fmaf(x[3], wa.w, s);
          s = fmaf(x[4], wb.x, s); s = fmaf(x[5], wb.y, s); s = fmaf(x[6], wb.z, s); s = fmaf(x[7], wb.w, s);
          acc[c] = s;
        }
      }
    }
    float best = -INFINITY;
    int arg = 0;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < C) {
        float v = warp_sum(acc[c]);
        v += (spe ? spe[p * C + c] : 0.f) + bc[c];
        if (part)      // spectral_logits_kernel: four hidden-quarter partials f32 [4][part_stride][part_width]
          v += (part[p * part_width + c] + part[(part_stride + p) * part_width + c]) +
               (part[(2 * part_stride + p) * part_width + c] + part[(3 * part_stride + p) * part_width + c]);
        if (logits && lane == 0) logits[p * C + c] = v;
        if (v > best) { best = v; arg = c; }   // strict '>' : first index wins ties
      }
    }
    if (lane == 0) labels[p] = (valid && !valid[p]) ? uint8_t(CMLPL_NODATA_LABEL) : uint8_t(arg);
  }
}

// argmax over dense fp32 logits (batch-mode test_whole path, hyper_tools.py:426)
__global__ void argmax_kernel(const float* __restrict__ logits, int64_t n, int C, uint8_t* __restrict__ labels) {
  for (int64_t p = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; p < n; p += int64_t(gridDim.x) * blockDim.x) {
    float best = -INFINITY; int arg = 0;
    for (int c = 0; c < C; ++c) { const float v = logits[p * C + c]; if (v > best) { best = v; arg = c; } }
    labels[p] = uint8_t(arg);
  }
}

// Scene inference runs the tensor-core spectral branch (spectral_logits_kernel, head_sm100.cu) for <= 224 bands and <= 32
// classes: on the dense path, and in path mode 0 for <= 16 classes or from the raw cube; otherwise (beyond 224 bands on
// either entry point, and in path mode 0 at 17-32 classes on the cube entry point) the CUDA-core spectral_head +
// classify kernels below run (same C ABI, same results contract).
static bool tc_spectral_fits(int B, int C) { return C <= 32 && ((B + 15) / 16) * 2 <= 28; }   // <= 224 bands
// widest spectrum of the raw entry point (conv0_sm100.cu: the K-sliced kernel's resident weights)
constexpr int kRawMaxBands = 512;

// 1 (default): the exact-compute-sharing kernels where they apply; 0: the per-pixel tensor-core kernels everywhere (the
// independent implementation the tests compare against).  Per host thread; the workspace layout follows the mode.
static thread_local int g_scene_path_mode = 1;

struct SceneWs {
  size_t f0pad, p2, spe, hidden, x16, h16, pm, yq, lmap, total;
  int64_t chunk;
  bool tc, dense;
};
// tensor-core path: conv0 map, spectral tiles, partial spectral logits, pooled parity planes, the 9 half-pooled conv2
// maps, the 5 class-partial row maps.  CUDA-core path: conv0 map, per-pixel pooled features, spectral logits, hidden
// chunk.  Path mode 0 at 17-32 classes holds both spectral branches: the cube entry point runs the CUDA-core one, the raw
// entry point the tensor-core one.  Beyond 224 bands both entry points run the CUDA-core one.
static SceneWs scene_ws(int band_rows, int cols, int B, int C, int w) {
  SceneWs s;
  const int64_t n = int64_t(band_rows) * cols;
  const int64_t mtiles = (n + 127) / 128;
  const int P = ((w / 2) / 2) * ((w / 2) / 2);
  const int NC = class_width(C);
  const bool tc_fits = tc_spectral_fits(B, C);
  // the exact-compute-sharing kernels: w = 20 (9 / 25 border classes) and w = 11, whose 4 / 9 classes and 2x2 pooled cells
  // are a subset of them (conv1 rows 0..9 and conv2 rows 0..3 of an 11-window are top / mid class only)
  s.dense = tc_fits && (w == 20 || w == 11) && g_scene_path_mode == 1;
  s.tc = s.dense || (tc_fits && C <= 16);
  size_t o = 0;
  s.f0pad = o; o = align256(o + size_t(band_rows + w - 1) * (cols + w - 1) * 64 * 2);
  s.p2 = s.spe = s.hidden = s.x16 = s.h16 = s.pm = s.yq = s.lmap = 0;
  s.chunk = n < 16384 ? n : 16384;
  if (tc_fits) {
    s.x16 = o; o = align256(o + size_t(mtiles) * (((B + 15) / 16) * 2) * 2048);
    s.h16 = o; o = align256(o + size_t(4) * mtiles * 128 * NC * 4);   // partial spectral logits f32 [4 quarters][mtiles*128][NC]
  }
  if (s.dense) {
    const size_t qpos = size_t(4) * ((band_rows + w) / 2) * ((cols + w) / 2);     // positions of the 4 parity planes
    s.pm = o; o = align256(o + qpos * 9 * 64 * 2);         // pooled variants, f16 parity planes [9][4][8][PR2][PC2][8]
    s.yq = o; o = align256(o + qpos * 9 * 64 * 2);         // half-pooled conv2 maps, f16 [9][4][8][PR2][PC2][8]
    s.lmap = o; o = align256(o + qpos * 5 * NC * 4);       // class partials per pooled row, f32 [4][5][NC/4][PR2][PC2][4]
  } else {
    s.p2 = o; o = align256(o + size_t(n) * P * 64 * 2);     // per-pixel pooled conv features (patch_cnn_sm100.cu)
    if (!s.tc) {
      s.spe = o; o = align256(o + size_t(n) * C * 4);
      s.hidden = o; o = align256(o + size_t(s.chunk) * 1024 * 4);
    }
  }
  s.total = o;
  return s;
}

}  // namespace cmlpl

using namespace cmlpl;

extern "C" int cmlpl_set_scene_path_mode(int mode) {
  CMLPL_CHECK_ARG(mode == 0 || mode == 1, "set_scene_path_mode: 0 (per-pixel kernels) or 1 (exact compute sharing, default)");
  g_scene_path_mode = mode;
  return CMLPL_OK;
}

extern "C" size_t cmlpl_scene_workspace_bytes(int band_rows, int cols, int num_features, int num_classes, int w) {
  if (band_rows <= 0 || cols <= 0 || num_classes <= 0 || num_features <= 0 || w < 4) return 0;
  return scene_ws(band_rows, cols, num_features, num_classes, w).total;
}

extern "C" int cmlpl_scene_workspace_layout(int band_rows, int cols, int num_features, int num_classes, int w,
                                            size_t* offsets) {
  CMLPL_CHECK_ARG(offsets && band_rows > 0 && cols > 0 && num_classes > 0 && num_features > 0 && w >= 4,
                  "scene_workspace_layout: bad args");
  const SceneWs s = scene_ws(band_rows, cols, num_features, num_classes, w);
  // offset 3 (g, an empty region that keeps the 12 offsets in place) starts where pm does
  const size_t v[12] = {s.f0pad, s.x16, s.h16, s.pm, s.pm, s.yq, s.lmap, s.p2, s.spe, s.hidden, s.total, size_t(s.dense)};
  for (int i = 0; i < 12; ++i) offsets[i] = v[i];
  return CMLPL_OK;
}

// Where a scene call reads the scene from.  The two entry points differ only in their first two launches: conv0, and the
// spectral branch's conversion or the CUDA-core spectral head's A operand (z-scored spectra, or the raw band z-scored on
// load).
struct SceneSrc {
  const char* fn;                          // the entry point, named in the error messages
  bool from_raw;
  const float* cube;                       // cmlpl_scene_infer: the PCA cube slab and the band's z-scored spectra
  const float* spectra;
  const void* raw;                         // cmlpl_scene_infer_raw: the raw slab (dtype = sample | interleave) and the
  int dtype;                               // preprocessing folded into conv0 and into the spectral branch (include/cmlpl.h)
  const float *wf, *bf, *mu, *inv_sigma;
  bool masked;                             // cmlpl_scene_infer_raw_masked: the slab's validity mask u8 [slab_rows * cols]
  const uint8_t* valid;
};

// The conv0 map's conditions on the scene geometry (`fn` names the caller): the window fits the scene, the band lies
// inside it, and the slab holds every (mirrored) source row of the band's halo.  The halo holds the band's own rows,
// so the band's spectra, which the raw entry point reads from the slab, are inside the slab too.
static int check_band(const char* fn, int scene_rows, int cols, int slab_row0, int slab_rows, int w, int band_row0,
                      int band_rows) {
  CMLPL_CHECK_ARG(w / 2 <= scene_rows && w / 2 <= cols, "%s: window larger than the scene", fn);
  CMLPL_CHECK_ARG(band_row0 >= 0 && band_row0 + band_rows <= scene_rows, "%s: band outside the scene", fn);
  const int a = band_row0 + window_lo(w), b = band_row0 + band_rows - 1 + window_lo(w) + w - 1;
  int rmin = a < 0 ? 0 : a, rmax = b >= scene_rows ? scene_rows - 1 : b;
  if (a < 0 && -a - 1 > rmax) rmax = -a - 1;                          // rows -1..a reflect to 0..-a-1
  if (b >= scene_rows && 2 * scene_rows - 1 - b < rmin) rmin = 2 * scene_rows - 1 - b;
  CMLPL_CHECK_ARG(rmin >= slab_row0 && rmax < slab_row0 + slab_rows, "%s: slab rows [%d,%d) do not cover the band's halo [%d,%d]",
                  fn, slab_row0, slab_row0 + slab_rows, rmin, rmax);
  return CMLPL_OK;
}

// Every condition of a scene call, checked before it enqueues anything.  Pure host arithmetic without a CUDA call, so a
// rejected call leaves the caller's buffers and streams untouched.  *ws receives the workspace layout.
static int check_scene(const SceneSrc& src, int scene_rows, int cols, int slab_row0, int slab_rows, int B, int C, int w,
                       int band_row0, int band_rows, const void* packed, const void* workspace, size_t workspace_bytes,
                       const uint8_t* labels, SceneWs* ws) {
  const char* fn = src.fn;
  CMLPL_CHECK_ARG(packed && workspace && labels &&
                      (src.from_raw ? src.raw && src.wf && src.bf && src.mu && src.inv_sigma : src.cube && src.spectra),
                  "%s: null pointer", fn);
  CMLPL_CHECK_ARG(!src.masked || src.valid, "%s: null valid mask", fn);
  if (src.from_raw) {
    const int rc = check_raw_code(fn, "raw", src.raw, src.dtype);
    if (rc != CMLPL_OK) return rc;
  }
  // w = 20: the reference's BaseNet2 (classifier hard-wired to 2624 inputs, tools/models.py:127).  w = 11: the odd-window
  // variant BASELINE configs[4] names (ExtractPatches_for_base windows, hyper_tools.py:300-317; pooled 5 -> 2, classifier
  // over 64*2*2 + 1024 = 1280 inputs) -- a documented extension; its border classes and pooled cells are a subset of the
  // w = 20 ones, so the same scene-level kernels run (DESIGN 4.5); patch_cnn_kernel<11> per pixel behind path mode 0.
  CMLPL_CHECK_ARG(w == 20 || w == 11, "%s: w=%d unsupported (20, or 11 for the odd-window variant)", fn, w);
  CMLPL_CHECK_ARG(band_rows > 0 && cols > 0 && B > 0, "%s: bad dims (band_rows=%d cols=%d bands=%d)", fn, band_rows, cols, B);
  CMLPL_CHECK_ARG(C > 0 && C <= 32, "%s: needs 1..32 classes, got %d", fn, C);
  // the raw entry point: conv0 keeps the folded weights resident in shared memory as fp16 hi + lo, 128 KB at 512 bands
  CMLPL_CHECK_ARG(!src.from_raw || B <= kRawMaxBands, "%s: needs <= %d bands, got %d", fn, kRawMaxBands, B);
  const int rc = check_band(fn, scene_rows, cols, slab_row0, slab_rows, w, band_row0, band_rows);
  if (rc != CMLPL_OK) return rc;
  CMLPL_CHECK_ARG(src.from_raw || reinterpret_cast<uintptr_t>(src.cube) % 16 == 0, "%s: cube must be 16-byte aligned", fn);
  CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(packed) % 16 == 0, "%s: packed weights must be 16-byte aligned", fn);
  *ws = scene_ws(band_rows, cols, B, C, w);
  CMLPL_CHECK_ARG(workspace_bytes >= ws->total, "%s: workspace %zu < required %zu", fn, workspace_bytes, ws->total);
  CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 256 == 0, "%s: workspace must be 256-byte aligned", fn);
  return CMLPL_OK;
}

extern "C" int cmlpl_conv0_map_f16(const float* cube, int scene_rows, int cols, int slab_row0, int slab_rows, int w,
                                   int band_row0, int band_rows, const void* packed, void* f0pad,
                                   cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(cube && packed && f0pad, "conv0_map: null pointer");
  CMLPL_CHECK_ARG(scene_rows > 0 && cols > 0 && w >= 2 && band_rows > 0, "conv0_map: bad dims");
  const int rc = check_band("conv0_map", scene_rows, cols, slab_row0, slab_rows, w, band_row0, band_rows);
  if (rc != CMLPL_OK) return rc;
  CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(cube) % 16 == 0, "conv0_map: cube must be 16-byte aligned");
  const PackedLayout L = packed_layout(1, 1, w);  // w0/b0 offsets do not depend on B, C
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const int prow_n = band_rows + w - 1, pcol_n = cols + w - 1;
  return launch_conv0_tc<float, true, false>(cube, 60, scene_rows, cols, slab_row0, w, band_row0, prow_n, pcol_n,
                                      reinterpret_cast<const float*>(pk + L.w0), reinterpret_cast<const float*>(pk + L.b0), nullptr,
                                      nullptr, static_cast<__half*>(f0pad), nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

// CUDA-core spectral head of the per-pixel path: spe_logits f32 [n][C] = Wc_spe . relu(Wspe . x + bspe), over chunks of
// `chunk` pixels through the f32 scratch hidden [chunk][1024]
// `spectra` is StridedA over the z-scored f32 spectra, or RawZA / RawBandZA over the raw band (z-scored on load)
template <class FA> static FA rows_from(FA a, int64_t s0) { a.p += s0 * a.rs; return a; }          // pixel-major rows
template <typename T> static RawZA<T> rows_from(RawZA<T> a, int64_t s0) {
  a.p += s0 * a.rs;
  if (a.valid) a.valid += s0;
  return a;
}
template <typename T> static RawBandZA<T> rows_from(RawBandZA<T> a, int64_t s0) { a.m0 += s0; return a; }
template <class FA>
static int spectral_head(FA spectra, int64_t n, int num_features, int num_classes, int w, const void* packed,
                         float* hidden, int64_t chunk, float* spe_logits, cudaStream_t s) {
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const PackedLayout L = packed_layout(num_features, num_classes, w);
  const float* wspe = reinterpret_cast<const float*>(pk + L.wspe);
  const float* bspe = reinterpret_cast<const float*>(pk + L.bspe);
  const float* wc_spe = reinterpret_cast<const float*>(pk + L.wc_spe);
  for (int64_t s0 = 0; s0 < n; s0 += chunk) {
    const int m = int((n - s0) < chunk ? (n - s0) : chunk);
    // hidden = relu(X . Wspe^T + bspe)         (models.py:142-143)
    int rc = launch_gemm(m, 1024, num_features, 1, rows_from(spectra, s0),
                         StridedB{wspe, 1, num_features},
                         StridedC{hidden, 1024, 1, bspe, 1.f, 0.f, 1}, s, "spectral_hidden");
    if (rc != CMLPL_OK) return rc;
    // spe_logits = hidden . Wc_spe^T           (spectral columns of models.py:150)
    rc = launch_gemm(m, num_classes, 1024, 1, StridedA{hidden, 1024, 1}, StridedB{wc_spe, 1, 1024},
                     StridedC{spe_logits + s0 * num_classes, num_classes, 1, nullptr, 1.f, 0.f, 0}, s,
                     "spectral_logits");
    if (rc != CMLPL_OK) return rc;
  }
  return CMLPL_OK;
}

// classify_kernel over the per-pixel pooled features p2, adding the spectral logits spe_logits f32 [n][C] (CUDA-core
// head) or the tensor-core branch's four quarter partials `part`
static int classify_launch(const void* p2, const float* spe_logits, const float* part, int64_t part_stride, int64_t n,
                           int num_features, int num_classes, int w, const void* packed, const uint8_t* valid,
                           uint8_t* labels, float* logits, cudaStream_t s) {
  const int part_width = class_width(num_classes);        // row width of spectral_logits_kernel's partials
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  const PackedLayout L = packed_layout(num_features, num_classes, w);
  const int K = L.conv_pos * 64;
  const float* wc = reinterpret_cast<const float*>(pk + L.wc_conv);
  const float* bc = reinterpret_cast<const float*>(pk + L.bc);
  int64_t grid = (n + 7) / 8;
  const int64_t cap = int64_t(sm_count()) * 8;
  if (grid > cap) grid = cap;
  if (num_classes <= 16)
    classify_kernel<16><<<int(grid), 256, 0, s>>>(static_cast<const __half*>(p2), spe_logits, part, part_stride, part_width, n,
                                                  K, num_classes, wc, bc, valid, labels, logits);
  else
    classify_kernel<32><<<int(grid), 256, 0, s>>>(static_cast<const __half*>(p2), spe_logits, part, part_stride, part_width, n,
                                                  K, num_classes, wc, bc, valid, labels, logits);
  CMLPL_CHECK_LAUNCH("classify");
  return CMLPL_OK;
}

extern "C" int cmlpl_argmax_u8(const float* logits, int64_t n, int num_classes, uint8_t* labels, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(logits && labels && n >= 0 && num_classes > 0 && num_classes <= 255, "argmax: bad args");
  if (n == 0) return CMLPL_OK;
  int64_t grid = (n + 255) / 256;
  const int64_t cap = int64_t(sm_count()) * 8;
  if (grid > cap) grid = cap;
  argmax_kernel<<<int(grid), 256, 0, static_cast<cudaStream_t>(stream)>>>(logits, n, num_classes, labels);
  CMLPL_CHECK_LAUNCH("argmax");
  return CMLPL_OK;
}

// One scene call of either entry point: check_scene, then the path the workspace layout was sized for.
static int scene_infer(const SceneSrc& src, int scene_rows, int cols, int slab_row0, int slab_rows, int B, int C, int w,
                       int band_row0, int band_rows, const void* packed, void* workspace, size_t workspace_bytes,
                       uint8_t* labels, float* logits, cmlpl_stream_t stream) {
  SceneWs ws;
  int rc = check_scene(src, scene_rows, cols, slab_row0, slab_rows, B, C, w, band_row0, band_rows, packed, workspace,
                       workspace_bytes, labels, &ws);
  if (rc != CMLPL_OK) return rc;
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t n = int64_t(band_rows) * cols;
  float* part = reinterpret_cast<float*>(wsb + ws.h16);
  // the raw slab: sample type, and for BIL / BSQ its band-major strides (pixel-major BIP has row stride cols * B)
  const int sample = src.dtype & 0x0f, il = src.dtype & 0xf0;
  const BandMajor bmv = band_major(src.dtype, B, slab_rows, cols);
  const BandMajor* bm = src.from_raw && il != CMLPL_RAW_BIP ? &bmv : nullptr;
  // the spectral branch reads the band's z-scored spectra, or the band's rows of the raw slab: in every interleave they
  // start band_row0 - slab_row0 rows (of cols * B samples; of cols samples in every plane for BSQ) into the slab
  const int64_t row_stride = bm ? bm->rs : int64_t(cols) * B;
  const void* band_spectra =
      src.from_raw ? static_cast<const unsigned char*>(src.raw) + (band_row0 - slab_row0) * row_stride * raw_sample_bytes(src.dtype)
                   : static_cast<const void*>(src.spectra);
  // the band's validity: band pixel p is slab pixel (band_row0 - slab_row0) * cols + p
  const uint8_t* band_valid = src.valid ? src.valid + int64_t(band_row0 - slab_row0) * cols : nullptr;
  auto spectral_tc = [&](cudaStream_t st) {
    return launch_spectral_logits(band_spectra, src.from_raw ? sample : -1, bm, n, B, C, w, src.mu, src.inv_sigma, band_valid,
                                  packed, wsb + ws.x16, part, st);
  };
  auto conv0 = [&]() {
    if (!src.from_raw)
      return cmlpl_conv0_map_f16(src.cube, scene_rows, cols, slab_row0, slab_rows, w, band_row0, band_rows, packed,
                                 wsb + ws.f0pad, stream);
    const int prow_n = band_rows + w - 1, pcol_n = cols + w - 1;
    __half* f0 = reinterpret_cast<__half*>(wsb + ws.f0pad);
    if (sample == CMLPL_RAW_U16)
      return launch_conv0_tc<uint16_t, false, true>(static_cast<const uint16_t*>(src.raw), B, scene_rows, cols, slab_row0, w,
                                                    band_row0, prow_n, pcol_n, src.wf, src.bf, src.mu, src.inv_sigma, f0, bm, src.valid, s);
    if (sample == CMLPL_RAW_I16)
      return launch_conv0_tc<int16_t, false, true>(static_cast<const int16_t*>(src.raw), B, scene_rows, cols, slab_row0, w,
                                                   band_row0, prow_n, pcol_n, src.wf, src.bf, src.mu, src.inv_sigma, f0, bm, src.valid, s);
    return launch_conv0_tc<float, false, true>(static_cast<const float*>(src.raw), B, scene_rows, cols, slab_row0, w,
                                               band_row0, prow_n, pcol_n, src.wf, src.bf, src.mu, src.inv_sigma, f0, bm, src.valid, s);
  };
  if (ws.dense) {
    // The spectral branch (fp16 tiles of the spectra + the two spectral GEMMs) does not depend on the conv tower until
    // the head: forked onto the side stream, its conversion kernel shares the SMs with conv0 and its tail with the head
    // of conv1_pool.  Then conv1 (9 border classes) -> pooled parity planes -> conv2 (25 classes) -> pool + conv
    // classifier columns, and the head joins the branch: spectral partials + gathered conv partials + argmax.
    SideStream* sd = side_stream();
    CMLPL_CHECK_ARG(sd, "%s: cannot create the side stream", src.fn);
    std::lock_guard<std::mutex> lock(sd->mu);
    CMLPL_CUDA(cudaEventRecord(sd->fork[0], s));
    CMLPL_CUDA(cudaStreamWaitEvent(sd->s, sd->fork[0], 0));
    if ((rc = spectral_tc(sd->s)) != CMLPL_OK) return rc;
    CMLPL_CUDA(cudaEventRecord(sd->join[0], sd->s));
    if ((rc = conv0()) != CMLPL_OK) return rc;
    if ((rc = cmlpl_conv1_pool_planes_f16(wsb + ws.f0pad, cols, w, band_rows, packed, wsb + ws.pm, stream)) != CMLPL_OK) return rc;
    if ((rc = cmlpl_conv2_scene_f16(wsb + ws.pm, cols, w, band_rows, packed, wsb + ws.yq, stream)) != CMLPL_OK) return rc;
    float* lmap = reinterpret_cast<float*>(wsb + ws.lmap);
    if ((rc = cmlpl_pool2_cls_f16(wsb + ws.yq, cols, w, band_rows, B, C, packed, lmap, stream)) != CMLPL_OK) return rc;
    CMLPL_CUDA(cudaStreamWaitEvent(s, sd->join[0], 0));
    return launch_head_sum(part, lmap, cols, band_rows, B, C, w, packed, band_valid, labels, logits, stream);
  }
  // per pixel: the tensor-core spectral branch; or the CUDA-core spectral head beyond 224 bands (both entry points) and in
  // path mode 0 at 17-32 classes on the cube entry point, where the workspace holds both branches and the raw entry point
  // runs the tensor-core one
  if ((rc = conv0()) != CMLPL_OK) return rc;
  const bool tc = ws.tc || (src.from_raw && tc_spectral_fits(B, C));
  float* spe = reinterpret_cast<float*>(wsb + ws.spe);
  float* hidden = reinterpret_cast<float*>(wsb + ws.hidden);
  // the CUDA-core spectral head's A operand from the raw band: z-scored on load, pixel-major or band-major
  auto raw_head = [&](auto sample_type) {
    using T = decltype(sample_type);
    const T* x = static_cast<const T*>(band_spectra);
    return bm ? spectral_head(RawBandZA<T>{x, *bm, 0, src.mu, src.inv_sigma, band_valid, 0, false}, n, B, C, w, packed, hidden,
                              ws.chunk, spe, s)
              : spectral_head(RawZA<T>{x, B, src.mu, src.inv_sigma, band_valid, false}, n, B, C, w, packed, hidden, ws.chunk,
                              spe, s);
  };
  if (tc)
    rc = spectral_tc(s);
  else if (!src.from_raw)
    rc = spectral_head(StridedA{src.spectra, B, 1}, n, B, C, w, packed, hidden, ws.chunk, spe, s);
  else if (sample == CMLPL_RAW_U16)
    rc = raw_head(uint16_t{});
  else if (sample == CMLPL_RAW_I16)
    rc = raw_head(int16_t{});
  else
    rc = raw_head(float{});
  if (rc != CMLPL_OK) return rc;
  if ((rc = cmlpl_patch_cnn_f16(wsb + ws.f0pad, cols, w, band_rows, packed, wsb + ws.p2, stream)) != CMLPL_OK) return rc;
  return classify_launch(wsb + ws.p2, tc ? nullptr : spe, tc ? part : nullptr, ((n + 127) / 128) * 128, n, B, C, w, packed,
                         band_valid, labels, logits, s);
}

extern "C" int cmlpl_scene_infer(const float* cube, int scene_rows, int cols, int slab_row0, int slab_rows,
                                 const float* spectra, int num_features, int num_classes, int w, int band_row0,
                                 int band_rows, const void* packed, void* workspace, size_t workspace_bytes,
                                 uint8_t* labels, float* logits, cmlpl_stream_t stream) {
  const SceneSrc src{"scene_infer", false, cube, spectra};
  return scene_infer(src, scene_rows, cols, slab_row0, slab_rows, num_features, num_classes, w, band_row0, band_rows, packed,
                     workspace, workspace_bytes, labels, logits, stream);
}


// ---------------------------------------------------------------------------------------------
// Scene inference from the RAW cube (uint16 / float32 / int16; BIP, BIL or BSQ): the preprocessing of
// tools/hyper_tools.py:285-292 is folded into the first kernels (no PCA cube / z-scored spectra in HBM).
//   raw       raw scene rows slab_row0..  (dtype = sample | interleave, include/cmlpl.h: CMLPL_RAW_*)
//   wf f32 [B][64], bf f32 [64]    conv0 folded with the PCA projection and both z-scores
//   mu, inv_sigma f32 [B]          band means / 1/std (z-score of the spectral branch)
extern "C" int cmlpl_scene_infer_raw(const void* raw, int dtype, int scene_rows, int cols, int slab_row0, int slab_rows,
                                     int num_features, int num_classes, int w, int band_row0, int band_rows,
                                     const float* wf, const float* bf, const float* mu, const float* inv_sigma,
                                     const void* packed, void* workspace, size_t workspace_bytes, uint8_t* labels,
                                     float* logits, cmlpl_stream_t stream) {
  const SceneSrc src{"scene_infer_raw", true, nullptr, nullptr, raw, dtype, wf, bf, mu, inv_sigma};
  return scene_infer(src, scene_rows, cols, slab_row0, slab_rows, num_features, num_classes, w, band_row0, band_rows, packed,
                     workspace, workspace_bytes, labels, logits, stream);
}

// The same with a validity mask valid u8 [slab_rows * cols] (1 = valid, 0 = no-data) over the slab's pixels in raster
// order: a no-data pixel stands in as its band means wherever it is read (in its neighbours' windows, through the mirror
// too, and as its own spectral input), and its label is CMLPL_NODATA_LABEL.  Same workspace size and layout.
extern "C" int cmlpl_scene_infer_raw_masked(const void* raw, int dtype, int scene_rows, int cols, int slab_row0, int slab_rows,
                                            int num_features, int num_classes, int w, int band_row0, int band_rows,
                                            const float* wf, const float* bf, const float* mu, const float* inv_sigma,
                                            const uint8_t* valid, const void* packed, void* workspace,
                                            size_t workspace_bytes, uint8_t* labels, float* logits, cmlpl_stream_t stream) {
  const SceneSrc src{"scene_infer_raw_masked", true, nullptr, nullptr, raw, dtype, wf, bf, mu, inv_sigma, true, valid};
  return scene_infer(src, scene_rows, cols, slab_row0, slab_rows, num_features, num_classes, w, band_row0, band_rows, packed,
                     workspace, workspace_bytes, labels, logits, stream);
}
