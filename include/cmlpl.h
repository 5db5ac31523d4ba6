/*
 * cmlpl.h -- C ABI of libcmlpl_sm100.so: the B200 (sm_100a) kernels behind the CMLPL
 * hot path (patch gather -> BaseNet2 -> losses -> full-scene inference -> OA/AA/kappa).
 *
 * The reference (liuli33/CMLPL) has no FFI: its "API" is Python names.  Each entry
 * point below names the reference code it replaces (file:line under the reference
 * root); cmlpl_b200/ binds them with ctypes and re-exposes the reference's Python
 * names on top (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns every buffer; the library allocates nothing persistent;
 *   - all launches are asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = ok, <0 = error; cmlpl_last_error() gives the message
 *     (thread-local);
 *   - tensors are dense row-major with the shapes written in the comments.
 */
#ifndef CMLPL_H_
#define CMLPL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CMLPL_OK 0
#define CMLPL_ERR_ARG (-1)
#define CMLPL_ERR_CUDA (-2)
#define CMLPL_ERR_UNSUPPORTED (-3)

typedef void* cmlpl_stream_t;

int cmlpl_version(void);
const char* cmlpl_last_error(void);
/* 1 if the device the current context runs on is sm_100 (B200), else 0 (or <0). */
int cmlpl_device_ok(void);
/* cudaMemcpy2DAsync (kind cudaMemcpyDefault): `height` rows of `width_bytes`, `spitch` / `dpitch` bytes apart, e.g. one
 * row band of a host BSQ cube, B plane segments, into the same rows of a device slab. */
int cmlpl_memcpy2d_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes, size_t height,
                         cmlpl_stream_t stream);

/* ------------------------------------------------------------------ patches --
 * tools/hyper_tools.py:35-55 (MirrowCut), :226-243 (ExtractPatches, even w) and
 * :300-317 (ExtractPatches_for_base, odd w; odd_mode=1).
 * cube   f32 [slab_rows, cols, feat]   channels-last slab = scene rows
 *                                       [slab_row0, slab_row0+slab_rows) of a scene with
 *                                       scene_rows rows (band sharding; mirror padding is
 *                                       applied at true scene edges only)
 * idx    i64 [n] raster pixel indices r*cols+c, or NULL for first, first+1, ...
 * noise  f32 [n, feat, w, w] or NULL;  out = patch + noise*noise_scale (train.py:157)
 * out    f32 [n, feat, w, w]
 */
int cmlpl_patch_gather_f32(const float* cube, int scene_rows, int cols, int feat,
                           int slab_row0, int slab_rows, int w, int odd_mode,
                           const int64_t* idx, int64_t first, int64_t n,
                           const float* noise, float noise_scale,
                           float* out, cmlpl_stream_t stream);

/* ------------------------------------------------------------ fp32 building --
 * Dense fp32 building blocks of BaseNet2 (tools/models.py:97-152) in batch mode,
 * NCHW like the reference; used by training forward/backward (a5, a12).
 */

/* C[M,N] = act( alpha * op(A)[M,K] . op(B)[K,N] + bias[N] + beta*C ) with arbitrary
 * element strides (so any transpose is a stride choice).  act: 0 none, 1 relu.
 * nn.Linear forward / dgrad / wgrad (models.py:142,150). */
int cmlpl_sgemm_f32(int M, int N, int K, float alpha,
                    const float* A, int64_t a_rs, int64_t a_cs,
                    const float* B, int64_t b_rs, int64_t b_cs,
                    const float* bias, float beta,
                    float* C, int64_t c_rs, int64_t c_cs, int act,
                    cmlpl_stream_t stream);

/* y[b,co,h,w] = act( conv_kxk(x, wgt, pad=k/2) + bias + (res ? res : 0) ), k in {1,3}.
 * models.py:132-135,138-139.   x f32 [b,ci,h,w], wgt f32 [co,ci,k,k], res/y f32 [b,co,h,w].
 * transpose_w=1 computes the data gradient: uses wgt[ci_out... ] flipped/transposed, i.e.
 * y = conv(x, flip(wgt)^T) with x = dL/dy [b,co,h,w] -> y = dL/dx [b,ci,h,w]. */
int cmlpl_conv2d_f32(const float* x, const float* wgt, const float* bias, const float* res,
                     float* y, int b, int ci, int co, int h, int w, int k, int act,
                     int transpose_w, cmlpl_stream_t stream);

/* dW[co,ci,k,k] = sum_{b,y,x} dy[b,co,y,x] * x[b,ci,y+ky-p,x+kx-p];  db[co] = sum dy. */
int cmlpl_conv2d_wgrad_f32(const float* x, const float* dy, float* dw, float* db,
                           int b, int ci, int co, int h, int w, int k, cmlpl_stream_t stream);

/* 2x2/2 average pool forward / backward (models.py:136,140), NCHW. */
int cmlpl_avgpool2_f32(const float* x, float* y, int64_t planes, int h, int w, cmlpl_stream_t stream);
int cmlpl_avgpool2_bwd_f32(const float* dy, float* dx, int64_t planes, int h, int w, cmlpl_stream_t stream);

/* relu backward with optional residual fan-out: dx = dy * (y > 0). */
int cmlpl_relu_bwd_f32(const float* y, const float* dy, float* dx, int64_t n, cmlpl_stream_t stream);
/* column sums: out[n] = sum_m x[m,n] (bias gradients of nn.Linear). */
int cmlpl_colsum_f32(const float* x, float* out, int64_t m, int64_t n, cmlpl_stream_t stream);

/* Row L2 normalisation: y = x / max(norm, eps), norm = sqrt(sum x^2) per row (stored unclamped), and its backward
 * dx = (dy - y * sum(dy*y)) / norm, or dy / eps where norm < eps.  eps = 0 is models.py:87-90 Normalize (no epsilon:
 * a zero row gives NaN); eps = 1e-12 is F.normalize (models.py:23-24, ContrastiveLoss). */
int cmlpl_l2norm_f32(const float* x, float* y, float* norm, int64_t rows, int64_t cols, float eps,
                     cmlpl_stream_t stream);
int cmlpl_l2norm_bwd_f32(const float* y, const float* norm, const float* dy, float* dx,
                         int64_t rows, int64_t cols, float eps, cmlpl_stream_t stream);

/* ------------------------------------------------------------ scene inference --
 * tools/hyper_tools.py:416-437 (test_whole) over a whole scene / row band without ever
 * materialising patches: conv0 is evaluated once per scene pixel into a mirrored,
 * halo-padded fp16 map; conv1 (+residual, ReLU, 2x2 avg-pool), conv2 and the pool + conv columns of
 * the classifier are evaluated ONCE PER SCENE POSITION in the 9 / 25 classes of how a patch border can
 * cut them (exact compute sharing; persistent tcgen05 kernels fed by TMA tile loads); the spectral
 * branch is one fused two-GEMM kernel; a sum head adds each pixel's 25 gathered conv partials to its
 * spectral partials and takes the argmax.  This path takes up to 32 classes (class width 16 up to 16 classes, 32
 * beyond) and up to 224 bands.  The per-pixel path (patch_cnn_kernel: conv1 + conv2 per patch window staged in shared
 * memory, then the classifier heads) is the independent implementation selected by cmlpl_set_scene_path_mode(0); it
 * also serves > 224 bands on both entry points, with the CUDA-core spectral head (cmlpl_scene_infer_raw reads it from
 * the raw band, z-scored on load).  cmlpl_scene_infer / cmlpl_scene_infer_raw refuse more than 32 classes, and
 * cmlpl_scene_infer_raw more than 512 bands.
 *
 * Packed weights: cmlpl_pack_basenet2() converts the reference state_dict tensors
 * (models.py:102-127: conv0/1/2.{weight,bias}, feat_spe.*, classifier.*) into the
 * kernel layouts inside a caller-owned buffer of cmlpl_packed_bytes() bytes.
 */
size_t cmlpl_packed_bytes(int num_features, int num_classes, int w);
int cmlpl_pack_basenet2(const float* conv0_w, const float* conv0_b,
                        const float* conv1_w, const float* conv1_b,
                        const float* conv2_w, const float* conv2_b,
                        const float* spe_w, const float* spe_b,
                        const float* cls_w, const float* cls_b,
                        int num_features, int num_classes, int w,
                        void* packed, cmlpl_stream_t stream);

/* Which kernels cmlpl_scene_infer / cmlpl_scene_infer_raw run on the tensor-core path (<= 32 classes, <= 224 bands), per
 * calling host thread: 1 (default) = the scene-level kernels with exact compute sharing (w = 20 and w = 11), 0 = the
 * per-pixel kernels (patch_cnn_kernel<w> per pixel; the independent implementation the tests compare the default against,
 * models.py:133-150 per patch; at 17-32 classes with the CUDA-core heads, the raw entry point with the tensor-core
 * spectral branch).  The workspace size and layout follow the mode: set it before sizing the workspace. */
int cmlpl_set_scene_path_mode(int mode);

/* Workspace needed to infer `band_rows` rows of a scene with `cols` columns. */
size_t cmlpl_scene_workspace_bytes(int band_rows, int cols, int num_features, int num_classes, int w);

/* Byte offsets of the workspace regions (for stage-level profiling): offsets[12] =
 * {f0pad, x16, h16 (partial spectral logits f32 [4][ceil(n/128)*128][NC], NC = 16 for <= 16 classes, 32 for 17-32),
 *  g (unused, zero-sized),
 *  pmq, yq, lmap, p2, spe_logits, hidden, total, uses_tensor_core_path}. */
int cmlpl_scene_workspace_layout(int band_rows, int cols, int num_features, int num_classes, int w,
                                 size_t* offsets);

/* cube     f32 [slab_rows, cols, 60]  PCA cube slab (rows slab_row0.. of the scene)
 * spectra  f32 [band_rows*cols, num_features]   rows of X for the band's pixels
 * labels   u8  [band_rows*cols]  argmax (first index on ties, hyper_tools.py:426)
 * logits   f32 [band_rows*cols, num_classes] or NULL
 * Band = scene rows [band_row0, band_row0+band_rows). */
int cmlpl_scene_infer(const float* cube, int scene_rows, int cols, int slab_row0, int slab_rows,
                      const float* spectra, int num_features, int num_classes, int w,
                      int band_row0, int band_rows, const void* packed,
                      void* workspace, size_t workspace_bytes,
                      uint8_t* labels, float* logits, cmlpl_stream_t stream);

/* Raw cube codes: dtype = sample | interleave.  Codes 0 and 1 are uint16 and float32 band-interleaved-by-pixel. */
#define CMLPL_RAW_U16 0x00    /* sample types */
#define CMLPL_RAW_F32 0x01
#define CMLPL_RAW_I16 0x02
#define CMLPL_RAW_BIP 0x00    /* interleave: band-interleaved-by-pixel, by line, band-sequential */
#define CMLPL_RAW_BIL 0x10
#define CMLPL_RAW_BSQ 0x20

/* The same from the RAW cube (dtype = CMLPL_RAW_{U16,F32,I16} | CMLPL_RAW_{BIP,BIL,BSQ}; <= 32 classes, <= 512
 * bands): the PCA projection and both z-scores of tools/hyper_tools.py:285-292 are folded into conv0
 * (wf f32 [B][64] = (W0 . (U/s)^T)^T, bf f32 [64] = b0 - W0 . m/s) and into the spectral branch (mu, inv_sigma
 * f32 [B]: the fp16 conversion of the tensor-core branch up to 224 bands, the operand loads of the CUDA-core spectral
 * head beyond); neither the PCA cube nor the z-scored spectra touch HBM.  Above 256 bands conv0 streams each tile's
 * bands through shared memory in 64-band slices.
 * raw holds scene rows slab_row0.. (halo included, like `cube` above), aligned to its sample size.  With
 * sr = scene row - slab_row0, c = column, b = band, the sample is at
 *   BIP  raw[(sr*cols + c)*B + b]          ([slab_rows*cols, B], a pixel's bands contiguous)
 *   BIL  raw[(sr*B + b)*cols + c]          ([slab_rows, B, cols], AVIRIS-NG, Hyperion, PRISMA)
 *   BSQ  raw[(b*slab_rows + sr)*cols + c]  ([B, slab_rows, cols]: the planes are the slab's, not the scene's)
 * The band's spectra are read from the same slab.  Results do not depend on the interleave. */
int cmlpl_scene_infer_raw(const void* raw, int dtype, int scene_rows, int cols, int slab_row0, int slab_rows,
                          int num_features, int num_classes, int w, int band_row0, int band_rows,
                          const float* wf, const float* bf, const float* mu, const float* inv_sigma,
                          const void* packed, void* workspace, size_t workspace_bytes,
                          uint8_t* labels, float* logits, cmlpl_stream_t stream);

/* No-data pixels of raw sensor cubes (swath edges, dropped scan lines, masked detectors).
 *   missing sample  equal to the fill value, compared in the sample type; a float32 sample that is not finite is
 *                   always missing
 *   no-data pixel   a pixel with ANY band missing (every pixel is used whole or imputed whole)
 *   validity mask   u8 [rows, cols] in raster order over the raw slab's rows, whatever the interleave: 1 = valid,
 *                   0 = no-data.  Any mask of this layout works in its place (a cloud or water mask).
 *   imputation      a no-data pixel stands in as its band-mean spectrum x = mu wherever it is read: in every
 *                   neighbour's window (through the mirror at scene edges too), as its own spectral input (z-scored
 *                   spectrum 0), and in cmlpl_preprocess_apply_masked's outputs (spectra row 0, PCA row -shift).  Its
 *                   label is CMLPL_NODATA_LABEL; its logits, when requested, are those of the imputed pixel.
 * At most 32 classes, so CMLPL_NODATA_LABEL is never a class and cmlpl_confusion_i64 never counts it. */
#define CMLPL_NODATA_LABEL 255

/* Validity mask of a raw cube of `rows` x `cols` pixels (any CMLPL_RAW_* code; BIP rows may be pixels with cols = 1,
 * BSQ planes hold `rows` rows) in one read of the cube: valid u8 [rows*cols], *n_valid i64 = its number of valid
 * pixels, band_missing i64 [B] (or NULL) = the number of pixels in which band b is missing, e.g. a band that is fill
 * everywhere.  `fill` must be a value of the sample type (CMLPL_ERR_ARG otherwise, e.g. -9999 for uint16, 0.5 for
 * int16); for float32, fill = NaN marks the non-finite samples only.  At most 8192 bands. */
int cmlpl_valid_mask_u8(const void* raw, int dtype, int64_t rows, int cols, int B, double fill, uint8_t* valid,
                        int64_t* n_valid, int64_t* band_missing, cmlpl_stream_t stream);

/* cmlpl_scene_infer_raw with the slab's validity mask valid u8 [slab_rows*cols] (cmlpl_valid_mask_u8, or the caller's):
 * no-data pixels are imputed as above and labelled CMLPL_NODATA_LABEL.  conv0's loaders and the spectral branch's
 * operands read the mask; a pixel whose window (after mirroring) holds no no-data pixel gets exactly the logits of
 * cmlpl_scene_infer_raw.  Same workspace, checks before anything is enqueued (a NULL valid included). */
int cmlpl_scene_infer_raw_masked(const void* raw, int dtype, int scene_rows, int cols, int slab_row0, int slab_rows,
                                 int num_features, int num_classes, int w, int band_row0, int band_rows,
                                 const float* wf, const float* bf, const float* mu, const float* inv_sigma,
                                 const uint8_t* valid, const void* packed, void* workspace, size_t workspace_bytes,
                                 uint8_t* labels, float* logits, cmlpl_stream_t stream);

/* Individual stages of cmlpl_scene_infer (exposed for tests / profiling). */
int cmlpl_conv0_map_f16(const float* cube, int scene_rows, int cols, int slab_row0, int slab_rows,
                        int w, int band_row0, int band_rows, const void* packed,
                        void* f0pad /* f16 [8, band_rows+w-1, cols+w-1, 8]: chunk-planar (8 channels per 16-B chunk) */, cmlpl_stream_t stream);
int cmlpl_patch_cnn_f16(const void* f0pad, int cols, int w, int band_rows, const void* packed,
                        void* p2 /* f16 [band_rows*cols, (w/4)^2, 64] */, cmlpl_stream_t stream);
/* Dense (scene-level) conv tower, exact compute sharing of conv1 / conv2 / pools / classifier (SURVEY section 7;
 * tools/models.py:133-150 for all patches at once; csrc/conv1_scene_sm100.cu, csrc/conv2_scene_sm100.cu).
 * PR = band_rows+w-1, PC = cols+w-1, PR2 = (band_rows+w)/2, PC2 = (cols+w)/2; "planes" = the 4 parity planes
 * (pr&1)*2+(pc&1) of the padded map, y' = pr>>1, x' = pc>>1.
 *   cmlpl_conv1_pool_planes_f16   : conv1 + bias + residual + ReLU once per position of the conv0 map f0pad
 *                                   f16 [8][PR][PC][8] in 3x3 = 9 patch-border classes, and their 2x2 average pools for
 *                                   every top-left position in the 9 pooled border classes, in ONE kernel (no fp32
 *                                   scratch in HBM):  pmq f16 [9 = A*3+B][4][8 chunks][PR2][PC2][8] (A,B in top/mid/bot,
 *                                   left/mid/right; entries without a pooled cell are 0; w = 11 stores A,B in top/mid)
 *   cmlpl_conv2_scene_f16         : conv2+bias+residual+ReLU in 25 border classes (rho, kap in {i=0, 1, 2..7, 8, 9}); the
 *                                   border halves of the 2x2 pool (rho 0 + rho 1 one row down, rho 3 + rho 4, same for
 *                                   kap) are averaged in the epilogue:  yq f16 [9 = Al*3+Be][4][8][PR2][PC2][8],
 *                                   yq[Al][Be][y',x'] = mean over the border partners of Y[rho][kap][y'+u, x'+v]
 *   cmlpl_pool2_cls_f16           : rest of the 2x2 avg-pool (middle classes) + conv columns of the classifier per
 *                                   pooled cell (I,J), summed over the pooled columns J of a pooled row I:
 *                                   lmap f32 [4][5 = I][NC/4 class quads][PR2][PC2][4] (NC = 16 up to 16 classes, 32 for
 *                                   17-32),
 *                                   lmap[I][y',x'] = sum_J L[I][J][y', x'+2J] */
int cmlpl_conv1_pool_planes_f16(const void* f0pad, int cols, int w, int band_rows, const void* packed, void* pmq,
                                cmlpl_stream_t stream);
int cmlpl_conv2_scene_f16(const void* pmq, int cols, int w, int band_rows, const void* packed, void* yq,
                          cmlpl_stream_t stream);
int cmlpl_pool2_cls_f16(const void* yq, int cols, int w, int band_rows, int num_features, int num_classes,
                        const void* packed, float* lmap, cmlpl_stream_t stream);
/* Fused spectral branch + sum head:
 *   cmlpl_spectral_logits_tc     : part f32 [4 hidden quarters][ceil(n/128)*128][NC] = Wc_spe . relu(Wspe . x + b) per
 *                                  quarter of the 1024 hidden features (tools/models.py:142-143,150), <= 32 classes
 *                                  (NC = 16 up to 16 classes, 32 for 17-32), as many bands as the kernel's input tiles
 *                                  fit shared memory for (cmlpl_scene_infer uses it up to 224)
 *   cmlpl_head_sum_lmap          : 4 quarter partials + the 5 gathered conv partials + bias, argmax */
int cmlpl_spectral_logits_tc(const float* spectra, int64_t n, int num_features, int num_classes, int w,
                             const void* packed, void* x16, float* part, cmlpl_stream_t stream);
int cmlpl_head_sum_lmap(const float* part, const float* lmap, int cols, int band_rows, int num_features,
                        int num_classes, int w, const void* packed, uint8_t* labels, float* logits,
                        cmlpl_stream_t stream);
/* hyper_tools.py:426 torch.max(outputs, 1): first index on ties.  logits f32 [n, C] -> u8 [n]. */
int cmlpl_argmax_u8(const float* logits, int64_t n, int num_classes, uint8_t* labels,
                    cmlpl_stream_t stream);

/* ------------------------------------------------------------- preprocessing --
 * tools/hyper_tools.py:8-32 (featureNormalize, PCANorm) as called at :289-292, on device (SURVEY 8-f1).
 * x: raw scene [n, B] band-interleaved-by-pixel, dtype CMLPL_RAW_U16 / F32 / I16.
 * fit  : mean f64 [B] = column means, gram f64 [B,B] = sum_n (x-mean)(x-mean)^T, upper 32x32 tiles only
 *        (mirror on the host; np.cov = gram/(n-1), np.std^2 = diag(gram)/n).  The B x B SVD stays on the host.
 *        cmlpl_preprocess_fit_cube_f64 takes a [rows, cols] cube in any raw code of cmlpl_scene_infer_raw (BIL needs
 *        cols); cmlpl_preprocess_fit_f64 is the same for BIP [n, B] (rows = n, cols = 1).
 * apply: spectra f32 [n,B] = (x-mu)*inv_sigma (may be NULL);  cube f32 [n,npc] = (x-mu).Us - shift with
 *        Us f32 [B,npc] = U[:, :npc]/s and shift = m/s (m, s = mean/std of the projected data). */
int cmlpl_preprocess_fit_cube_f64(const void* x, int dtype, int rows, int cols, int B, double* mean, double* gram,
                                  cmlpl_stream_t stream);
int cmlpl_preprocess_fit_f64(const void* x, int dtype, int64_t n, int B, double* mean, double* gram,
                             cmlpl_stream_t stream);
/* The fit over the valid pixels only (valid u8 [rows*cols], cmlpl_valid_mask_u8): mean and Gram sum over the pixels
 * with a nonzero byte, *n_valid i64 (device) = their number; np.cov = gram/(n_valid-1), sigma^2 = diag(gram)/n_valid.
 * Any raw code, as cmlpl_preprocess_fit_cube_f64 (BIP: rows = pixels and cols = 1 works too). */
int cmlpl_preprocess_fit_masked_f64(const void* raw, int dtype, int64_t rows, int cols, int B, const uint8_t* valid,
                                    double* mean, double* gram, int64_t* n_valid, cmlpl_stream_t stream);
int cmlpl_preprocess_apply(const void* x, int dtype, int64_t n, int B, int npc, const float* mu,
                           const float* inv_sigma, const float* Us, const float* shift, float* cube,
                           float* spectra, cmlpl_stream_t stream);
/* apply with valid u8 [n]: a no-data pixel is written as its band means, spectra row 0 and cube row -shift. BIP only. */
int cmlpl_preprocess_apply_masked(const void* x, int dtype, int64_t n, int B, int npc, const float* mu,
                                  const float* inv_sigma, const float* Us, const float* shift, const uint8_t* valid,
                                  float* cube, float* spectra, cmlpl_stream_t stream);

/* ------------------------------------------------------------------ metrics --
 * tools/hyper_tools.py:208-223 (CalAccuracy): integer confusion matrix
 * cm[label, pred] += 1 for pairs with both in [0, C).  pred u8 [n], label i64 [n],
 * cm i64 [C, C] (accumulated into; zero it first).  OA/AA/kappa are float64 host
 * arithmetic on these counts. */
int cmlpl_confusion_i64(const uint8_t* pred, const int64_t* label, int64_t n, int num_classes,
                        int64_t* cm, cmlpl_stream_t stream);

/* ------------------------------------------------------------------- losses --
 * train.py:191-265 and tools/models.py:14-39.  All fp32, rows = samples; `loss` is a device
 * scalar that is ACCUMULATED into (zero it first).
 */
/* Hard-label CE (train.py:191-192) or soft/masked CE (train.py:239-242):
 *   loss_i = -sum_c log_softmax(z_i)_c * t_ic * m_i ;  *loss += scale * mean_i loss_i
 *   dz_ic  = scale/rows * m_i * (softmax(z_i)_c * sum_c t_ic - t_ic)
 * labels i64 [rows] (hard) XOR probs f32 [rows, C] (soft); mask f32 [rows] or NULL; dlogits may be NULL. */
int cmlpl_ce_fwd_bwd_f32(const float* logits, const int64_t* labels, const float* probs,
                         const float* mask, int64_t rows, int C, float scale,
                         float* loss, float* dlogits, cmlpl_stream_t stream);

/* S = A . B^T with A f32 [M, K], B f32 [N, K] (K contiguous, K % 64 == 0) on tcgen05: operands rounded to fp16, fp32
 * accumulation; C f32 [M, N].  The similarity matrices of train.py:213,246 and tools/models.py:27.
 * cmlpl_set_loss_gemm_mode(1) makes cmlpl_bank_smooth_f32 / cmlpl_graph_contrast_f32 / cmlpl_ntxent_f32 use it for
 * their similarity GEMM (default 0: fp32 CUDA-core tiles, the 1e-5 parity path).  The setting is per host thread. */
int cmlpl_sim_nt_tc_f32(const float* A, const float* B, int M, int N, int K, float* C, cmlpl_stream_t stream);
int cmlpl_set_loss_gemm_mode(int mode);

/* trian_CCT.py:76-84 softmax_js_loss: *loss += scale * 0.5 * (kl_div(log_softmax(z), M, 'mean') +
 * kl_div(log(t + 1e-5), M, 'mean')) with M = (softmax(z) + t)/2 and 'mean' over all rows*C elements;
 * dlogits (may be NULL) = scale * dL/dz, targets are constants.  logits, targets f32 [rows, C]. */
int cmlpl_softmax_js_f32(const float* logits, const float* targets, int64_t rows, int C, float scale,
                         float* loss, float* dlogits, cmlpl_stream_t stream);

/* loss_helper.py:247-248: entropy_i = -sum_c p_ic log(p_ic + eps), p = softmax(logits_i).  f32 [rows]. */
int cmlpl_softmax_entropy_f32(const float* logits, int64_t rows, int C, float eps, float* entropy,
                              cmlpl_stream_t stream);

/* train.py:203,213-215,220-222: probs_orig = softmax(logits); if smooth: A = exp(feats.Q^T/T)
 * row-normalised, probs = alpha*probs_orig + (1-alpha)*A.Qp; mask = max(probs) >= thr.
 * feats f32 [rows, dim], queue_feats f32 [queue, dim], queue_probs f32 [queue, C],
 * work f32 [rows, queue] scratch (only when smooth).  probs_orig may be NULL. */
int cmlpl_bank_smooth_f32(const float* logits, const float* feats, const float* queue_feats,
                          const float* queue_probs, int64_t rows, int C, int dim, int64_t queue,
                          float alpha, float T, int smooth, float thr, float* work,
                          float* probs_orig, float* probs, float* mask, cmlpl_stream_t stream);

/* train.py:246-265: pseudo-label-graph contrastive loss, forward + gradient.
 * f_row, f_col f32 [n, dim]; p1 (rows), p (cols) f32 [n, C].
 *   L = mean_i( -sum_j log(sp_ij) Q_ij + sum_j log(sp_ij + 1) Qn_ij ),  sp = row-softmax(f_row.f_col^T / T)
 * grad_side 0 -> dfeat = scale*dL/df_row (loss_contrast, :260-262); 1 -> scale*dL/df_col (loss_contrast1,
 * :263-265).  work f32 [3*n*n] scratch.  *loss += scale*L.  dfeat f32 [n, dim] may be NULL. */
int cmlpl_graph_contrast_f32(const float* f_row, const float* f_col, const float* p1, const float* p,
                             int64_t n, int dim, int C, float T, int grad_side, float scale,
                             float* work, float* loss, float* dfeat, cmlpl_stream_t stream);

/* tools/models.py:22-39 ContrastiveLoss (NT-Xent) on z = [normalize(emb_i); normalize(emb_j)]
 * f32 [2*bs, dim] (unit rows; use cmlpl_l2norm_f32 / _bwd around it).  *loss += L;
 * dz f32 [2*bs, dim] = dL/dz or NULL.  work f32 [2*(2bs)^2] scratch. */
int cmlpl_ntxent_f32(const float* z, int64_t bs, int dim, float T, float* work, float* loss,
                     float* dz, cmlpl_stream_t stream);

/* torch.optim.Adam (train.py:131-132,268,272; default betas/eps) over a list of tensors, one launch
 * per 16 tensors.  *_host are HOST arrays of n_tensors device pointers / element counts; step is the
 * 1-based step count.  Tensors whose grad pointer is NULL are skipped (grad=None). */
int cmlpl_adam_multi_f32(int n_tensors, float* const* p_host, const float* const* g_host,
                         float* const* m_host, float* const* v_host, const int64_t* numel_host,
                         float lr, float beta1, float beta2, float eps, int step,
                         cmlpl_stream_t stream);


/* ------------------------------------------------------------- collectives --
 * The two exchanges at the end of a row-band sharded scene inference (SURVEY 8e), for hosts that do not bring their
 * own process group (the Python layer of this repo uses torch.distributed): NCCL over NVLink, one communicator per
 * process / device, resolved at run time from libnccl.so.2.
 *   cmlpl_comm_unique_id        rank 0 fills id128 (128 bytes), the host hands it to the other ranks
 *   cmlpl_comm_init             collective over all ranks; *out is owned by the caller until cmlpl_comm_destroy
 *   cmlpl_comm_allgather_labels out u8 [world * per_rank] <- every rank's local u8 [per_rank] (bands padded to the
 *                               common height, hyper_tools.py:426-431 label map in raster order)
 *   cmlpl_comm_allreduce_confusion  cm i64 [count] summed in place (hyper_tools.py:208-223 counts) */
typedef struct cmlpl_comm cmlpl_comm;
int cmlpl_comm_unique_id(void* id128);
int cmlpl_comm_init(int rank, int world, const void* id128, cmlpl_comm** out);
int cmlpl_comm_allgather_labels(cmlpl_comm* comm, const uint8_t* local, int64_t per_rank, uint8_t* out,
                                cmlpl_stream_t stream);
int cmlpl_comm_allreduce_confusion(cmlpl_comm* comm, int64_t* cm, int count, cmlpl_stream_t stream);
int cmlpl_comm_destroy(cmlpl_comm* comm);

/* ------------------------------------------------------- fused training step --
 * One mutual-learning step of train.py:150-272 for BOTH BaseNet2 peers as 15 kernel launches (+ memsets of the gradient
 * block) on `stream`
 * (CUDA-graph capturable: every per-step scalar lives in the device-side cmlpl_train_params block).
 * Contractions run on tcgen05 (fp16 operands = TF32's 11-bit significand, fp32 accumulate in TMEM): conv0 / conv1 /
 * conv2 forward (tools/models.py:132-140), their data gradients and weight gradients (train.py:267,271); gradient
 * operands are scaled by a power of two chosen on device from max|dL/dcat| so they sit in fp16's normal range.
 * Bar: |d| <= 1e-3 * max|ref| against the fp32 path (cmlpl_conv2d_f32 & co. stay the 1e-5 reference).
 *
 * Row order inside a net: [bs labelled ; btu unlabelled] (train.py:174,184); nb = bs + btu.
 * Tensor index order in cmlpl_train_net arrays: 0 conv0.weight [64,60,1,1], 1 conv0.bias, 2 conv1.weight
 * [64,64,3,3], 3 conv1.bias, 4 conv2.weight, 5 conv2.bias, 6 feat_spe.weight [1024,B], 7 feat_spe.bias,
 * 8 classifier.weight [C,cat], 9 classifier.bias (state-dict layouts, tools/models.py:102-127).
 * Window w = 20 (the reference's BaseNet2, cat = 64*5*5 + 1024 = 2624) or w = 11 (ExtractPatches_for_base windows,
 * hyper_tools.py:300-317; both 2x2 pools floor, 11 -> 5 -> 2, so cat = 64*2*2 + 1024 = 1280).
 */
#define CMLPL_TRAIN_TENSORS 10
typedef struct cmlpl_train_net {
  float* p[CMLPL_TRAIN_TENSORS];   /* parameters, updated in place by the Adam phase */
  float* g[CMLPL_TRAIN_TENSORS];   /* gradients of total_loss (train.py:266/270), overwritten every step */
  float* m[CMLPL_TRAIN_TENSORS];   /* Adam exp_avg */
  float* v[CMLPL_TRAIN_TENSORS];   /* Adam exp_avg_sq */
  float* queue_feats;              /* f32 [queue, 1024]  memory bank this net's targets are smoothed with (train.py:138-145) */
  float* queue_probs;              /* f32 [queue, C] */
} cmlpl_train_net;

typedef struct cmlpl_train_params {   /* lives in DEVICE memory; the host refreshes it before every step */
  float noise_scale;      /* train.py:157 args.noise (ignored for inputs passed with cube == NULL) */
  float dropout_p;        /* tools/models.py:147; used only when drop_mask == NULL */
  float temperature;      /* train.py:213,246 */
  float alpha;            /* train.py:215 */
  float adap_thr;         /* args.thr * exp(-0.5 (epoch/num_epochs)^2), train.py:147-148,221 */
  float lr, beta1, beta2, eps, bc1, bc2_sqrt;   /* Adam: bias corrections 1-beta1^t, sqrt(1-beta2^t) */
  int smooth;             /* epoch > 0 or batch_index > queue_batch, train.py:212 */
  int queue_ptr[2];       /* write positions of the two banks for THIS step (train.py:232-237, host keeps the quirk) */
  unsigned long long seed, offset;   /* device Philox stream for noise / dropout when no tensors are injected */
  float grad_amax;        /* scratch: max |dL/dcat[:, :conv]| of this step, conv = cat - 1024 (head backward) */
  int pad_;
} cmlpl_train_params;

typedef struct cmlpl_train_io {
  int bs, btu, bands, classes, w, queue;      /* w = 20 or 11, classes <= 32, bands <= 512 */
  /* ---- inputs */
  const float* cube; int scene_rows, cols;    /* f32 [R, cols, 60] PCA cube, or NULL: patch_noise then HOLDS the input patches */
  const int64_t* pix;                         /* i64 [nb] raster pixel per row (both nets read the same pixels) */
  const float* patch_noise;                   /* f32 [2, nb, 60, w, w] N(0,1) draws (train.py:157-182) or NULL -> Philox */
  const float* spectra;                       /* f32 [rows, B] z-scored spectra */
  const int64_t* spec_row;                    /* i64 [nb] row of `spectra` per sample; NULL: row pix[i] (cube mode) or the
                                                 assembled inputs f32 [2, nb, B] themselves (cube == NULL) */
  const float* spec_noise;                    /* f32 [2, nb, B] or NULL -> Philox (none when cube == NULL) */
  const float* drop_mask;                     /* f32 [2, nb, cat] inverted-dropout mask (0 or 1/(1-p)) or NULL -> Philox */
  const int64_t* labels;                      /* i64 [bs] 0-based (train.py:159) */
  cmlpl_train_net net[2];
  cmlpl_train_params* params;                 /* device */
  /* ---- outputs (all device) */
  float* logits;      /* f32 [2, nb, C] */
  float* feat;        /* f32 [2, nb, 1024] unit rows (models.py:145-146) */
  float* probs;       /* f32 [2, btu, C]: [0] = probs (target of net 0, from net 1), [1] = probs1 (train.py:203-217) */
  float* mask;        /* f32 [2, btu]:    [0] = mask, [1] = masks (train.py:222,228) */
  float* hist;        /* f32 [12]: lc, total, cls, con, acc(net1 on labelled), total1, cls1, con1, lc1, 3 spare */
  float* grad_flat; size_t grad_flat_bytes;   /* optional: one block holding every g[] tensor of both nets (cleared with ONE
                                                 memset instead of one per tensor) */
  void* work; size_t work_bytes;              /* cmlpl_train_workspace_bytes() */
} cmlpl_train_io;

/* The size of the w = 20 layout, which bounds a w = 11 step of the same (bs, btu, bands, classes, queue): both windows
 * use this size and the same region offsets. */
size_t cmlpl_train_workspace_bytes(int bs, int btu, int bands, int classes, int queue);
/* Byte offsets of the workspace regions (tests / profiling): offsets[20] = {x16, a0, p1, m1, m2, cat, dmask, ynoisy,
 * norm, dlogits, dfeat, dcat, dhp, dz1, da0, S, G, dG, probs_orig, total}.  Per-sample activations x16 / a0 / dz1 / da0
 * are f16 [2*nb][8 chunks][P1][8], p1 f16 [2*nb][8][P2][8]; m1 / m2 are ReLU masks u32 [2*nb][P1 | P2][2] (bit c%32 of
 * word c/32); cat / dmask / dcat f32 [2*nb][cat]; positions are row-major (y*side + x).  Each region is packed densely
 * from its offset at the window's own sizes:
 *   w = 20: P1 = 400 (20x20), P2 = 100 (10x10), cat = 2624 -- per sample 51 200 B (x16 / a0 / dz1 / da0),
 *           12 800 B (p1), 3 200 B (m1), 800 B (m2); row stride of cat / dmask / dcat 2624 floats
 *   w = 11: P1 = 121 (11x11), P2 = 25 (5x5), cat = 1280 -- per sample 15 488 B, 3 200 B, 968 B, 200 B; row stride 1280
 * At w = 11 the pools drop the last row / column of each map: their m1 / m2 bits and dz1 entries are stored as 0.
 * dz1 / da0 carry the power-of-two gradient scale 2^(12 - exponent(grad_amax)). */
int cmlpl_train_workspace_layout(int bs, int btu, int bands, int classes, int queue, size_t* offsets);
/* phases: bit 0 forward (gather+noise -> logits, feat), bit 1 losses (+ bank update, dlogits, dfeat),
 * bit 2 backward (all gradients), bit 3 Adam.  15 = the whole step. */
int cmlpl_train_step(const cmlpl_train_io* io, int phases, cmlpl_stream_t stream);
/* number of kernel launches cmlpl_train_step(io, phases) enqueues (for bench.py's gpu_launches) */
int cmlpl_train_step_launches(int phases);

#ifdef __cplusplus
}
#endif
#endif /* CMLPL_H_ */
