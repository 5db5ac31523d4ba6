// cmlpl_train_step: one mutual-learning step of train.py:150-272 for both BaseNet2 peers as 15 kernel launches
// (+ memsets of the gradient block) on one stream; every per-step scalar is read from the device-side
// cmlpl_train_params, so the sequence can be captured once in a CUDA graph and replayed.
#include "common.cuh"
#include "train_common.cuh"
#include "train_kernels.cuh"
#include "train_head.cuh"

using namespace cmlpl;

namespace {
constexpr int64_t kNumel[CMLPL_TRAIN_TENSORS] = {64 * 60, 64, 64 * 64 * 9, 64, 64 * 64 * 9, 64, 0 /*1024*B*/, 1024, 0 /*C*cat*/, 0 /*C*/};
int64_t numel(int i, int B, int C, int cat) {
  if (i == 6) return int64_t(1024) * B;
  if (i == 8) return int64_t(C) * cat;
  if (i == 9) return C;
  return kNumel[i];
}
}  // namespace

extern "C" size_t cmlpl_train_workspace_bytes(int bs, int btu, int bands, int classes, int queue) {
  if (bs <= 0 || btu <= 0 || bands <= 0 || classes <= 0 || queue <= 0) return 0;
  return train_ws_layout(bs, btu, bands, classes, queue).total;
}

extern "C" int cmlpl_train_workspace_layout(int bs, int btu, int bands, int classes, int queue, size_t* offsets) {
  CMLPL_CHECK_ARG(offsets && bs > 0 && btu > 0 && bands > 0 && classes > 0 && queue > 0, "train_workspace_layout: bad args");
  const TrainWs L = train_ws_layout(bs, btu, bands, classes, queue);
  const size_t v[20] = {L.x16, L.a0, L.p1, L.m1, L.m2, L.cat, L.dmask, L.ynoisy, L.norm, L.dlogits,
                        L.dfeat, L.dcat, L.dhp, L.dz1, L.da0, L.S, L.G, L.dG, L.probs_orig, L.total};   // (+ wpack, gstage: internal)
  for (int i = 0; i < 20; ++i) offsets[i] = v[i];
  return CMLPL_OK;
}

extern "C" int cmlpl_train_step_launches(int phases) {
  return ((phases & 1) ? 4 : 0) + ((phases & 2) ? 4 : 0) + ((phases & 4) ? 6 : 0) + ((phases & 8) ? 1 : 0);
}

extern "C" int cmlpl_train_step(const cmlpl_train_io* io, int phases, cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(io, "train_step: null io");
  CMLPL_CHECK_ARG(io->w == 20 || io->w == 11, "train_step: w=%d unsupported (20 = the reference's BaseNet2, "
                  "tools/models.py:127; 11 = the odd window of ExtractPatches_for_base)", io->w);
  CMLPL_CHECK_ARG(io->bs > 0 && io->btu > 0 && io->bands > 0 && io->classes > 0 && io->classes <= 32 &&
                      io->queue > 0, "train_step: bad dims (bs=%d btu=%d bands=%d classes=%d queue=%d)", io->bs, io->btu,
                  io->bands, io->classes, io->queue);
  // the spectral noise counter (train_common.cuh: spec_noise_counter) keeps its draws disjoint up to 512 bands
  CMLPL_CHECK_ARG(io->bands <= 512, "train_step: needs <= 512 bands, got %d", io->bands);
  CMLPL_CHECK_ARG(io->params && io->work && io->spectra && io->labels && io->logits && io->feat && io->probs && io->mask &&
                      io->hist, "train_step: null pointer");
  CMLPL_CHECK_ARG(io->cube ? (io->pix != nullptr && io->scene_rows >= 10 && io->cols >= 10) : io->patch_noise != nullptr,
                  "train_step: pass the PCA cube + pixel indices, or the assembled patches in patch_noise");
  const int bs = io->bs, btu = io->btu, nb = bs + btu, B = io->bands, C = io->classes, Q = io->queue, w = io->w;
  // classifier input width and its conv-feature head (2624 / 1600 at w = 20, 1280 / 256 at w = 11); a w = 11 step
  // uses the w = 20 workspace layout, packing each region at its own per-sample strides
  const int cat = w == 11 ? TrainGeom<11>::CatDim : kCatDim, conv = cat - kHid;
  const TrainWs L = train_ws_layout(bs, btu, B, C, Q);
  CMLPL_CHECK_ARG(io->work_bytes >= L.total, "train_step: workspace of %zu bytes, need %zu", io->work_bytes, L.total);
  CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(io->work) % 256 == 0, "train_step: workspace must be 256-byte aligned");
  for (int e = 0; e < 2; ++e) {
    for (int i = 0; i < CMLPL_TRAIN_TENSORS; ++i)
      CMLPL_CHECK_ARG(io->net[e].p[i] && io->net[e].g[i] && io->net[e].m[i] && io->net[e].v[i], "train_step: net %d tensor %d is null", e, i);
    CMLPL_CHECK_ARG(io->net[e].queue_feats && io->net[e].queue_probs, "train_step: net %d has no memory bank", e);
    CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(io->net[e].p[8]) % 16 == 0 && reinterpret_cast<uintptr_t>(io->net[e].queue_feats) % 16 == 0,
                    "train_step: classifier weight / bank must be 16-byte aligned");
  }
  CMLPL_CHECK_ARG(reinterpret_cast<uintptr_t>(io->feat) % 16 == 0 && (!io->cube || reinterpret_cast<uintptr_t>(io->cube) % 16 == 0) &&
                      (!io->drop_mask || reinterpret_cast<uintptr_t>(io->drop_mask) % 16 == 0),
                  "train_step: feat / cube / drop_mask must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the library's side stream (common.cuh) carries the step's two forks; its lock is held for the whole enqueue
  SideStream* sd = side_stream();
  CMLPL_CHECK_ARG(sd, "train_step: could not create the side stream");
  std::lock_guard<std::mutex> lock(sd->mu);
  unsigned char* ws = static_cast<unsigned char*>(io->work);
  auto f32 = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
  auto f16 = [&](size_t off) { return reinterpret_cast<__half*>(ws + off); };
  const cmlpl_train_params* prm = io->params;
  int rc;

  HeadArgs ha{};
  ha.prm = prm; ha.prm_rw = io->params; ha.nb = nb; ha.bs = bs; ha.btu = btu; ha.C = C; ha.training = 1;
  ha.cat = f32(L.cat); ha.dmask = f32(L.dmask); ha.drop_mask = io->drop_mask;
  ha.logits = io->logits; ha.feat = io->feat; ha.norm = f32(L.norm);
  ha.dlogits = f32(L.dlogits); ha.dfeat = f32(L.dfeat); ha.dcat = f32(L.dcat); ha.dhp = f32(L.dhp);
  for (int e = 0; e < 2; ++e) {
    ha.wc[e] = io->net[e].p[8]; ha.bc[e] = io->net[e].p[9];
    ha.g_wc[e] = io->net[e].g[8]; ha.g_bc[e] = io->net[e].g[9]; ha.g_bs[e] = io->net[e].g[7];
  }

  if (phases & 1) {
    Conv0Args a{};
    a.cube = io->cube; a.scene_rows = io->scene_rows; a.cols = io->cols; a.pix = io->pix; a.noise = io->patch_noise;
    a.prm = prm; a.x16 = f16(L.x16); a.a0 = f16(L.a0); a.nb = nb;
    a.spectra = io->spectra; a.spec_row = io->spec_row; a.spec_noise = io->spec_noise; a.ynoisy = f32(L.ynoisy); a.bands = B;
    a.hist = io->hist; a.prm_rw = io->params;
    a.wpack = ws + L.wpack;
    TrainCnnArgs t{};
    t.a0 = f16(L.a0); t.wpack = ws + L.wpack; t.p1 = f16(L.p1); t.m1 = reinterpret_cast<uint32_t*>(ws + L.m1);
    t.m2 = reinterpret_cast<uint32_t*>(ws + L.m2); t.cat = f32(L.cat); t.nb = nb;
    MultiGemm mg{};
    mg.count = 2;
    for (int e = 0; e < 2; ++e) {
      a.w0[e] = io->net[e].p[0]; a.b0[e] = io->net[e].p[1];
      a.w3[e][0] = io->net[e].p[2]; a.w3[e][1] = io->net[e].p[4];
      t.b1[e] = io->net[e].p[3]; t.b2[e] = io->net[e].p[5];
      // h = relu(feat_spe(y)) into the tail of cat (models.py:142-144)
      mg.p[e] = GemmProb{f32(L.ynoisy) + int64_t(e) * nb * B, B, 1, io->net[e].p[6], 1, B,
                         f32(L.cat) + int64_t(e) * nb * cat + conv, cat, 1, io->net[e].p[7], nullptr,
                         nb, kHid, B, 1.f, 1};
    }
    if ((rc = launch_train_conv0(a, w, st)) != CMLPL_OK) return rc;
    // fork: the spectral GEMM (needs only the noisy spectra of kernel 1) next to the conv trunk
    CMLPL_CUDA(cudaEventRecord(sd->fork[0], st));
    CMLPL_CUDA(cudaStreamWaitEvent(sd->s, sd->fork[0], 0));
    if ((rc = launch_multi_gemm(mg, sd->s, "train_spectral_fwd")) != CMLPL_OK) return rc;
    CMLPL_CUDA(cudaEventRecord(sd->join[0], sd->s));
    if ((rc = launch_train_cnn(t, w, st)) != CMLPL_OK) return rc;
    CMLPL_CUDA(cudaStreamWaitEvent(st, sd->join[0], 0));
    if ((rc = launch_head_fwd(ha, w, st)) != CMLPL_OK) return rc;
  }

  if (phases & 2) {
    LossArgs la{};
    la.prm = prm; la.bs = bs; la.btu = btu; la.C = C; la.queue = Q;
    la.logits = io->logits; la.feat = io->feat; la.labels = io->labels;
    la.S = f32(L.S); la.G = f32(L.G); la.dG = f32(L.dG);
    la.probs_orig = f32(L.probs_orig); la.probs = io->probs; la.mask = io->mask;
    la.dlogits = f32(L.dlogits); la.hist = io->hist;
    const float* xs = io->feat + int64_t(bs) * kHid;              // unlabelled features of net 0 (xs_feature)
    const float* xw = io->feat + (int64_t(nb) + bs) * kHid;       // unlabelled features of net 1 (xw_feature)
    SimBatch sims{};
    sims.count = 3;
    sims.prm = prm;
    const int nparts = 2 * ((Q + 127) / 128);
    for (int t = 0; t < 2; ++t) {
      la.queue_feats[t] = io->net[t].queue_feats; la.queue_probs[t] = io->net[t].queue_probs;
      // bank t: feats_u(net 1-t) . queue_feats[t]^T, streamed into exp sums (train.py:213-217), never materialised
      sims.p[t] = SimProb{t == 0 ? xw : xs, io->net[t].queue_feats, kHid, kHid, btu, Q, kHid, 1, nullptr, 0,
                          io->net[t].queue_probs, f32(L.S) + int64_t(t) * nparts * btu * 33, C, &prm->smooth};
    }
    sims.p[2] = SimProb{xs, xw, kHid, kHid, btu, btu, kHid, 0, f32(L.G), btu, nullptr, nullptr, 0, nullptr};   // train.py:246
    MultiGemm dfe{};
    dfe.count = 2;
    // d xs = dG . xw (loss_contrast -> net 0), d xw = dG^T . xs (loss_contrast1 -> net 1); dG carries 0.5/T/n
    dfe.p[0] = GemmProb{f32(L.dG), btu, 1, xw, kHid, 1, f32(L.dfeat), kHid, 1, nullptr, nullptr, btu, kHid, btu, 1.f, 0};
    dfe.p[1] = GemmProb{f32(L.dG), 1, btu, xs, kHid, 1, f32(L.dfeat) + int64_t(btu) * kHid, kHid, 1, nullptr, nullptr,
                        btu, kHid, btu, 1.f, 0};
    if ((rc = launch_sim_tc(sims, st, "train_sims")) != CMLPL_OK) return rc;
    if ((rc = launch_loss_rows(la, st)) != CMLPL_OK) return rc;
    if ((rc = launch_loss_graph(la, st)) != CMLPL_OK) return rc;
    if ((rc = launch_multi_gemm(dfe, st, "train_dfeat")) != CMLPL_OK) return rc;
  }

  if (phases & 4) {
    if (io->grad_flat) {
      CMLPL_CUDA(cudaMemsetAsync(io->grad_flat, 0, io->grad_flat_bytes, st));
    } else {
      for (int e = 0; e < 2; ++e)
        for (int i = 0; i < CMLPL_TRAIN_TENSORS; ++i)
          CMLPL_CUDA(cudaMemsetAsync(io->net[e].g[i], 0, size_t(numel(i, B, C, cat)) * 4, st));
    }
    CMLPL_CUDA(cudaMemsetAsync(ws + L.gstage, 0, size_t(4) * 36864 * 4, st));
    if ((rc = launch_head_bwd(ha, w, st)) != CMLPL_OK) return rc;
    MultiGemm dws{};
    dws.count = 2;
    ConvBwdArgs b2{}, b1{};
    Conv0BwdArgs b0{};
    b2.prm = b1.prm = b0.prm = prm;
    b2.nb = b1.nb = b0.nb = nb;
    b2.dcat = f32(L.dcat); b2.m2 = reinterpret_cast<const uint32_t*>(ws + L.m2);
    b2.m1 = reinterpret_cast<const uint32_t*>(ws + L.m1); b2.act = f16(L.p1); b2.dz_out = f16(L.dz1);
    b1.act = f16(L.a0); b1.dz_in = f16(L.dz1); b1.dz_out = f16(L.da0);
    b0.da0 = f16(L.da0); b0.x16 = f16(L.x16); b0.gstage = f32(L.gstage);
    for (int e = 0; e < 2; ++e) {
      // dWs[j][b] = sum_s dhp[s][j] * y[s][b]  (feat_spe weight gradient)
      dws.p[e] = GemmProb{f32(L.dhp) + int64_t(e) * nb * kHid, 1, kHid, f32(L.ynoisy) + int64_t(e) * nb * B, B, 1,
                          io->net[e].g[6], B, 1, nullptr, nullptr, kHid, B, nb, 1.f, 0};
      b2.wpack[e] = ws + L.wpack + size_t(e * 2 + 1) * 2 * kWPackBytes + kWPackBytes;
      b1.wpack[e] = ws + L.wpack + size_t(e * 2 + 0) * 2 * kWPackBytes + kWPackBytes;
      b2.g_stage[e] = f32(L.gstage) + size_t(e * 2 + 1) * 36864; b2.g_b[e] = io->net[e].g[5];
      b1.g_stage[e] = f32(L.gstage) + size_t(e * 2 + 0) * 36864; b1.g_b[e] = io->net[e].g[3];
      b0.g_w[e] = io->net[e].g[0]; b0.g_b[e] = io->net[e].g[1];
      b0.g_w3[e][0] = io->net[e].g[2]; b0.g_w3[e][1] = io->net[e].g[4];
    }
    // fork: the head weight gradients (classifier, feat_spe) next to the conv backward chain
    CMLPL_CUDA(cudaEventRecord(sd->fork[1], st));
    CMLPL_CUDA(cudaStreamWaitEvent(sd->s, sd->fork[1], 0));
    if ((rc = launch_head_wgrad(ha, w, sd->s)) != CMLPL_OK) return rc;
    if ((rc = launch_multi_gemm(dws, sd->s, "train_spectral_wgrad")) != CMLPL_OK) return rc;
    CMLPL_CUDA(cudaEventRecord(sd->join[1], sd->s));
    if ((rc = launch_train_conv_bwd(w / 2, b2, st)) != CMLPL_OK) return rc;      // conv2: 10 x 10 / 5 x 5
    if ((rc = launch_train_conv_bwd(w, b1, st)) != CMLPL_OK) return rc;          // conv1: 20 x 20 / 11 x 11
    if ((rc = launch_train_conv0_bwd(b0, w, st)) != CMLPL_OK) return rc;
    CMLPL_CUDA(cudaStreamWaitEvent(st, sd->join[1], 0));
  }

  if (phases & 8) {
    AdamAll t{};
    t.prm = prm;
    t.count = 0;
    for (int e = 0; e < 2; ++e)
      for (int i = 0; i < CMLPL_TRAIN_TENSORS; ++i) {
        const int k = t.count++;
        t.p[k] = io->net[e].p[i]; t.g[k] = io->net[e].g[i]; t.m[k] = io->net[e].m[i]; t.v[k] = io->net[e].v[i];
        t.n[k] = numel(i, B, C, cat);
      }
    if ((rc = launch_adam_all(t, st)) != CMLPL_OK) return rc;
  }
  return CMLPL_OK;
}
