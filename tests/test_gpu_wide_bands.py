"""Spectra beyond 256 bands on the GPU (-m gpu): the fused training step and the raw-cube scene entry point up to 512
bands, and the WHU-Hi scenes through the CLIs.

  * the step's spectral noise in cube mode (device Philox) against a numpy port of the stream: the draws below 256
    bands are those of every earlier build, and at 425 bands no two (sample, band) positions share a draw;
  * one step against the oracle's ref_step at 270 / 425 / 274 bands (w = 20 and w = 11), at the bars of
    test_gpu_fused_step.py, and eight consecutive CUDA-graph replays at 270 bands with Adam checked exactly;
  * cmlpl_scene_infer_raw at 240 / 270 / 425 bands (the per-pixel path, the K-sliced conv0 above 256 bands and the
    CUDA-core spectral head reading the raw band) against cmlpl_scene_infer on the device-preprocessed scene, against the
    oracle, in row bands, and its conv0 map against torch;
  * sample_generation --dataID 7 --synthetic + train on a small HongHu-shaped scene, at w = 20 and w = 11.
"""
import numpy as np
import pytest
import torch

from fused_step_harness import eight_steps_graph_replay, one_step_against_oracle
from oracle import cmlpl_oracle as O
from scene_harness import near_ties_only, raw_scene, rel, scene_net
from test_wide_bands_cpu import spectral_noise

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- 1. noise layout
@pytest.mark.parametrize("B", [103, 270, 425])
def test_spectral_noise_matches_the_philox_port(dev, B):
    """Cube mode, noise from the device Philox stream: (ynoisy - spectra) / sigma of every sample and band equals the
    numpy port of philox_normal4 at the counters of spec_noise_counter to 1e-4 (the kernel's __logf / __sincosf differ
    from float64 in the last bits; a wrong counter gives O(1) differences)."""
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.tools.models import BaseNet2
    R, C, K, nb = 40, 50, 9, 256
    g = torch.Generator().manual_seed(B)
    cube = torch.randn(R, C, 60, generator=g).to(dev)
    spectra = torch.randn(R * C, B, generator=g).to(dev)
    pix = torch.randint(0, R * C, (nb,), generator=g)
    labels = torch.randint(0, K, (128,), generator=g).to(dev)
    torch.manual_seed(B)
    nets = [BaseNet2(B, 0.8, K).to(dev) for _ in range(2)]
    sigma = 0.5
    fs = FusedMutualStep(nets[0], nets[1], noise=sigma, seed=1088, thr=0.5)
    assert (fs.seed, fs.offset) == (1088, 0)
    fs.step(labels, 1, 0, cube=cube, pix=pix.to(dev), spectra=spectra)
    torch.cuda.synchronize()
    lay, ns = fs.workspace_layout(), 2 * nb
    y = fs.work[lay["ynoisy"]:lay["ynoisy"] + ns * B * 4].view(torch.float32).view(ns, B).cpu().double().numpy()
    x = spectra[pix.to(dev)].cpu().double().numpy()
    got = (y - np.concatenate([x, x])) / sigma
    want = spectral_noise(1088, 0, ns, B)
    err = np.abs(got - want)
    print("B = %d: max |draw - port| %.1e" % (B, err.max()))
    assert err.max() < 1e-4
    assert abs(got.mean()) < 1e-2 and abs(got.var() - 1.0) < 2e-2
    if B > 256:
        # the aliasing a 64-quad counter stride would cause: sample s at bands 256.. == sample s+1 at bands 0..
        n = B - 256
        assert np.abs(got[:-1, 256:] - got[1:, :n]).max(1).min() > 1.0
        assert np.unique(want).size == want.size


# ------------------------------------------------------------------------------------------ 2. one step, oracle
#   id           bs   btu  B    K   w   epoch batch (queue_ptr, queue_ptr1) seed
STEP_SHAPES = {
    "b270_k22":  (128, 128, 270, 22, 20, 1, 5, (512, 768), 2701),     # WHU-Hi-HongHu
    "b425_k16":  (64, 64, 425, 16, 20, 2, 9, (256, 384), 4251),       # AVIRIS-NG radiance
    "b274_k16_w11": (128, 128, 274, 16, 11, 1, 7, (1024, 256), 2741),  # WHU-Hi-HanChuan, 11 x 11 windows
}


@pytest.mark.parametrize("case", list(STEP_SHAPES))
def test_one_step_wide_bands(dev, golden_dir, case):
    bs, btu, B, K, w, epoch, batch_index, ptrs, seed = STEP_SHAPES[case]
    one_step_against_oracle(dev, golden_dir, w, bs, btu, B, K, epoch, batch_index, ptrs, "random", seed)


def test_consecutive_steps_graph_replay_270_bands(dev, golden_dir):
    """Eight 128 + 128 steps at 270 bands / 22 classes of one FusedMutualStep captured once as a CUDA graph and replayed
    on new inputs, re-anchored on the oracle before every step (fused_step_harness.eight_steps_graph_replay): smoothing
    switches on at batch 4, the bank pointer wraps at 1280, and Adam at steps 1..8 is checked exactly against float64."""
    eight_steps_graph_replay(dev, golden_dir, 20, 270, 22, 270, 2702)


# ------------------------------------------------------------------------------------------ 3. raw entry point
@pytest.mark.parametrize("dtype", ["u16", "f32"])
@pytest.mark.parametrize("B,K,w", [(240, 16, 20), (270, 22, 20), (425, 16, 20), (270, 9, 11)])
def test_raw_entry_point_wide_bands(dev, B, K, w, dtype):
    """The raw entry point against the cube entry point on the same scene preprocessed by preprocess.apply (2e-3) and
    against the oracle's test_whole (1e-3); labels = argmax of the logits; row bands with their halo slabs reproduce the
    one-call labels and logits bit for bit."""
    from cmlpl_b200 import ops, preprocess
    R, C = 29, 37
    _, raw, pp, ref_cube, ref_spec = raw_scene(dev, R, C, B, K, seed=B + K)
    net, sd = scene_net(B, K, w, B * 7 + K, dev)
    packed = net.packed_weights(w)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    raw_in = raw if dtype == "u16" else raw.float()
    lab, lg = ops.scene_infer_raw(raw_in, folded, packed, K, C, w, want_logits=True)
    cube, spec = preprocess.apply(raw, pp)
    lab_c, lg_c = ops.scene_infer(cube.view(R, C, 60), spec, packed, K, w, want_logits=True)
    lab_ref, log_ref = O.test_whole(sd, ref_cube, ref_spec, w, odd_mode=(w == 11), return_logits=True)
    lab, lg, lg_c = lab.cpu().numpy(), lg.cpu().numpy(), lg_c.cpu().numpy()
    print("B = %d, K = %d, w = %d, %s: rel err vs cube entry %.1e, vs oracle %.1e" % (B, K, w, dtype, rel(lg, lg_c),
                                                                                   rel(lg, log_ref)))
    assert rel(lg, lg_c) < 2e-3
    assert rel(lg, log_ref) < 1e-3
    assert np.array_equal(lab, lg.argmax(1))
    assert near_ties_only(lab, lab_ref, log_ref)
    bands = [(0, 1), (1, 9), (9, 10), (10, 22), (22, 29)]
    lo, hi = w // 2, w - w // 2 - 1
    parts = []
    for a, b in bands:
        s0, s1 = max(0, a - lo), min(R, b + hi)
        parts.append(ops.scene_infer_raw(raw_in[s0 * C:s1 * C].contiguous(), folded, packed, K, C, w, band_row0=a,
                                         band_rows=b - a, scene_rows=R, slab_row0=s0, want_logits=True))
    assert np.array_equal(torch.cat([p[0] for p in parts]).cpu().numpy(), lab)
    assert np.array_equal(torch.cat([p[1] for p in parts]).cpu().numpy(), lg)


@pytest.mark.parametrize("B", [270, 512])
def test_raw_conv0_map_matches_torch(dev, B):
    """The conv0 map the K-sliced kernel writes (workspace offset 0, chunk-planar f16 [8][R+w-1][C+w-1][8]) against a
    float64 torch evaluation of the folded 1x1 conv on the mirror-padded raw scene: 1e-3 of its largest entry."""
    from cmlpl_b200 import ops
    R, C, K, w = 23, 31, 22, 20
    _, raw, pp, _, _ = raw_scene(dev, R, C, B, K, seed=B)
    net, sd = scene_net(B, K, w, B, dev)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    ws = ops.scene_workspace(R, C, B, K, w, dev)
    ops.scene_infer_raw(raw, folded, net.packed_weights(w), K, C, w, workspace=ws)
    torch.cuda.synchronize()
    PR, PC = R + w - 1, C + w - 1
    got = ws[:8 * PR * PC * 16].view(torch.float16).view(8, PR, PC, 8).permute(1, 2, 0, 3).reshape(PR, PC, 64).double()
    mirror = lambda o, n: torch.where(o < 0, -o - 1, torch.where(o >= n, 2 * n - 1 - o, o))
    rr = mirror(torch.arange(PR, device=dev) - w // 2, R)
    cc = mirror(torch.arange(PC, device=dev) - w // 2, C)
    x = raw.view(R, C, B).double()[rr][:, cc]
    z = (x - folded["mu"].double()) * folded["inv_sigma"].double()
    want = (z / folded["inv_sigma"].double()) @ folded["wf"].double() + folded["bf"].double()
    err = float((got - want).abs().max() / want.abs().max())
    print("B = %d: conv0 map rel err %.1e" % (B, err))
    assert err < 1e-3


# ---------------------------------------------------------------------------------------------------- 4. the CLIs
@pytest.mark.parametrize("w", [20, 11])
def test_train_cli_honghu_synthetic(dev, tmp_path, monkeypatch, w):
    """sample_generation --dataID 7 --synthetic on a small HongHu-shaped scene (270 bands, 22 classes), then train for
    2 epochs: the fused step runs by default, test_whole labels the scene and OA / AA / kappa come out; the trained
    net's label map matches the oracle's outside near ties."""
    from cmlpl_b200 import sample_generation as SG, synth, train as T
    monkeypatch.setitem(synth.SHAPES, "whu_honghu", (48, 44, 270, 22))
    root = str(tmp_path) + "/"
    SG.main(SG.build_parser().parse_args(["--dataID", "7", "--root", root, "--synthetic", "--w", str(w)]))
    T.seed_torch()
    out = T.main(T.build_parser().parse_args(["--dataID", "7", "--root", root, "--num_epochs", "2", "--num_unlabel",
                                              "512", "--print_per_batches", "2"]))
    st = out["state"]
    assert "fused" in st.extras and st.extras["fused"].B == 270 and st.extras["fused"].w == w
    assert st.Base.num_features == 270 and st.Base.num_classes == 22 and st.Base.w == w
    assert np.isfinite(out["loss_hist"]).all()
    assert out["predict_label"].shape == (48 * 44,)
    OA, kappa, pa = out["results"][0]
    assert 1.0 / 22 < OA <= 1.0 and np.isfinite(kappa) and pa.shape == (22,)
    d = root + "WHU_Hi_HongHu/"
    cube, spectra = np.load(d + "XPCA.npy"), np.load(d + "X.npy").astype(np.float32)
    assert spectra.shape == (48 * 44, 270)
    sd = {k: v.detach().cpu() for k, v in st.Base.state_dict().items()}
    lab_ref, log_ref = O.test_whole(sd, cube, spectra, w, odd_mode=(w == 11), return_logits=True)
    got = out["predict_label"]
    print("w = %d: OA %.3f, label agreement with the oracle %.5f" % (w, OA, float(np.mean(got == lab_ref))))
    assert near_ties_only(got, lab_ref, log_ref)
