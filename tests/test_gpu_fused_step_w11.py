"""GPU parity of the fused training step at w = 11 (-m gpu): cmlpl_train_step on 11x11 windows (ExtractPatches_for_base,
pools flooring 11 -> 5 -> 2, a 1280-input classifier) against the oracle's ref_step, at the bars of
test_gpu_fused_step.py's module docstring:
  * logits / probabilities / losses / head gradients: 1e-3 * max|ref|;
  * every convolution-backward kernel against torch fp32 convolutions on the kernel's own saved tensors: 1e-3;
  * convolution gradients end to end against the fp32 oracle (on the fused forward's ReLU masks): 3e-2, with the mask
    bits that differ from fp32's counted and bounded.
The pools drop row / column 10 of conv1's map and row / column 4 of conv2's: no gradient reaches them, so the kernels
store their mask bits and dz1 entries as 0 and the checks here compare the kept positions with fp32 and the dropped
ones with what the floor pool implies.  The one-step shape matrix at w = 11 is test_gpu_fused_step_shapes.py's,
parametrised over the window; the eight graph replays run fused_step_harness's body shared with the w = 20 test.
"""
import functools
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from fused_step_harness import (CONV, GEOMETRY, assembled, cube_mode_steps, eight_steps_graph_replay, fused_for,
                                init_nets, make_inputs, random_banks, saved)
from oracle import cmlpl_oracle as O
from oracle import golden
from scene_harness import rel

pytestmark = pytest.mark.gpu

W, H2, _, CONVF, CAT = GEOMETRY[11]


# ---------------------------------------------------------------------------------------------------- 1. floor pooling
def test_floor_pool_backward(dev, golden_dir):
    """The pool backward with floor semantics, on the kernel's own saved tensors: torch autograd through F.avg_pool2d
    (which floors 11 -> 5 and 5 -> 2) of conv2 on p1 and of conv1 on a0, both with the saved ReLU masks imposed, gives
    the conv weight / bias gradients, and dL/da0 -- at the dropped row / column too, where only the neighbours' taps
    contribute; dz1 is exactly 0 on the dropped row / column."""
    B, K, bs = 103, 9, 64
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    g = torch.Generator().manual_seed(2201)
    inp = make_inputs(ti, bs, bs, B, K, g, W)
    sd, sd1 = init_nets(B, K, 2201, W)
    sa = O.StepArgs(num_epochs=20, labeled_batch_size=bs)
    sa.thr = 0.2
    fs = fused_for(dev, sd, sd1, bs, bs, B, K, random_banks(5 * bs * 2, K, g), (0, 256), sa, W)
    w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
    patches, spectra = (t.to(dev) for t in assembled(inp, sa.noise))
    fs.step(inp["Y_l"].to(dev), 1, 0, patches=patches, spectra=spectra, drop_masks=inp["masks"].to(dev))
    torch.cuda.synchronize()
    nb = 2 * bs
    t = saved(fs, nb)
    dz1 = t["dz1"]
    assert float(dz1[:, :, W - 1, :].abs().max()) == 0.0 and float(dz1[:, :, :, W - 1].abs().max()) == 0.0
    assert float(dz1[:, :, :W - 1, :W - 1].abs().max()) > 0.0
    for e in range(2):
        sl = slice(e * nb, (e + 1) * nb)
        wb = w_before[e]
        W1, b1 = wb["conv1.weight"].clone().requires_grad_(True), wb["conv1.bias"].clone().requires_grad_(True)
        W2, b2 = wb["conv2.weight"].clone().requires_grad_(True), wb["conv2.bias"].clone().requires_grad_(True)
        p1 = t["p1"][sl].clone().requires_grad_(True)
        feat = F.avg_pool2d((F.conv2d(p1, W2, b2, padding=1) + p1) * t["m2"][sl], 2, 2).flatten(1)
        assert feat.shape[1] == CONVF
        (feat * t["dcat"][sl, :CONVF]).sum().backward()
        a0 = t["a0"][sl].clone().requires_grad_(True)
        pooled = F.avg_pool2d((F.conv2d(a0, W1, b1, padding=1) + a0) * t["m1"][sl], 2, 2)
        assert pooled.shape[-1] == H2
        (pooled * p1.grad).sum().backward()
        got = dict(zip(CONV, [fs.grads[e][i] for i in range(6)]))
        errs = {"conv2.weight": rel(got["conv2.weight"], W2.grad), "conv2.bias": rel(got["conv2.bias"], b2.grad),
                "conv1.weight": rel(got["conv1.weight"], W1.grad), "conv1.bias": rel(got["conv1.bias"], b1.grad),
                "da0": rel(t["da0"][sl], a0.grad),
                "da0 dropped row / col": max(rel(t["da0"][sl][:, :, W - 1, :], a0.grad[:, :, W - 1, :]),
                                             rel(t["da0"][sl][:, :, :, W - 1], a0.grad[:, :, :, W - 1]))}
        print("net %d, floor-pool backward errors:" % e, {k: f"{v:.1e}" for k, v in errs.items()})
        for k, v in errs.items():
            assert v < 1e-3, (e, k, v)
        # the dropped row / column of da0 is not zero: the taps of row / column 9 reach it
        assert float(a0.grad[:, :, W - 1, :].abs().max()) > 0.0


# --------------------------------------------------------------------------------------------- 2. cube mode, Philox
def test_cube_mode_philox_and_graph_w11(dev, golden_dir):
    """Inputs gathered from the PCA cube in the first kernel (11x11 odd-mode windows), noise and dropout from the device
    Philox stream: the gather is exact, the draws have the right moments, reproduce for the same (seed, step) and differ
    between nets and steps; a CUDA-graph replay computes the same step as the eager launch sequence."""
    from cmlpl_b200.tools.models import BaseNet2
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    cube = torch.from_numpy(ti["cube_pca"]).to(dev).contiguous()
    spectra = torch.from_numpy(ti["spectra"]).to(dev).contiguous()
    R, C = cube.shape[:2]
    g = torch.Generator().manual_seed(5)
    # every corner and edge of the scene, then random pixels
    edge = torch.tensor([0, C - 1, (R - 1) * C, R * C - 1, 3, 2 * C, 5 * C - 1, (R - 1) * C + 7])
    pix = torch.cat([edge, torch.randint(0, R * C, (256 - edge.numel(),), generator=g)])
    labels = torch.randint(0, 9, (128,), generator=g).to(dev)
    torch.manual_seed(3)
    nets = [BaseNet2(103, 0.8, 9, w=W).to(dev) for _ in range(2)]
    sd0 = [{k: v.detach().clone() for k, v in n.state_dict().items()} for n in nets]
    ns = 512
    run = functools.partial(cube_mode_steps, nets, sd0, labels, cube, pix, spectra)
    want = torch.from_numpy(O.extract_patches_at(ti["cube_pca"], W, pix.numpy(), odd_mode=True))
    clean, _ = run(0.0, False)
    x = clean[0]["x16"]
    assert torch.equal(x[:256, :60].cpu(), want.half().float()) and torch.equal(x[256:, :60].cpu(), want.half().float())
    assert float(x[:, 60:].abs().max()) == 0.0
    assert torch.equal(clean[0]["y"][:256].cpu(), torch.from_numpy(ti["spectra"][pix.numpy()]))
    noisy, _ = run(0.5, False, steps=2)
    zn = (noisy[0]["x16"][:, :60].cpu() - torch.cat([want, want])) / 0.5                      # 3.7 M draws
    assert abs(float(zn.mean())) < 2e-3 and abs(float(zn.var()) - 1.0) < 1e-2
    assert abs(float((zn ** 4).mean()) - 3.0) < 5e-2
    zy = (noisy[0]["y"].cpu() - torch.from_numpy(ti["spectra"][pix.numpy()]).repeat(2, 1)) / 0.5
    assert abs(float(zy.mean())) < 2e-2 and abs(float(zy.var()) - 1.0) < 3e-2
    keep = float((noisy[0]["dmask"] > 0).float().mean())
    assert abs(keep - 0.2) < 3e-3 and float(noisy[0]["dmask"].max()) == pytest.approx(5.0)
    assert not torch.equal(noisy[0]["x16"][:256], noisy[0]["x16"][256:])
    assert not torch.equal(noisy[0]["x16"], noisy[1]["x16"])
    dm = noisy[0]["dmask"].view(ns, CAT)
    assert not torch.equal(dm[:256], dm[256:]) and not torch.equal(noisy[0]["dmask"], noisy[1]["dmask"])
    again, _ = run(0.5, False, steps=2)
    assert torch.equal(again[0]["x16"], noisy[0]["x16"]) and torch.equal(again[1]["dmask"], noisy[1]["dmask"])
    other, _ = run(0.5, False, seed=7)
    assert not torch.equal(other[0]["x16"], noisy[0]["x16"])
    eager, _ = run(0.5, False, steps=3)
    graph, fsg = run(0.5, True, steps=3)
    assert torch.equal(eager[0]["logits"], graph[0]["logits"])
    for a, b in zip(eager[2]["w"], graph[2]["w"]):
        assert rel(a, b) < 1e-4
    assert fsg.launches() == 15 and np.isfinite(graph[2]["hist"].cpu().numpy()).all()


# -------------------------------------------------------------------------------------------- 3. consecutive steps
def test_consecutive_steps_graph_replay_w11(dev, golden_dir):
    """Eight 128 + 128 w = 11 steps of one FusedMutualStep captured once as a CUDA graph and replayed on new inputs,
    re-anchored on the oracle before every step: bank smoothing switches on at batch 4, the bank pointer wraps at 1280,
    and Adam at steps 2..8 is checked exactly against float64 (fused_step_harness.eight_steps_graph_replay)."""
    eight_steps_graph_replay(dev, golden_dir, W, 103, 9, 42, 4243)


# ------------------------------------------------------------------------------------------------- 4. the CLI
@pytest.mark.parametrize("fp32_step", [False, True], ids=["fused", "fp32_step"])
def test_train_cli_w11_end_to_end_synthetic(dev, tmp_path, fp32_step):
    """sample_generation --w 11, then train for 2 epochs, on a tiny synthetic scene: the fused step by default, the fp32
    mutual_step with --fp32_step; the trained net's label map through the w = 11 scene path against the oracle."""
    from cmlpl_b200 import sample_generation as SG, synth, train as T
    synth.SHAPES["paviau"] = (48, 44, 103, 9)
    try:
        root = str(tmp_path) + "/"
        SG.main(SG.build_parser().parse_args(["--dataID", "1", "--root", root, "--synthetic", "--w", "11"]))
        T.seed_torch()
        argv = ["--dataID", "1", "--root", root, "--num_epochs", "2", "--num_unlabel", "512", "--print_per_batches", "2"]
        out = T.main(T.build_parser().parse_args(argv + (["--fp32_step"] if fp32_step else [])))
    finally:
        synth.SHAPES["paviau"] = (610, 340, 103, 9)
    st = out["state"]
    assert st.Base.w == W and st.Base1.w == W and st.Base.classifier.in_features == CAT
    assert ("fused" in st.extras) != fp32_step
    h = out["loss_hist"]
    assert h.shape == (8, 5) and np.isfinite(h).all()
    assert h[-1, 2] < h[0, 2]                                   # supervised CE goes down
    assert out["predict_label"].shape == (48 * 44,) and out["predict_label"].dtype == np.int64
    OA, kappa, pa = out["results"][0]
    assert 0.5 < OA <= 1.0 and pa.shape == (9,)
    if fp32_step:
        return
    d = root + "PaviaU/"
    cube, spectra = np.load(d + "XPCA.npy"), np.load(d + "X.npy").astype(np.float32)
    sd = {k: v.detach().cpu() for k, v in st.Base.state_dict().items()}
    lab_ref, log_ref = O.test_whole(sd, cube, spectra, W, odd_mode=True, return_logits=True)
    got = out["predict_label"]
    agree = float(np.mean(got == lab_ref))
    print("fused-trained w = 11 net: label agreement with the oracle %.5f" % agree)
    assert agree >= 0.999
    scale = float(np.abs(log_ref).max())
    for i in np.nonzero(got != lab_ref)[0]:                     # every disagreement is a near tie
        assert log_ref[i, lab_ref[i]] - log_ref[i, got[i]] < 2e-3 * scale, (i, log_ref[i])


# ------------------------------------------------------------------------------------------------- 5. loud failures
def test_w11_argument_checks(dev):
    from cmlpl_b200 import _lib
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.tools.models import BaseNet2
    torch.manual_seed(0)
    with pytest.raises(_lib.CmlplError, match="w=13"):
        FusedMutualStep(BaseNet2(103, 0, 9, w=13).to(dev), BaseNet2(103, 0, 9, w=13).to(dev))
    with pytest.raises(_lib.CmlplError, match="different windows"):
        FusedMutualStep(BaseNet2(103, 0, 9, w=11).to(dev), BaseNet2(103, 0, 9, w=20).to(dev))
    fs = FusedMutualStep(BaseNet2(103, 0, 9, w=11).to(dev), BaseNet2(103, 0, 9, w=11).to(dev), bs=16, btu=16)
    y = torch.zeros(16, dtype=torch.int64, device=dev)
    spectra = torch.zeros(2, 32, 103, device=dev)
    with pytest.raises(_lib.CmlplError, match="patches"):
        fs.step(y, 0, 0, patches=torch.zeros(2, 32, 60, 20, 20, device=dev), spectra=spectra)
    with pytest.raises(_lib.CmlplError, match="drop_masks"):
        fs.step(y, 0, 0, patches=torch.zeros(2, 32, 60, W, W, device=dev), spectra=spectra,
                drop_masks=torch.ones(2, 32, 2624, device=dev))
    with pytest.raises(_lib.CmlplError, match="patch_noise"):
        fs.step(y, 0, 0, cube=torch.zeros(16, 16, 60, device=dev), pix=torch.zeros(32, dtype=torch.int64, device=dev),
                spectra=torch.zeros(256, 103, device=dev), patch_noise=torch.zeros(2, 32, 60, 20, 20, device=dev))
