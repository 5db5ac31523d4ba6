"""GPU parity of the fused training step (cmlpl_train_step) beyond the 128 + 128 / 9-16-class shapes of
test_gpu_fused_step.py, with the same bars (its module docstring).  The gradients are compared with the oracle's on
the fused forward's own ReLU masks (on_fused_masks); the masks themselves are compared with fp32's and bounded.

  * a shape matrix for each window (w = 20 and 11), one step each against the oracle's ref_step: 17-32 classes (every
    <32> instantiation of the head and loss kernels, sim_tc_kernel's C > 16 branch), 224 and 256 bands, banks that end
    in a partial 128-row tile, bs != btu, btu > 128 and btu < 32, and the first steps of a run (bank smoothing off,
    zero banks);
  * eight consecutive steps through one FusedMutualStep replayed as a CUDA graph, re-anchored on the oracle before
    every step: smoothing switching on, the bank pointers wrapping, and Adam at steps 2..8 checked exactly (the same
    body runs at w = 11 in test_gpu_fused_step_w11.py and at 270 bands in test_gpu_wide_bands.py);
  * the fp16 range of the backward pass: trained weights, 3x3 weights scaled up to 16x and a classifier that drives
    max|dL/dcat| small.

Every FusedMutualStep is built at exactly the batch it runs, so workspace_layout() (the constructor's sizes) is the
layout the kernels used.
"""
import copy
import math
import os

import numpy as np
import pytest
import torch

from fused_step_harness import (assert_soft_ce_exercised, compare_with_oracle, eight_steps_graph_replay, fused_for,
                                fused_step, linearised_check, make_inputs, on_fused_masks, one_step_against_oracle,
                                oracle_step, planes_to_nchw, random_banks, set_banks)
from oracle import cmlpl_oracle as O
from oracle import golden

pytestmark = pytest.mark.gpu

FP16_MAX = 65504.0


# ---------------------------------------------------------------------------------------------------- A. shape matrix
#   id       bs   btu  B    K  epoch batch (queue_ptr, queue_ptr1) banks  seed   thr     alpha  net seed
SHAPES = {20: {
    "k24":   (128, 128, 103, 24, 1, 10, (512, 768), "random", 1209, 0.0829, 0.95, 31),  # every <32> kernel, sim_tc C > 16
    "k32":   (128, 128, 256, 32, 2, 40, (1024, 256), "random", 1208, 0.0987, 0.95, 31), # the largest classes / bands the ABI takes
    "q1000": (100, 100, 144, 15, 1, 3, (768, 24), "signed", 1306, 0.1315, 0.5, 31),     # queue 1000 = 7*128 + 104, nb = 200
    "uneq":  (64, 192, 103, 9, 3, 7, (384, 128), "random", 1442, 0.2609, 0.95, 31),   # bs != btu, btu > 128: two M tiles
    "tiny":  (5, 7, 7, 2, 1, 2, (37, 3), "random", 1452, 0.7496, 0.95, 31),             # nb = 12, B = 7, btu < 32, queue 50
    "cold":  (128, 128, 103, 9, 0, 5, (0, 0), "zero", 1418, 0.1873, 0.95, 31),          # smoothing off, zero banks: a run's start
}, 11: {  # thr: the widest gap of each step's scores (thr_for); the nets from the case's seed
    "k9_b103":  (128, 128, 103, 9, 1, 10, (512, 768), "random", 2101),
    "k16_b224": (128, 128, 224, 16, 2, 3, (256, 1024), "random", 2102),     # BASELINE configs[4]'s spectrum
    "k32_b224": (128, 128, 224, 32, 1, 40, (1024, 256), "random", 2103),
    "uneq":     (64, 192, 103, 9, 3, 7, (384, 128), "random", 2104),        # bs != btu, two M tiles
    "tiny":     (5, 7, 7, 2, 0, 2, (0, 0), "zero", 2105),                   # a run's cold start: smoothing off, zero banks
    "q1000":    (100, 100, 103, 9, 1, 3, (768, 24), "signed", 2106),        # 1000-row banks: partial last bank tile
}}
# q1000: signed bank features (similarities near 0, so every bank row weighs ~1 in the exp sums) and alpha = 0.5 make
# the 24 padded columns of the last bank tile a visible error if they were counted.
# The w = 20 thresholds sit in a wide gap between the oracle's scores (>= 0.4 % of thr away from every one of them), so
# that the fp16-operand probabilities cannot flip a mask bit.


@pytest.mark.parametrize("w,case", [pytest.param(w, c, id=c if w == 20 else c + "_w11")
                                    for w in SHAPES for c in SHAPES[w]])
def test_one_step_shapes(dev, golden_dir, w, case):
    one_step_against_oracle(dev, golden_dir, w, *SHAPES[w][case])


# ---------------------------------------------------------------------------------------------- B. consecutive steps
def test_consecutive_steps_graph_replay(dev, golden_dir):
    """Eight 128 + 128 steps of one FusedMutualStep replayed as a CUDA graph at 103 bands / 9 classes, re-anchored on
    the oracle before every step (fused_step_harness.eight_steps_graph_replay)."""
    eight_steps_graph_replay(dev, golden_dir, 20, 103, 9, 42, 4242)


# -------------------------------------------------------------------------------------- C. fp16 range of the backward
def test_trained_weights_full_bars(dev, golden_dir):
    """One 128 + 128 step from the weights the reference itself trained (train_infer.npz): realistic magnitudes
    through the fp16 operands, against the oracle at the full bars."""
    B, K, bs = 103, 9, 128
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    sd = {k[3:]: torch.from_numpy(np.array(v)) for k, v in ti.items() if k.startswith("sd.")}
    sd1 = {k: v.clone() for k, v in sd.items()}
    g = torch.Generator().manual_seed(606)
    inp = make_inputs(ti, bs, bs, B, K, g)
    sa = O.StepArgs(num_epochs=20)
    sa.thr = 0.2963
    ost = O.make_state(sd, sd1, K, sa)
    queues = random_banks(1280, K, g)
    set_banks(ost, queues, (256, 512))
    ost_before = copy.deepcopy(ost)
    r = oracle_step(ost, inp, 2, 11, sa)
    assert_soft_ce_exercised(r)
    fs = fused_for(dev, sd, sd1, bs, bs, B, K, queues, (256, 512), sa)
    w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
    hist, patches = fused_step(fs, dev, inp, 2, 11, sa.noise)
    r = on_fused_masks(r, ost_before, inp, 2, 11, sa, fs, 2 * bs)
    compare_with_oracle(fs, hist, r, ost, w_before, patches, 2 * bs)
    print("trained weights: fp16 headroom", headroom(fs, 2 * bs))


def headroom(fs, nb):
    """max|plane| / 65504 of the scaled fp16 data-gradient planes dz1 and da0."""
    lay, ws, ns = fs.workspace_layout(), fs.work, 2 * nb
    return {k: float(planes_to_nchw(ws[lay[k]:], ns, 400, 20).abs().max()) / FP16_MAX for k in ("dz1", "da0")}


@pytest.mark.parametrize("conv_scale,cls_conv_scale", [(4.0, 1.0), (8.0, 1.0), (16.0, 1.0), (1.0, 1e-4)],
                         ids=["conv_x4", "conv_x8", "conv_x16", "classifier_conv_cols_1e-4"])
def test_backward_fp16_range(dev, golden_dir, conv_scale, cls_conv_scale):
    """conv1 / conv2 weights of both nets scaled by 4-16 (the data-gradient planes dz1 / da0 grow with the 3x3 weight
    magnitudes while the gradient scale is chosen from max|dL/dcat| alone), or the classifier's conv columns scaled by
    1e-4 (max|dL/dcat| at the small end): every conv-backward kernel still holds the linearised bar and nothing in the
    gradients, the updated weights or the fp16 planes is inf / NaN."""
    B, K, bs = 103, 9, 128
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    torch.manual_seed(51)
    sds = [O.basenet2_init(B, K), O.basenet2_init(B, K)]
    for sd in sds:
        sd["conv1.weight"] *= conv_scale
        sd["conv2.weight"] *= conv_scale
        sd["classifier.weight"][:, :1600] *= cls_conv_scale
    g = torch.Generator().manual_seed(707)
    inp = make_inputs(ti, bs, bs, B, K, g)
    sa = O.StepArgs(num_epochs=20)
    sa.thr = 0.2
    fs = fused_for(dev, sds[0], sds[1], bs, bs, B, K, random_banks(1280, K, g), (0, 256), sa)
    w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
    hist, _ = fused_step(fs, dev, inp, 1, 0, sa.noise)
    torch.cuda.synchronize()
    nb, ns = 2 * bs, 4 * bs
    lay = fs.workspace_layout()
    dcat = fs.work[lay["dcat"]:lay["dcat"] + ns * 2624 * 4].view(torch.float32).view(ns, 2624)[:, :1600]
    room = headroom(fs, nb)
    print("conv weights x%g, classifier conv columns x%g: max|dL/dcat| %.2e, gradient scale 2^%d, "
          "max|dz1*S|/65504 %.3f, max|da0*S|/65504 %.3f" % (conv_scale, cls_conv_scale, float(dcat.abs().max()),
                                                         round(math.log2(fs.grad_scale())), room["dz1"], room["da0"]))
    for k in ("dz1", "da0"):
        assert torch.isfinite(planes_to_nchw(fs.work[lay[k]:], ns, 400, 20)).all(), k
    assert torch.isfinite(hist).all()
    for e in range(2):
        for i in range(10):
            assert torch.isfinite(fs.grads[e][i]).all() and torch.isfinite(fs.params[e][i]).all(), (e, i)
    linearised_check(fs, w_before, nb)
