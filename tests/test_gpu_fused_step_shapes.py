"""GPU parity of the fused training step (cmlpl_train_step) beyond the 128 + 128 / 9-16-class shapes of
test_gpu_fused_step.py, with the same bars (its module docstring).  The gradients are compared with the oracle's on
the fused forward's own ReLU masks (on_fused_masks); the masks themselves are compared with fp32's and bounded.

  * a shape matrix, one step each against the oracle's ref_step: 17-32 classes (every <32> instantiation of the head
    and loss kernels, sim_tc_kernel's C > 16 branch), 256 bands, banks that end in a partial 128-row tile, bs != btu,
    btu > 128 and btu < 32, and the first steps of a run (bank smoothing off, zero banks);
  * eight consecutive steps through one FusedMutualStep replayed as a CUDA graph, re-anchored on the oracle before
    every step: smoothing switching on, the bank pointers wrapping, and Adam at steps 2..8 checked exactly;
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

from oracle import cmlpl_oracle as O
from oracle import golden
from test_gpu_fused_step import bits_to_mask, compare_with_oracle, linearised_check, make_fused, planes_to_nchw

pytestmark = pytest.mark.gpu

DROP_P = 0.8
NOISE_KEYS = ("xp_l1", "x_l1", "xp_l2", "x_l2", "xp_u1", "x_u1", "xp_u2", "x_u2")
FP16_MAX = 65504.0


def make_inputs(ti, bs, btu, B, K, g):
    """Patches from the PCA cube, spectra (the fixture's when B matches, else N(0,1)), labels, the eight noise tensors
    and the two scaled dropout masks (p = 0.8) of one step."""
    Xp, Xs = ti["cube_pca"], ti["spectra"]
    R, C = Xp.shape[:2]
    li = torch.randint(0, R * C, (bs,), generator=g).numpy()
    ui = torch.randint(0, R * C, (btu,), generator=g).numpy()
    XP_l = torch.from_numpy(O.extract_patches_at(Xp, 20, li))
    XP_u = torch.from_numpy(O.extract_patches_at(Xp, 20, ui))
    if B == Xs.shape[1]:
        X_l, X_u = torch.from_numpy(Xs[li]), torch.from_numpy(Xs[ui])
    else:
        X_l, X_u = torch.randn(bs, B, generator=g), torch.randn(btu, B, generator=g)
    Y_l = torch.randint(0, K, (bs,), generator=g)
    shapes = dict(xp_l=XP_l.shape, x_l=X_l.shape, xp_u=XP_u.shape, x_u=X_u.shape)
    nz = {k: torch.randn(shapes[k[:-1]], generator=g) for k in NOISE_KEYS}
    masks = torch.stack([(torch.rand(bs + btu, 2624, generator=g) >= DROP_P).float() / (1 - DROP_P) for _ in range(2)])
    return dict(XP_l=XP_l, X_l=X_l, Y_l=Y_l, XP_u=XP_u, X_u=X_u, nz=nz, masks=masks)


def assembled(inp, noise):
    """The noisy inputs of both nets as FusedMutualStep's assembled mode takes them (train.py:157-184)."""
    nz = inp["nz"]
    cat = lambda lab, unl, kl, ku: torch.cat([inp[lab] + nz[kl] * noise, inp[unl] + nz[ku] * noise], 0)
    patches = torch.stack([cat("XP_l", "XP_u", "xp_l1", "xp_u1"), cat("XP_l", "XP_u", "xp_l2", "xp_u2")])
    spectra = torch.stack([cat("X_l", "X_u", "x_l1", "x_u1"), cat("X_l", "X_u", "x_l2", "x_u2")])
    return patches.contiguous(), spectra.contiguous()


def random_banks(queue, K, g, signed=False):
    feats = lambda: O.normalize(torch.randn(queue, 1024, generator=g) if signed else torch.randn(queue, 1024, generator=g).abs())
    return [feats(), torch.softmax(torch.randn(queue, K, generator=g) * 2, 1),
            feats(), torch.softmax(torch.randn(queue, K, generator=g) * 2, 1)]


def set_banks(ost, queues, ptrs):
    for dst, src in zip((ost.queue_feats, ost.queue_probs, ost.queue_feats1, ost.queue_probs1), queues):
        dst.copy_(src)
    ost.queue_ptr, ost.queue_ptr1 = ptrs


def oracle_step(ost, inp, epoch, batch_index, sa, **kw):
    return O.ref_step(ost, inp["XP_l"], inp["X_l"], inp["Y_l"], inp["XP_u"], inp["X_u"], inp["nz"], epoch=epoch,
                      batch_index=batch_index, args=sa, drop_masks=tuple(inp["masks"]), **kw)


def on_fused_masks(r, ost_before, inp, epoch, batch_index, sa, fs, nb):
    """``r`` with the oracle's gradients replaced by those of the same step with the fused forward's trunk ReLU masks
    imposed.  Those masks differ from fp32's only where an activation is within ~2^-11 of zero (mask_flips counts them
    and bounds them at 1e-4 of all bits), yet one flip moves a conv weight gradient by a whole term: against the
    unconditioned oracle the end-to-end conv gradient bar measures how many flips landed where, and draws at
    64 + 192 rows or eight steps in a row reach 3.0-3.4e-2.  Conditioned on the masks, the bar measures the step."""
    lay, ws, ns = fs.workspace_layout(), fs.work, 2 * nb
    m1 = bits_to_mask(ws[lay["m1"]:], ns, 400, 20)
    m2 = bits_to_mask(ws[lay["m2"]:], ns, 100, 10)
    masks = tuple((m1[e * nb:(e + 1) * nb], m2[e * nb:(e + 1) * nb]) for e in range(2))
    rf = oracle_step(copy.deepcopy(ost_before), inp, epoch, batch_index, sa, relu_masks=masks)
    return dict(r, grads=rf["grads"], grads1=rf["grads1"])


def fused_for(dev, sd, sd1, bs, btu, B, K, queues, ptrs, sa, **kw):
    fs = make_fused(dev, sd, sd1, B, K, queues, bs=bs, btu=btu, thr=sa.thr, num_epochs=sa.num_epochs, lr=sa.lr,
                    temperature=sa.temperature, alpha=sa.alpha, queue_batch=sa.queue_batch, dropout=DROP_P, **kw)
    fs.queue_ptr, fs.queue_ptr1 = ptrs
    return fs


def fused_step(fs, dev, inp, epoch, batch_index, noise):
    patches, spectra = assembled(inp, noise)
    patches, spectra = patches.to(dev), spectra.to(dev)
    hist = fs.step(inp["Y_l"].to(dev), epoch, batch_index, patches=patches, spectra=spectra,
                   drop_masks=inp["masks"].to(dev))
    return hist, patches


def assert_soft_ce_exercised(r):
    # 5-95 % of the unlabelled rows of each net pass the adaptive threshold
    for m in (r["mask"], r["masks"]):
        assert 0.05 <= float(m.mean()) <= 0.95, float(m.mean())


# ---------------------------------------------------------------------------------------------------- A. shape matrix
#   id       bs   btu  B    K   thr     epoch batch (queue_ptr, queue_ptr1) banks   alpha  seed
SHAPES = {
    "k24":   (128, 128, 103, 24, 0.0829, 1, 10, (512, 768), "random", 0.95, 1209),  # every <32> kernel, sim_tc C > 16
    "k32":   (128, 128, 256, 32, 0.0987, 2, 40, (1024, 256), "random", 0.95, 1208), # the largest classes / bands the ABI takes
    "q1000": (100, 100, 144, 15, 0.1315, 1, 3, (768, 24), "signed", 0.5, 1306),     # queue 1000 = 7*128 + 104, nb = 200
    "uneq":  (64, 192, 103, 9, 0.2609, 3, 7, (384, 128), "random", 0.95, 1442),   # bs != btu, btu > 128: two M tiles
    "tiny":  (5, 7, 7, 2, 0.7496, 1, 2, (37, 3), "random", 0.95, 1452),             # nb = 12, B = 7, btu < 32, queue 50
    "cold":  (128, 128, 103, 9, 0.1873, 0, 5, (0, 0), "zero", 0.95, 1418),          # smoothing off, zero banks: a run's start
}
# q1000: signed bank features (similarities near 0, so every bank row weighs ~1 in the exp sums) and alpha = 0.5 make
# the 24 padded columns of the last bank tile a visible error if they were counted.
# thr sits in a wide gap between the oracle's scores (>= 0.4 % of thr away from every one of them), so that the
# fp16-operand probabilities cannot flip a mask bit


@pytest.mark.parametrize("case", list(SHAPES))
def test_one_step_shapes(dev, golden_dir, case):
    bs, btu, B, K, thr, epoch, batch_index, ptrs, banks, alpha, seed = SHAPES[case]
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    g = torch.Generator().manual_seed(seed)
    inp = make_inputs(ti, bs, btu, B, K, g)
    torch.manual_seed(31)
    sd, sd1 = O.basenet2_init(B, K), O.basenet2_init(B, K)
    sa = O.StepArgs(num_epochs=20, labeled_batch_size=bs)
    sa.thr, sa.alpha = thr, alpha
    ost = O.make_state(sd, sd1, K, sa)
    queue = 5 * bs * 2                                                     # train.py:138
    if banks == "zero":
        queues = [torch.zeros_like(t) for t in (ost.queue_feats, ost.queue_probs) * 2]
    else:
        queues = random_banks(queue, K, g, signed=banks == "signed")
    set_banks(ost, queues, ptrs)
    smooth = epoch > 0 or batch_index > sa.queue_batch
    assert smooth == (banks != "zero")
    ost_before = copy.deepcopy(ost)
    r = oracle_step(ost, inp, epoch, batch_index, sa)
    assert_soft_ce_exercised(r)
    fs = fused_for(dev, sd, sd1, bs, btu, B, K, queues, ptrs, sa)
    assert fs.queue == queue and fs.cur == (bs, btu)
    w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
    hist, patches = fused_step(fs, dev, inp, epoch, batch_index, sa.noise)
    assert fs.prm.smooth == int(smooth)
    r = on_fused_masks(r, ost_before, inp, epoch, batch_index, sa, fs, bs + btu)
    compare_with_oracle(fs, hist, r, ost, w_before, patches, bs + btu, w_before)


# ---------------------------------------------------------------------------------------------- B. consecutive steps
def oracle_state_of(fs, sa):
    """An oracle TrainState holding the fused step's current state: parameters, Adam moments and step, both banks and
    both pointers."""
    from cmlpl_b200.fused_step import TENSORS
    sds = [{k: fs.params[e][i].detach().cpu().clone().requires_grad_(True) for i, k in enumerate(TENSORS)} for e in range(2)]
    opts = [torch.optim.Adam(list(sd.values()), lr=sa.lr) for sd in sds]
    if fs.adam_step > 0:
        for e in range(2):
            for i, k in enumerate(TENSORS):
                opts[e].state[sds[e][k]] = {"step": torch.tensor(float(fs.adam_step)),
                                            "exp_avg": fs.ms[e][i].detach().cpu().clone(),
                                            "exp_avg_sq": fs.vs[e][i].detach().cpu().clone()}
    banks = [t.detach().cpu().clone() for t in (fs.queue_feats[0], fs.queue_probs[0], fs.queue_feats[1], fs.queue_probs[1])]
    return O.TrainState(sds[0], sds[1], opts[0], opts[1], *banks, queue_ptr=fs.queue_ptr, queue_ptr1=fs.queue_ptr1)


def snapshot_adam(fs):
    return [[(fs.params[e][i].detach().double().cpu(), fs.ms[e][i].double().cpu(), fs.vs[e][i].double().cpu())
             for i in range(10)] for e in range(2)]


def check_adam_exact(fs, before, step):
    """torch.optim.Adam's update (lerp form of _single_tensor_adam) in float64 on the fused step's OWN gradients, from
    the parameters and moments before the step: isolates adam_all_kernel (bias corrections of step `step`) from the
    precision of the gradients.  The constants are the float32 values the kernel reads."""
    f32 = lambda x: float(np.float32(x))
    b1, b2, lr, eps = f32(fs.betas[0]), f32(fs.betas[1]), f32(fs.lr), f32(fs.eps)
    bc1, bc2 = 1.0 - fs.betas[0] ** step, 1.0 - fs.betas[1] ** step
    worst = 0.0
    for e in range(2):
        for i in range(10):
            p0, m0, v0 = before[e][i]
            gr = fs.grads[e][i].double().cpu()
            m = m0 + (gr - m0) * (1.0 - b1)
            v = b2 * v0 + (1.0 - b2) * gr * gr
            p = p0 - (lr / bc1) * (m / (v.sqrt() / math.sqrt(bc2) + eps))
            for got, want in ((fs.params[e][i], p), (fs.ms[e][i], m), (fs.vs[e][i], v)):
                err = float((got.double().cpu() - want).abs().max() / max(float(want.abs().max()), 1e-30))
                worst = max(worst, err)
                assert err < 1e-6, (step, e, i, err)
    return worst


def thr_in_widest_gap(r):
    """A threshold (epoch 0: adap_thr = thr) in the widest gap between the middle half of this step's scores of both
    nets: a real split of the rows, and no score within reach of the fp16-operand error."""
    s = np.sort(np.concatenate([r["probs"].max(1)[0].numpy(), r["probs1"].max(1)[0].numpy()]).astype(np.float64))
    lo, hi = len(s) // 4, 3 * len(s) // 4
    i = lo + int(np.argmax(s[lo + 1:hi + 1] - s[lo:hi]))
    return float(0.5 * (s[i] + s[i + 1]))


def test_consecutive_steps_graph_replay(dev, golden_dir):
    """Eight 128 + 128 steps (epoch 0, batch 0..7, queue_batch 3) of one FusedMutualStep captured once as a CUDA graph
    and replayed on new inputs copied into the same tensors.  Before every step the oracle is re-anchored on the fused
    state, so each step is judged on its own: bank smoothing switches on at batch 4, the bank pointer wraps at 1280
    (with the queue_ptr1 quirk), and Adam runs with carried moments and the bias corrections of steps 2..8."""
    B, K, bs = 103, 9, 128
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    torch.manual_seed(42)
    sd, sd1 = O.basenet2_init(B, K), O.basenet2_init(B, K)
    sa = O.StepArgs(num_epochs=20, queue_batch=3)
    zero = [torch.zeros(1280, 1024), torch.zeros(1280, K)] * 2
    fs = fused_for(dev, sd, sd1, bs, bs, B, K, zero, (0, 0), sa, use_graph=True)
    patches = torch.zeros(2, 2 * bs, 60, 20, 20, device=dev)
    spectra = torch.zeros(2, 2 * bs, B, device=dev)
    masks = torch.zeros(2, 2 * bs, 2624, device=dev)
    labels = torch.zeros(bs, dtype=torch.int64, device=dev)
    g = torch.Generator().manual_seed(4242)
    seen = []
    for it in range(8):
        inp = make_inputs(ti, bs, bs, B, K, g)
        p_, s_ = assembled(inp, sa.noise)
        patches.copy_(p_); spectra.copy_(s_); masks.copy_(inp["masks"]); labels.copy_(inp["Y_l"])
        ost = oracle_state_of(fs, sa)
        before = snapshot_adam(fs)
        w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
        ptrs = (fs.queue_ptr, fs.queue_ptr1)
        ost_before = copy.deepcopy(ost)
        sa.thr = fs.thr = thr_in_widest_gap(oracle_step(copy.deepcopy(ost), inp, 0, it, sa))
        r = oracle_step(ost, inp, 0, it, sa)
        hist = fs.step(labels, 0, it, patches=patches, spectra=spectra, drop_masks=masks)
        assert fs.adam_step == it + 1 and len(fs._graphs) == 1
        assert fs.prm.smooth == int(it > 3)
        r = on_fused_masks(r, ost_before, inp, 0, it, sa, fs, 2 * bs)
        compare_with_oracle(fs, hist, r, ost, w_before, patches, 2 * bs, w_before, adam=it == 0)
        worst = check_adam_exact(fs, before, it + 1)
        seen.append((ptrs, (fs.queue_ptr, fs.queue_ptr1), float(r["mask"].mean()), worst))
        print("step %d: pointers %s -> %s, mask fraction %.2f, Adam max rel error %.1e" % (it + 1, *seen[-1]))
        assert 0.05 <= seen[-1][2] <= 0.95
    # the pointer sequence crossed the end of the 1280-row bank and restarted at 0 (train.py:234-237)
    assert [s[0][0] for s in seen] == [0, 256, 512, 768, 1024, 0, 256, 512]


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
    compare_with_oracle(fs, hist, r, ost, w_before, patches, 2 * bs, w_before)
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
