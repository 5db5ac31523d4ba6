"""The fused training step's test harness, for both windows: inputs and oracle plumbing, read-back of the step's saved
tensors, and the bars every fused-step test holds (test_gpu_fused_step.py's module docstring states them).  Imported
as a plain module (pytest puts tests/ on sys.path); it holds no tests.

Everything that depends on the window goes through GEOMETRY.  At w = 11 the pools floor 11 -> 5 -> 2 and drop the last
row and column of conv1's and conv2's maps: no gradient reaches them, so the kernels store their mask bits and dz1
entries as 0, and the checks compare the kept positions with fp32 and the dropped ones with what the floor pool
implies.  At w = 20 nothing is dropped.
"""
import copy
import math
import os
from typing import NamedTuple

import numpy as np
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O
from oracle import golden
from scene_harness import rel

HEAD = ("feat_spe.weight", "feat_spe.bias", "classifier.weight", "classifier.bias")
CONV = ("conv0.weight", "conv0.bias", "conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias")
NOISE_KEYS = ("xp_l1", "x_l1", "xp_l2", "x_l2", "xp_u1", "x_u1", "xp_u2", "x_u2")
DROP_P = 0.8


class Geometry(NamedTuple):
    W: int          # conv0 / conv1 map side
    H2: int         # conv2 map side (conv1's map pooled)
    P2: int         # conv2's map pooled
    CONVF: int      # conv features, 64 * P2 * P2
    CAT: int        # classifier inputs: CONVF + 1024 spectral features


GEOMETRY = {20: Geometry(20, 10, 5, 1600, 2624), 11: Geometry(11, 5, 2, 256, 1280)}


def kept(side):
    """Rows (columns) of a side x side map that the floor pool reads."""
    return side - (side & 1)


# ------------------------------------------------------------------------------------------------ inputs and oracle
def make_inputs(ti, bs, btu, B, K, g, w=20):
    """Patches from the PCA cube (odd-mode windows at odd w), spectra (the fixture's when B matches, else N(0,1)),
    labels, the eight noise tensors and the two scaled dropout masks (p = 0.8) over the classifier inputs of one step."""
    Xp, Xs = ti["cube_pca"], ti["spectra"]
    R, C = Xp.shape[:2]
    li = torch.randint(0, R * C, (bs,), generator=g).numpy()
    ui = torch.randint(0, R * C, (btu,), generator=g).numpy()
    XP_l = torch.from_numpy(O.extract_patches_at(Xp, w, li, odd_mode=bool(w & 1)))
    XP_u = torch.from_numpy(O.extract_patches_at(Xp, w, ui, odd_mode=bool(w & 1)))
    if B == Xs.shape[1]:
        X_l, X_u = torch.from_numpy(Xs[li]), torch.from_numpy(Xs[ui])
    else:
        X_l, X_u = torch.randn(bs, B, generator=g), torch.randn(btu, B, generator=g)
    Y_l = torch.randint(0, K, (bs,), generator=g)
    shapes = dict(xp_l=XP_l.shape, x_l=X_l.shape, xp_u=XP_u.shape, x_u=X_u.shape)
    nz = {k: torch.randn(shapes[k[:-1]], generator=g) for k in NOISE_KEYS}
    cat = GEOMETRY[w].CAT
    masks = torch.stack([(torch.rand(bs + btu, cat, generator=g) >= DROP_P).float() / (1 - DROP_P) for _ in range(2)])
    return dict(XP_l=XP_l, X_l=X_l, Y_l=Y_l, XP_u=XP_u, X_u=X_u, nz=nz, masks=masks)


def assembled(inp, noise):
    """The noisy inputs of both nets as FusedMutualStep's assembled mode takes them (train.py:157-184)."""
    nz = inp["nz"]
    cat = lambda lab, unl, kl, ku: torch.cat([inp[lab] + nz[kl] * noise, inp[unl] + nz[ku] * noise], 0)
    patches = torch.stack([cat("XP_l", "XP_u", "xp_l1", "xp_u1"), cat("XP_l", "XP_u", "xp_l2", "xp_u2")])
    spectra = torch.stack([cat("X_l", "X_u", "x_l1", "x_u1"), cat("X_l", "X_u", "x_l2", "x_u2")])
    return patches.contiguous(), spectra.contiguous()


def init_nets(B, K, seed, w=20):
    torch.manual_seed(seed)
    convf = GEOMETRY[w].CONVF
    return O.basenet2_init(B, K, conv_feat=convf), O.basenet2_init(B, K, conv_feat=convf)


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
    64 + 192 rows or eight steps in a row reach 3.0-3.4e-2.  Conditioned on the masks, the bar measures the step.  The
    stored 0 bits of an odd map's dropped row / column change nothing: the floor pools never read those positions."""
    m1, m2 = relu_masks(fs, nb)
    masks = tuple((m1[e * nb:(e + 1) * nb], m2[e * nb:(e + 1) * nb]) for e in range(2))
    rf = oracle_step(copy.deepcopy(ost_before), inp, epoch, batch_index, sa, relu_masks=masks)
    return dict(r, grads=rf["grads"], grads1=rf["grads1"])


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


def thr_in_widest_gap(r):
    """A threshold (epoch 0: adap_thr = thr) in the widest gap between the middle half of this step's scores of both
    nets: a real split of the rows, and no score within reach of the fp16-operand error."""
    s = np.sort(np.concatenate([r["probs"].max(1)[0].numpy(), r["probs1"].max(1)[0].numpy()]).astype(np.float64))
    lo, hi = len(s) // 4, 3 * len(s) // 4
    i = lo + int(np.argmax(s[lo + 1:hi + 1] - s[lo:hi]))
    return float(0.5 * (s[i] + s[i + 1]))


def thr_for(r, epoch, num_epochs):
    """args.thr whose adaptive threshold at ``epoch`` sits in the widest gap of this step's scores."""
    return thr_in_widest_gap(r) / math.exp(-0.5 * ((epoch / num_epochs) ** 2))


def assert_soft_ce_exercised(r):
    # 5-95 % of the unlabelled rows of each net pass the adaptive threshold
    for m in (r["mask"], r["masks"]):
        assert 0.05 <= float(m.mean()) <= 0.95, float(m.mean())


# ------------------------------------------------------------------------------------------------------ the fused step
def make_fused(dev, sd, sd1, B, K, queues, w=20, **kw):
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.tools.models import BaseNet2
    nets = [BaseNet2(B, 0, K, w=w).to(dev) for _ in range(2)]
    nets[0].load_state_dict({k: v.detach() for k, v in sd.items()}, strict=False)
    nets[1].load_state_dict({k: v.detach() for k, v in sd1.items()}, strict=False)
    fs = FusedMutualStep(nets[0], nets[1], **kw)
    for dst, src in zip((fs.queue_feats[0], fs.queue_probs[0], fs.queue_feats[1], fs.queue_probs[1]), queues):
        dst.copy_(src)
    assert fs.w == w and fs.cat == GEOMETRY[w].CAT
    return fs


def fused_for(dev, sd, sd1, bs, btu, B, K, queues, ptrs, sa, w=20, **kw):
    fs = make_fused(dev, sd, sd1, B, K, queues, w, bs=bs, btu=btu, thr=sa.thr, num_epochs=sa.num_epochs, lr=sa.lr,
                    temperature=sa.temperature, alpha=sa.alpha, queue_batch=sa.queue_batch, dropout=DROP_P, **kw)
    fs.queue_ptr, fs.queue_ptr1 = ptrs
    return fs


def fused_step(fs, dev, inp, epoch, batch_index, noise):
    patches, spectra = assembled(inp, noise)
    patches, spectra = patches.to(dev), spectra.to(dev)
    hist = fs.step(inp["Y_l"].to(dev), epoch, batch_index, patches=patches, spectra=spectra,
                   drop_masks=inp["masks"].to(dev))
    return hist, patches


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


# ---------------------------------------------------------------------------------------------------------- read-back
def planes_to_nchw(buf, ns, npos, h):
    t = buf.view(torch.float16)[: ns * 8 * npos * 8].view(ns, 8, npos, 8).float()
    return t.permute(0, 1, 3, 2).reshape(ns, 64, h, h)


def bits_to_mask(buf, ns, npos, h):
    w = buf.view(torch.int32)[: ns * npos * 2].view(ns, npos, 2).cpu().numpy().astype(np.uint32)
    bits = ((w[..., None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(ns, npos, 64)
    return torch.from_numpy(bits.astype(np.float32)).permute(0, 2, 1).reshape(ns, 64, h, h)


def relu_masks(fs, nb):
    """The trunk ReLU masks the forward stored, on the host: conv1's [2 nb, 64, W, W] and conv2's [2 nb, 64, H2, H2]."""
    gm, lay, ns = GEOMETRY[fs.w], fs.workspace_layout(), 2 * nb
    return (bits_to_mask(fs.work[lay["m1"]:], ns, gm.W * gm.W, gm.W),
            bits_to_mask(fs.work[lay["m2"]:], ns, gm.H2 * gm.H2, gm.H2))


def saved(fs, nb):
    """The step's saved tensors read back at the window's per-sample strides (include/cmlpl.h); dz1 and da0 unscaled."""
    gm, lay, ws, ns = GEOMETRY[fs.w], fs.workspace_layout(), fs.work, 2 * nb
    S = fs.grad_scale()
    f32 = lambda k: ws[lay[k]:lay[k] + ns * gm.CAT * 4].view(torch.float32).view(ns, gm.CAT)
    planes = lambda k, h: planes_to_nchw(ws[lay[k]:], ns, h * h, h)
    m1, m2 = relu_masks(fs, nb)
    return dict(S=S, x16=planes("x16", gm.W), a0=planes("a0", gm.W), p1=planes("p1", gm.H2), m1=m1.to(fs.dev),
                m2=m2.to(fs.dev), cat=f32("cat"), dmask=f32("dmask"), dcat=f32("dcat"), dz1=planes("dz1", gm.W) / S,
                da0=planes("da0", gm.W) / S)


def pool_bwd(d, side):
    """avg_pool2d(2, 2) backward with floor semantics: each pooled gradient / 4 to its four inputs, 0 to the dropped
    last row / column of an odd map."""
    up = F.interpolate(d, scale_factor=2, mode="nearest") * 0.25
    return F.pad(up, (0, side - up.shape[-1], 0, side - up.shape[-2]))


# --------------------------------------------------------------------------------------------------------------- bars
def linearised_check(fs, w_before, nb, bar=1e-3):
    """Every convolution-backward kernel against torch fp32 on the kernel's own inputs."""
    gm, t, ns = GEOMETRY[fs.w], saved(fs, nb), 2 * nb
    dz2 = pool_bwd(t["dcat"][:, :gm.CONVF].reshape(ns, 64, gm.P2, gm.P2), gm.H2) * t["m2"]
    worst = {}
    for e in range(2):
        sl = slice(e * nb, (e + 1) * nb)
        W0, W1, W2 = w_before[e]["conv0.weight"], w_before[e]["conv1.weight"], w_before[e]["conv2.weight"]
        dp1 = F.conv_transpose2d(dz2[sl], W2, padding=1) + dz2[sl]                      # models.py:137-139 backward
        dz1 = pool_bwd(dp1, gm.W) * t["m1"][sl]                                         # :136 pool, :135 ReLU backward
        da0 = F.conv_transpose2d(t["dz1"][sl], W1, padding=1) + t["dz1"][sl]            # :133-135 backward
        g = dict(zip(CONV, [fs.grads[e][i] for i in range(6)]))
        errs = {
            "dz1": rel(t["dz1"][sl], dz1), "da0": rel(t["da0"][sl], da0),
            "conv2.weight": rel(g["conv2.weight"], torch.nn.grad.conv2d_weight(t["p1"][sl], W2.shape, dz2[sl], padding=1)),
            "conv2.bias": rel(g["conv2.bias"], dz2[sl].sum((0, 2, 3))),
            "conv1.weight": rel(g["conv1.weight"], torch.nn.grad.conv2d_weight(t["a0"][sl], W1.shape, t["dz1"][sl], padding=1)),
            "conv1.bias": rel(g["conv1.bias"], t["dz1"][sl].sum((0, 2, 3))),
            "conv0.weight": rel(g["conv0.weight"], torch.nn.grad.conv2d_weight(t["x16"][sl, :60], W0.shape, t["da0"][sl])),
            "conv0.bias": rel(g["conv0.bias"], t["da0"][sl].sum((0, 2, 3))),
        }
        for k, v in errs.items():
            worst[k] = max(worst.get(k, 0.0), v)
    print("linearised backward errors:", {k: f"{v:.1e}" for k, v in worst.items()})
    for k, v in worst.items():
        assert v < bar, (k, v)


def mask_flips(fs, sds, patches, nb):
    """Kept-position ReLU-mask bits that differ between the fp16-operand forward and torch fp32 (count, and fraction of
    all kept bits); the bits of an odd map's dropped row / column must be stored as 0."""
    m1, m2 = relu_masks(fs, nb)
    k1, k2 = kept(m1.shape[-1]), kept(m2.shape[-1])
    for m, k in ((m1, k1), (m2, k2)):
        assert float(m[:, :, k:, :].abs().sum() + m[:, :, :, k:].abs().sum()) == 0.0       # empty at an even side
    flips = 0
    for e in range(2):
        sd = sds[e]
        a0 = F.conv2d(patches[e], sd["conv0.weight"], sd["conv0.bias"])
        a1 = F.relu(F.conv2d(a0, sd["conv1.weight"], sd["conv1.bias"], padding=1) + a0)
        p1 = F.avg_pool2d(a1, 2, 2)
        a2 = F.relu(F.conv2d(p1, sd["conv2.weight"], sd["conv2.bias"], padding=1) + p1)
        flips += int(((a1 > 0).float().cpu()[:, :, :k1, :k1] != m1[e * nb:(e + 1) * nb, :, :k1, :k1]).sum())
        flips += int(((a2 > 0).float().cpu()[:, :, :k2, :k2] != m2[e * nb:(e + 1) * nb, :, :k2, :k2]).sum())
    return flips, flips / float(m1[:, :, :k1, :k1].numel() + m2[:, :, :k2, :k2].numel())


def compare_with_oracle(fs, hist, r, ost, w_before, patches, nb, adam=True):
    """The step-1 bars.  ``adam=False`` skips the Adam block, which compares against the oracle's update from ITS
    gradients and is only sound from a fresh Adam state (later steps: check_adam_exact)."""
    from cmlpl_b200.fused_step import TENSORS
    h = hist.cpu().numpy()
    want = np.array([r["hist"][0], r["hist"][1], r["hist"][2], r["hist"][3], r["hist"][4], r["total1"], r["cls1"],
                     r["con1"], r["lc1"]])
    assert np.abs(h[:9] - want).max() <= 1e-3 * np.abs(want).max(), (h[:9], want)
    assert rel(fs.logits[0], r["logits"]) < 1e-3 and rel(fs.logits[1], r["logits1"]) < 1e-3
    assert rel(fs.feat[0], r["feat"]) < 1e-5 and rel(fs.feat[1], r["feat1"]) < 1e-5          # fp32 branch
    assert rel(fs.probs[0], r["probs"]) < 1e-3 and rel(fs.probs[1], r["probs1"]) < 1e-3
    # the threshold compares a max-probability with a constant: allow a flip only where the oracle's own score is
    # within 1e-3 of the threshold
    for got, ref_mask, p in ((fs.mask[0], r["mask"], r["probs"]), (fs.mask[1], r["masks"], r["probs1"])):
        for i in (got.cpu() != ref_mask).nonzero().flatten().tolist():
            assert abs(float(p[i].max()) - fs.prm.adap_thr) < 1e-3 * fs.prm.adap_thr
    flips, frac = mask_flips(fs, w_before, patches, nb)
    print("ReLU mask bits differing from the fp32 forward: %d (%.2e of all kept bits)" % (flips, frac))
    assert frac < 1e-4
    g, g1 = r["grads"], r["grads1"]
    errs = [{k: rel(fs.grads[e][i], (g, g1)[e][k]) for i, k in enumerate(TENSORS)} for e in range(2)]
    print("gradient errors vs the fp32 oracle:", [{k: f"{v:.1e}" for k, v in d.items()} for d in errs])
    for d in errs:
        for k in HEAD:
            assert d[k] < 1e-3, (k, d[k])
        for k in CONV:
            assert d[k] < 3e-2, (k, d[k])
    linearised_check(fs, w_before, nb)
    # Adam: compare where the gradient is not ~0 (the first step moves every weight by ~lr*sign(g))
    for e, sd_new in enumerate((ost.sd, ost.sd1) if adam else ()):
        for i, k in enumerate(TENSORS):
            gr = (g, g1)[e][k].numpy()
            sel = np.abs(gr) > 5e-2 * np.abs(gr).max()
            new = fs.params[e][i].detach().cpu().numpy()
            assert np.abs(new - sd_new[k].detach().numpy())[sel].max() < 2e-5, k
    # memory banks (incl. the queue_ptr1 quirk, train.py:237)
    assert (fs.queue_ptr, fs.queue_ptr1) == (ost.queue_ptr, ost.queue_ptr1)
    for t, (qf, qp) in enumerate(((ost.queue_feats, ost.queue_probs), (ost.queue_feats1, ost.queue_probs1))):
        assert rel(fs.queue_feats[t], qf) < 1e-5 and rel(fs.queue_probs[t], qp) < 1e-3


# ---------------------------------------------------------------------------------------------------------- scenarios
def one_step_against_oracle(dev, golden_dir, w, bs, btu, B, K, epoch, batch_index, ptrs, banks, seed, thr=None,
                            alpha=0.95, net_seed=None):
    """One step of a FusedMutualStep built at exactly the batch it runs (so workspace_layout() is the layout the kernels
    used), against the oracle's ref_step on the fused forward's ReLU masks at the step-1 bars.  ``banks``: "zero",
    "random" or "signed" bank features; ``thr`` None: the threshold in the widest gap of the step's scores (thr_for);
    ``net_seed`` None: ``seed``."""
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    g = torch.Generator().manual_seed(seed)
    inp = make_inputs(ti, bs, btu, B, K, g, w)
    sd, sd1 = init_nets(B, K, seed if net_seed is None else net_seed, w)
    sa = O.StepArgs(num_epochs=20, labeled_batch_size=bs)
    sa.alpha = alpha
    ost = O.make_state(sd, sd1, K, sa)
    queue = 5 * bs * 2                                                     # train.py:138
    if banks == "zero":
        queues = [torch.zeros_like(t) for t in (ost.queue_feats, ost.queue_probs) * 2]
    else:
        queues = random_banks(queue, K, g, signed=banks == "signed")
    set_banks(ost, queues, ptrs)
    smooth = epoch > 0 or batch_index > sa.queue_batch
    assert smooth == (banks != "zero")
    sa.thr = thr_for(oracle_step(copy.deepcopy(ost), inp, epoch, batch_index, sa), epoch, sa.num_epochs) if thr is None else thr
    ost_before = copy.deepcopy(ost)
    r = oracle_step(ost, inp, epoch, batch_index, sa)
    assert_soft_ce_exercised(r)
    fs = fused_for(dev, sd, sd1, bs, btu, B, K, queues, ptrs, sa, w)
    assert fs.B == B and fs.queue == queue and fs.cur == (bs, btu)
    w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
    hist, patches = fused_step(fs, dev, inp, epoch, batch_index, sa.noise)
    assert fs.prm.smooth == int(smooth)
    r = on_fused_masks(r, ost_before, inp, epoch, batch_index, sa, fs, bs + btu)
    compare_with_oracle(fs, hist, r, ost, w_before, patches, bs + btu)


def eight_steps_graph_replay(dev, golden_dir, w, B, K, net_seed, seed):
    """Eight 128 + 128 steps (epoch 0, batch 0..7, queue_batch 3) of one FusedMutualStep captured once as a CUDA graph
    and replayed on new inputs copied into the same tensors.  Before every step the oracle is re-anchored on the fused
    state, so each step is judged on its own: bank smoothing switches on at batch 4, the bank pointer wraps at 1280
    (with the queue_ptr1 quirk), and Adam runs with carried moments and the bias corrections of steps 2..8, checked
    exactly against float64."""
    bs = 128
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    sd, sd1 = init_nets(B, K, net_seed, w)
    sa = O.StepArgs(num_epochs=20, queue_batch=3)
    zero = [torch.zeros(1280, 1024), torch.zeros(1280, K)] * 2
    fs = fused_for(dev, sd, sd1, bs, bs, B, K, zero, (0, 0), sa, w, use_graph=True)
    patches = torch.zeros(2, 2 * bs, 60, w, w, device=dev)
    spectra = torch.zeros(2, 2 * bs, B, device=dev)
    masks = torch.zeros(2, 2 * bs, GEOMETRY[w].CAT, device=dev)
    labels = torch.zeros(bs, dtype=torch.int64, device=dev)
    g = torch.Generator().manual_seed(seed)
    seen = []
    for it in range(8):
        inp = make_inputs(ti, bs, bs, B, K, g, w)
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
        compare_with_oracle(fs, hist, r, ost, w_before, patches, 2 * bs, adam=it == 0)
        worst = check_adam_exact(fs, before, it + 1)
        seen.append((ptrs, (fs.queue_ptr, fs.queue_ptr1), float(r["mask"].mean()), worst))
        print("step %d: pointers %s -> %s, mask fraction %.2f, Adam max rel error %.1e" % (it + 1, *seen[-1]))
        assert 0.05 <= seen[-1][2] <= 0.95
    # the pointer sequence crossed the end of the 1280-row bank and restarted at 0 (train.py:234-237)
    assert [s[0][0] for s in seen] == [0, 256, 512, 768, 1024, 0, 256, 512]


def cube_mode_steps(nets, sd0, labels, cube, pix, spectra, noise, graph, steps=1, seed=1088):
    """``steps`` steps of a FusedMutualStep over ``nets`` reset to ``sd0``, in cube mode (inputs gathered from the PCA
    cube in the first kernel, noise and dropout from the device Philox stream at ``seed``).  Per step: the fp16 input
    planes, logits, loss history, dropout masks, noisy spectra and net 0's parameters."""
    from cmlpl_b200.fused_step import FusedMutualStep
    for n, s in zip(nets, sd0):
        n.load_state_dict(s)
    fs = FusedMutualStep(nets[0], nets[1], noise=noise, seed=seed, use_graph=graph, thr=0.5)
    gm, ns, B = GEOMETRY[fs.w], 2 * pix.numel(), fs.B
    out, pix_d = [], pix.to(cube.device)
    for it in range(steps):
        fs.step(labels, 1, it, cube=cube, pix=pix_d, spectra=spectra)
        lay = fs.workspace_layout()
        out.append(dict(x16=planes_to_nchw(fs.work[lay["x16"]:], ns, gm.W * gm.W, gm.W).clone(), logits=fs.logits.clone(),
                        hist=fs.hist.clone(),
                        dmask=fs.work[lay["dmask"]:lay["dmask"] + ns * gm.CAT * 4].view(torch.float32).clone(),
                        y=fs.work[lay["ynoisy"]:lay["ynoisy"] + ns * B * 4].view(torch.float32).view(ns, B).clone(),
                        w=[p.detach().clone() for p in fs.params[0]]))
    return out, fs
