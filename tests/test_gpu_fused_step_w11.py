"""GPU parity of the fused training step at w = 11 (-m gpu): cmlpl_train_step on 11x11 windows (ExtractPatches_for_base,
pools flooring 11 -> 5 -> 2, a 1280-input classifier) against the oracle's ref_step, at the bars of
test_gpu_fused_step.py's module docstring:
  * logits / probabilities / losses / head gradients: 1e-3 * max|ref|;
  * every convolution-backward kernel against torch fp32 convolutions on the kernel's own saved tensors: 1e-3;
  * convolution gradients end to end against the fp32 oracle (on the fused forward's ReLU masks): 3e-2, with the mask
    bits that differ from fp32's counted and bounded.
The pools drop row / column 10 of conv1's map and row / column 4 of conv2's: no gradient reaches them, so the kernels
store their mask bits and dz1 entries as 0 and the checks here compare the kept positions with fp32 and the dropped
ones with what the floor pool implies.  The helpers of the w = 20 files hard-code 20 x 20 maps, so this file carries
w-generic versions of the ones it needs.
"""
import copy
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O
from oracle import golden
from test_gpu_fused_step import CONV, HEAD, bits_to_mask, planes_to_nchw, rel
from test_gpu_fused_step_shapes import (NOISE_KEYS, check_adam_exact, oracle_state_of, random_banks, set_banks,
                                        snapshot_adam, thr_in_widest_gap)

pytestmark = pytest.mark.gpu

W, H2, CAT, CONVF = 11, 5, 1280, 256
DROP_P = 0.8


# ------------------------------------------------------------------------------------------------------------ helpers
def make_inputs(ti, bs, btu, B, K, g):
    """Odd-mode 11x11 patches from the PCA cube, spectra (the fixture's when B matches, else N(0,1)), labels, the eight
    noise tensors and two scaled dropout masks (p = 0.8) over the 1280 classifier inputs."""
    Xp, Xs = ti["cube_pca"], ti["spectra"]
    R, C = Xp.shape[:2]
    li = torch.randint(0, R * C, (bs,), generator=g).numpy()
    ui = torch.randint(0, R * C, (btu,), generator=g).numpy()
    XP_l = torch.from_numpy(O.extract_patches_at(Xp, W, li, odd_mode=True))
    XP_u = torch.from_numpy(O.extract_patches_at(Xp, W, ui, odd_mode=True))
    if B == Xs.shape[1]:
        X_l, X_u = torch.from_numpy(Xs[li]), torch.from_numpy(Xs[ui])
    else:
        X_l, X_u = torch.randn(bs, B, generator=g), torch.randn(btu, B, generator=g)
    Y_l = torch.randint(0, K, (bs,), generator=g)
    shapes = dict(xp_l=XP_l.shape, x_l=X_l.shape, xp_u=XP_u.shape, x_u=X_u.shape)
    nz = {k: torch.randn(shapes[k[:-1]], generator=g) for k in NOISE_KEYS}
    masks = torch.stack([(torch.rand(bs + btu, CAT, generator=g) >= DROP_P).float() / (1 - DROP_P) for _ in range(2)])
    return dict(XP_l=XP_l, X_l=X_l, Y_l=Y_l, XP_u=XP_u, X_u=X_u, nz=nz, masks=masks)


def assembled(inp, noise):
    nz = inp["nz"]
    cat = lambda lab, unl, kl, ku: torch.cat([inp[lab] + nz[kl] * noise, inp[unl] + nz[ku] * noise], 0)
    patches = torch.stack([cat("XP_l", "XP_u", "xp_l1", "xp_u1"), cat("XP_l", "XP_u", "xp_l2", "xp_u2")])
    spectra = torch.stack([cat("X_l", "X_u", "x_l1", "x_u1"), cat("X_l", "X_u", "x_l2", "x_u2")])
    return patches.contiguous(), spectra.contiguous()


def oracle_step(ost, inp, epoch, batch_index, sa, **kw):
    return O.ref_step(ost, inp["XP_l"], inp["X_l"], inp["Y_l"], inp["XP_u"], inp["X_u"], inp["nz"], epoch=epoch,
                      batch_index=batch_index, args=sa, drop_masks=tuple(inp["masks"]), **kw)


def make_fused(dev, sd, sd1, B, K, queues, ptrs, sa, **kw):
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.tools.models import BaseNet2
    nets = [BaseNet2(B, 0, K, w=W).to(dev) for _ in range(2)]
    nets[0].load_state_dict({k: v.detach() for k, v in sd.items()}, strict=False)
    nets[1].load_state_dict({k: v.detach() for k, v in sd1.items()}, strict=False)
    kw.setdefault("dropout", DROP_P)
    fs = FusedMutualStep(nets[0], nets[1], thr=sa.thr, num_epochs=sa.num_epochs, lr=sa.lr, temperature=sa.temperature,
                         alpha=sa.alpha, queue_batch=sa.queue_batch, **kw)
    for dst, src in zip((fs.queue_feats[0], fs.queue_probs[0], fs.queue_feats[1], fs.queue_probs[1]), queues):
        dst.copy_(src)
    fs.queue_ptr, fs.queue_ptr1 = ptrs
    assert fs.w == W and fs.cat == CAT
    return fs


def saved(fs, nb):
    """The step's saved tensors read back at the w = 11 per-sample strides (include/cmlpl.h)."""
    lay, ws, ns = fs.workspace_layout(), fs.work, 2 * nb
    S = fs.grad_scale()
    f32 = lambda k, n: ws[lay[k]:lay[k] + ns * n * 4].view(torch.float32).view(ns, n)
    return dict(S=S, x16=planes_to_nchw(ws[lay["x16"]:], ns, W * W, W), a0=planes_to_nchw(ws[lay["a0"]:], ns, W * W, W),
                p1=planes_to_nchw(ws[lay["p1"]:], ns, H2 * H2, H2),
                m1=bits_to_mask(ws[lay["m1"]:], ns, W * W, W).to(fs.dev),
                m2=bits_to_mask(ws[lay["m2"]:], ns, H2 * H2, H2).to(fs.dev),
                cat=f32("cat", CAT), dmask=f32("dmask", CAT), dcat=f32("dcat", CAT),
                dz1=planes_to_nchw(ws[lay["dz1"]:], ns, W * W, W) / S, da0=planes_to_nchw(ws[lay["da0"]:], ns, W * W, W) / S)


def pool_bwd(d, side):
    """avg_pool2d(2, 2) backward with floor semantics: each pooled gradient / 4 to its four inputs, 0 to the dropped
    last row / column of an odd map."""
    up = F.interpolate(d, scale_factor=2, mode="nearest") * 0.25
    return F.pad(up, (0, side - up.shape[-1], 0, side - up.shape[-2]))


def linearised_check(fs, w_before, nb, bar=1e-3):
    """Every convolution-backward kernel against torch fp32 on the kernel's own inputs."""
    t = saved(fs, nb)
    ns = 2 * nb
    dz2 = pool_bwd(t["dcat"][:, :CONVF].reshape(ns, 64, 2, 2), H2) * t["m2"]
    worst = {}
    for e in range(2):
        sl = slice(e * nb, (e + 1) * nb)
        W0, W1, W2 = w_before[e]["conv0.weight"], w_before[e]["conv1.weight"], w_before[e]["conv2.weight"]
        dp1 = F.conv_transpose2d(dz2[sl], W2, padding=1) + dz2[sl]
        dz1 = pool_bwd(dp1, W) * t["m1"][sl]
        da0 = F.conv_transpose2d(t["dz1"][sl], W1, padding=1) + t["dz1"][sl]
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
    return t


def mask_flips(fs, sds, patches, nb):
    """Kept-position ReLU-mask bits that differ between the fp16-operand forward and torch fp32 (fraction of all kept
    bits); the bits of the dropped row / column must be stored as 0."""
    t = saved(fs, nb)
    m1, m2 = t["m1"].cpu(), t["m2"].cpu()
    assert float(m1[:, :, W - 1, :].abs().sum() + m1[:, :, :, W - 1].abs().sum()) == 0.0
    assert float(m2[:, :, H2 - 1, :].abs().sum() + m2[:, :, :, H2 - 1].abs().sum()) == 0.0
    flips = 0
    for e in range(2):
        sd = sds[e]
        a0 = F.conv2d(patches[e], sd["conv0.weight"], sd["conv0.bias"])
        a1 = F.relu(F.conv2d(a0, sd["conv1.weight"], sd["conv1.bias"], padding=1) + a0)
        p1 = F.avg_pool2d(a1, 2, 2)
        a2 = F.relu(F.conv2d(p1, sd["conv2.weight"], sd["conv2.bias"], padding=1) + p1)
        flips += int(((a1 > 0).float().cpu()[:, :, :W - 1, :W - 1] != m1[e * nb:(e + 1) * nb, :, :W - 1, :W - 1]).sum())
        flips += int(((a2 > 0).float().cpu()[:, :, :H2 - 1, :H2 - 1] != m2[e * nb:(e + 1) * nb, :, :H2 - 1, :H2 - 1]).sum())
    kept = m1[:, :, :W - 1, :W - 1].numel() + m2[:, :, :H2 - 1, :H2 - 1].numel()
    return flips, flips / float(kept)


def on_fused_masks(r, ost_before, inp, epoch, batch_index, sa, fs, nb):
    """``r`` with the oracle's gradients of the same step on the fused forward's trunk ReLU masks (see
    test_gpu_fused_step_shapes.on_fused_masks).  The stored 0 bits of the dropped row / column change nothing there:
    the floor pools never read those positions."""
    t = saved(fs, nb)
    m1, m2 = t["m1"].cpu(), t["m2"].cpu()
    masks = tuple((m1[e * nb:(e + 1) * nb], m2[e * nb:(e + 1) * nb]) for e in range(2))
    rf = oracle_step(copy.deepcopy(ost_before), inp, epoch, batch_index, sa, relu_masks=masks)
    return dict(r, grads=rf["grads"], grads1=rf["grads1"])


def compare_with_oracle(fs, hist, r, ost, w_before, patches, nb, adam=True):
    from cmlpl_b200.fused_step import TENSORS
    h = hist.cpu().numpy()
    want = np.array([r["hist"][0], r["hist"][1], r["hist"][2], r["hist"][3], r["hist"][4], r["total1"], r["cls1"],
                     r["con1"], r["lc1"]])
    assert np.abs(h[:9] - want).max() <= 1e-3 * np.abs(want).max(), (h[:9], want)
    assert rel(fs.logits[0], r["logits"]) < 1e-3 and rel(fs.logits[1], r["logits1"]) < 1e-3
    assert rel(fs.feat[0], r["feat"]) < 1e-5 and rel(fs.feat[1], r["feat1"]) < 1e-5
    assert rel(fs.probs[0], r["probs"]) < 1e-3 and rel(fs.probs[1], r["probs1"]) < 1e-3
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
    for e, sd_new in enumerate((ost.sd, ost.sd1) if adam else ()):
        for i, k in enumerate(TENSORS):
            gr = (g, g1)[e][k].numpy()
            sel = np.abs(gr) > 5e-2 * np.abs(gr).max()
            new = fs.params[e][i].detach().cpu().numpy()
            assert np.abs(new - sd_new[k].detach().numpy())[sel].max() < 2e-5, k
    assert (fs.queue_ptr, fs.queue_ptr1) == (ost.queue_ptr, ost.queue_ptr1)
    for t, (qf, qp) in enumerate(((ost.queue_feats, ost.queue_probs), (ost.queue_feats1, ost.queue_probs1))):
        assert rel(fs.queue_feats[t], qf) < 1e-5 and rel(fs.queue_probs[t], qp) < 1e-3


def init_nets(B, K, seed):
    torch.manual_seed(seed)
    return O.basenet2_init(B, K, conv_feat=CONVF), O.basenet2_init(B, K, conv_feat=CONVF)


def thr_for(r, epoch, num_epochs):
    """args.thr whose adaptive threshold at ``epoch`` sits in the widest gap of this step's scores."""
    return thr_in_widest_gap(r) / math.exp(-0.5 * ((epoch / num_epochs) ** 2))


# ---------------------------------------------------------------------------------------------------- 1. shape matrix
#   id         bs   btu  B    K   epoch batch (queue_ptr, queue_ptr1) banks   seed
SHAPES = {
    "k9_b103":  (128, 128, 103, 9, 1, 10, (512, 768), "random", 2101),
    "k16_b224": (128, 128, 224, 16, 2, 3, (256, 1024), "random", 2102),     # BASELINE configs[4]'s spectrum
    "k32_b224": (128, 128, 224, 32, 1, 40, (1024, 256), "random", 2103),
    "uneq":     (64, 192, 103, 9, 3, 7, (384, 128), "random", 2104),        # bs != btu, two M tiles
    "tiny":     (5, 7, 7, 2, 0, 2, (0, 0), "zero", 2105),                   # a run's cold start: smoothing off, zero banks
    "q1000":    (100, 100, 103, 9, 1, 3, (768, 24), "signed", 2106),        # 1000-row banks: partial last bank tile
}


@pytest.mark.parametrize("case", list(SHAPES))
def test_one_step_shapes_w11(dev, golden_dir, case):
    bs, btu, B, K, epoch, batch_index, ptrs, banks, seed = SHAPES[case]
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    g = torch.Generator().manual_seed(seed)
    inp = make_inputs(ti, bs, btu, B, K, g)
    sd, sd1 = init_nets(B, K, seed)
    sa = O.StepArgs(num_epochs=20, labeled_batch_size=bs)
    ost = O.make_state(sd, sd1, K, sa)
    if banks == "zero":
        queues = [torch.zeros_like(t) for t in (ost.queue_feats, ost.queue_probs) * 2]
    else:
        queues = random_banks(5 * bs * 2, K, g, signed=banks == "signed")
    set_banks(ost, queues, ptrs)
    sa.thr = thr_for(oracle_step(copy.deepcopy(ost), inp, epoch, batch_index, sa), epoch, sa.num_epochs)
    ost_before = copy.deepcopy(ost)
    r = oracle_step(ost, inp, epoch, batch_index, sa)
    m = torch.cat([r["mask"], r["masks"]])
    assert 0.0 < float(m.mean()) < 1.0                          # the soft-CE term is exercised
    fs = make_fused(dev, sd, sd1, B, K, queues, ptrs, sa, bs=bs, btu=btu)
    assert fs.cur == (bs, btu) and fs.queue == 5 * bs * 2
    w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
    patches, spectra = (t.to(dev) for t in assembled(inp, sa.noise))
    hist = fs.step(inp["Y_l"].to(dev), epoch, batch_index, patches=patches, spectra=spectra, drop_masks=inp["masks"].to(dev))
    assert fs.prm.smooth == int(banks != "zero")
    r = on_fused_masks(r, ost_before, inp, epoch, batch_index, sa, fs, bs + btu)
    compare_with_oracle(fs, hist, r, ost, w_before, patches, bs + btu)


# ---------------------------------------------------------------------------------------------------- 2. floor pooling
def test_floor_pool_backward(dev, golden_dir):
    """The pool backward with floor semantics, on the kernel's own saved tensors: torch autograd through F.avg_pool2d
    (which floors 11 -> 5 and 5 -> 2) of conv2 on p1 and of conv1 on a0, both with the saved ReLU masks imposed, gives
    the conv weight / bias gradients, and dL/da0 -- at the dropped row / column too, where only the neighbours' taps
    contribute; dz1 is exactly 0 on the dropped row / column."""
    B, K, bs = 103, 9, 64
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    g = torch.Generator().manual_seed(2201)
    inp = make_inputs(ti, bs, bs, B, K, g)
    sd, sd1 = init_nets(B, K, 2201)
    sa = O.StepArgs(num_epochs=20, labeled_batch_size=bs)
    sa.thr = 0.2
    fs = make_fused(dev, sd, sd1, B, K, random_banks(5 * bs * 2, K, g), (0, 256), sa, bs=bs, btu=bs)
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


# --------------------------------------------------------------------------------------------- 3. cube mode, Philox
def test_cube_mode_philox_and_graph_w11(dev, golden_dir):
    """Inputs gathered from the PCA cube in the first kernel (11x11 odd-mode windows), noise and dropout from the device
    Philox stream: the gather is exact, the draws have the right moments, reproduce for the same (seed, step) and differ
    between nets and steps; a CUDA-graph replay computes the same step as the eager launch sequence."""
    from cmlpl_b200.fused_step import FusedMutualStep
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

    def run(noise, graph, steps=1, seed=1088):
        for n, s in zip(nets, sd0):
            n.load_state_dict(s)
        fs = FusedMutualStep(nets[0], nets[1], noise=noise, seed=seed, use_graph=graph, thr=0.5)
        out, pix_d = [], pix.to(dev)
        for it in range(steps):
            fs.step(labels, 1, it, cube=cube, pix=pix_d, spectra=spectra)
            lay = fs.workspace_layout()
            out.append(dict(x16=planes_to_nchw(fs.work[lay["x16"]:], ns, W * W, W).clone(), logits=fs.logits.clone(),
                            hist=fs.hist.clone(),
                            dmask=fs.work[lay["dmask"]:lay["dmask"] + ns * CAT * 4].view(torch.float32).clone(),
                            y=fs.work[lay["ynoisy"]:lay["ynoisy"] + ns * 103 * 4].view(torch.float32).view(ns, 103).clone(),
                            w=[p.detach().clone() for p in fs.params[0]]))
        return out, fs

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


# -------------------------------------------------------------------------------------------- 4. consecutive steps
def test_consecutive_steps_graph_replay_w11(dev, golden_dir):
    """Eight 128 + 128 w = 11 steps of one FusedMutualStep captured once as a CUDA graph and replayed on new inputs,
    re-anchored on the oracle before every step: bank smoothing switches on at batch 4, the bank pointer wraps at 1280,
    and Adam at steps 2..8 is checked exactly against float64."""
    B, K, bs = 103, 9, 128
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    sd, sd1 = init_nets(B, K, 42)
    sa = O.StepArgs(num_epochs=20, queue_batch=3)
    zero = [torch.zeros(1280, 1024), torch.zeros(1280, K)] * 2
    fs = make_fused(dev, sd, sd1, B, K, zero, (0, 0), sa, use_graph=True)
    patches = torch.zeros(2, 2 * bs, 60, W, W, device=dev)
    spectra = torch.zeros(2, 2 * bs, B, device=dev)
    masks = torch.zeros(2, 2 * bs, CAT, device=dev)
    labels = torch.zeros(bs, dtype=torch.int64, device=dev)
    g = torch.Generator().manual_seed(4243)
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
        compare_with_oracle(fs, hist, r, ost, w_before, patches, 2 * bs, adam=it == 0)
        worst = check_adam_exact(fs, before, it + 1)
        seen.append((ptrs, (fs.queue_ptr, fs.queue_ptr1), float(r["mask"].mean()), worst))
        print("step %d: pointers %s -> %s, mask fraction %.2f, Adam max rel error %.1e" % (it + 1, *seen[-1]))
        assert 0.05 <= seen[-1][2] <= 0.95
    assert [s[0][0] for s in seen] == [0, 256, 512, 768, 1024, 0, 256, 512]


# ------------------------------------------------------------------------------------------------- 5. the CLI
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


# ------------------------------------------------------------------------------------------------- 6. loud failures
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
