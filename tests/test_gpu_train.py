"""GPU parity of the training path (-m gpu): loss kernels, fused Adam and one full mutual-learning
step against the CPU oracle (whose ref_step was pinned bit-exactly against the reference's
train.main) and against the committed step fixture.  fp32 bars: |d| <= 1e-5*max|ref| forward,
1e-4*max|ref| for gradients (different summation order / fp32 atomics in split-K wgrad)."""
import argparse
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O
from oracle import golden
from test_oracle_cpu import replay_step

pytestmark = pytest.mark.gpu


def rel(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def relu_flips(sd, x, y, dev):
    """Number of ReLU inputs whose sign differs between the CUDA fp32 forward and torch CPU fp32.
    Summation order moves activations by ~2e-6; an activation that is zero to within that flips its
    ReLU mask, and ONE flip moves a conv weight gradient (a sum of ~1e5 signed terms) by ~1e-3 of its
    max.  Gradient bars are therefore 1e-4 when no mask differs and 5e-3 otherwise."""
    from cmlpl_b200 import ops
    d = lambda t: t.detach().to(dev).contiguous()
    a0 = F.conv2d(x, sd["conv0.weight"], sd["conv0.bias"])
    a1 = F.relu(F.conv2d(a0, sd["conv1.weight"], sd["conv1.bias"], padding=1) + a0)
    p1 = F.avg_pool2d(a1, 2, 2)
    a2 = F.relu(F.conv2d(p1, sd["conv2.weight"], sd["conv2.bias"], padding=1) + p1)
    h = F.relu(F.linear(y, sd["feat_spe.weight"], sd["feat_spe.bias"]))
    m0 = ops.conv2d(d(x), d(sd["conv0.weight"]), d(sd["conv0.bias"]))
    m1 = ops.conv2d(m0, d(sd["conv1.weight"]), d(sd["conv1.bias"]), res=m0, relu=True)
    mp1 = ops.avgpool2(m1)
    m2 = ops.conv2d(mp1, d(sd["conv2.weight"]), d(sd["conv2.bias"]), res=mp1, relu=True)
    mh = ops.sgemm(d(y), d(sd["feat_spe.weight"]), transB=True, bias=d(sd["feat_spe.bias"]), act=1)
    assert rel(m1.cpu(), a1) < 1e-5 and rel(m2.cpu(), a2) < 1e-5 and rel(mh.cpu(), h) < 1e-5
    return sum(int(((m.cpu() > 0) != (a > 0)).sum()) for m, a in ((m1, a1), (m2, a2), (mh, h)))


def test_cross_entropy_hard_and_soft(dev):
    from cmlpl_b200 import losses
    g = torch.Generator().manual_seed(1)
    z = torch.randn(128, 9, generator=g)
    y = torch.randint(0, 9, (128,), generator=g)
    zr = z.clone().requires_grad_(True)
    F.cross_entropy(zr, y).backward()
    zd = z.to(dev).requires_grad_(True)
    l = losses.cross_entropy(zd, y.to(dev))
    l.backward()
    assert abs(float(l) - float(F.cross_entropy(z, y))) < 1e-6
    assert rel(zd.grad.cpu(), zr.grad) < 1e-5
    p = torch.softmax(torch.randn(128, 9, generator=g) * 2, 1) * 0.9        # rows need not sum to 1
    m = (torch.rand(128, generator=g) > 0.4).float()
    zr = z.clone().requires_grad_(True)
    (O.soft_ce(zr, p, m) * 4).backward()
    zd = z.to(dev).requires_grad_(True)
    l = losses.soft_cross_entropy(zd, p.to(dev), m.to(dev)) * 4
    l.backward()
    assert abs(float(l) - 4 * float(O.soft_ce(z, p, m))) < 1e-5
    assert rel(zd.grad.cpu(), zr.grad) < 1e-5


@pytest.mark.parametrize("smooth", [False, True])
def test_bank_smooth(dev, smooth):
    from cmlpl_b200 import ops
    g = torch.Generator().manual_seed(2)
    z = torch.randn(128, 16, generator=g)
    f = O.normalize(torch.rand(128, 1024, generator=g))
    qf = O.normalize(torch.rand(1280, 1024, generator=g)); qf[900:] = 0          # zero rows still count (exp(0)=1)
    qp = torch.softmax(torch.randn(1280, 16, generator=g), 1); qp[900:] = 0
    po, p, m = ops.bank_smooth(z.to(dev), f.to(dev), qf.to(dev), qp.to(dev), 0.95, 0.3, smooth, 0.2)
    ref_o = torch.softmax(z, 1)
    ref = O.bank_smooth(ref_o, f, qf, qp, 0.95, 0.3) if smooth else ref_o
    assert rel(po.cpu(), ref_o) < 1e-5 and rel(p.cpu(), ref) < 1e-5
    refm = ref.max(1)[0].ge(0.2).float()
    border = (ref.max(1)[0] - 0.2).abs() < 1e-6
    assert torch.equal(m.cpu()[~border], refm[~border])


@pytest.mark.parametrize("n", [128, 1024])        # 1024 = the config-3 InfoNCE stress shape
def test_graph_contrast(dev, n):
    from cmlpl_b200 import losses
    g = torch.Generator().manual_seed(3)
    fs = O.normalize(torch.rand(n, 1024, generator=g)); fw = O.normalize(torch.rand(n, 1024, generator=g))
    p1 = torch.softmax(torch.randn(n, 16, generator=g) * 3, 1); p = torch.softmax(torch.randn(n, 16, generator=g) * 3, 1)
    Q, Qn = O.graph_targets(p1, p)
    for side in (0, 1):
        a = fs.clone().requires_grad_(True); b = fw.clone().requires_grad_(True)
        ref = O.graph_contrast(a, b.detach(), Q, Qn, 0.3) if side == 0 else O.graph_contrast(a.detach(), b, Q, Qn, 0.3)
        ref.backward()
        ad = fs.to(dev).requires_grad_(True); bd = fw.to(dev).requires_grad_(True)
        l = losses.graph_contrast(ad, bd, p1.to(dev), p.to(dev), 0.3, side)
        l.backward()
        assert abs(float(l) - float(ref)) < 1e-5 * max(1.0, abs(float(ref)))
        got, want = (ad.grad, a.grad) if side == 0 else (bd.grad, b.grad)
        assert rel(got.cpu(), want) < 1e-4
        assert (bd.grad if side == 0 else ad.grad) is None


def test_ntxent_golden(dev, golden_dir):
    from cmlpl_b200.tools.models import ContrastiveLoss
    z = np.load(os.path.join(golden_dir, "metrics_losses.npz"))
    ei, ej = torch.from_numpy(z["ntx_i"]), torch.from_numpy(z["ntx_j"])
    a = ei.clone().requires_grad_(True); b = ej.clone().requires_grad_(True)
    O.nt_xent(a, b, 0.5).backward()
    ad = ei.to(dev).requires_grad_(True); bd = ej.to(dev).requires_grad_(True)
    l = ContrastiveLoss(24, device=dev, temperature=0.5)(ad, bd)
    l.backward()
    assert abs(float(l) - float(z["ntx_loss"])) < 1e-5          # the reference module's own output
    assert rel(ad.grad.cpu(), a.grad) < 1e-4 and rel(bd.grad.cpu(), b.grad) < 1e-4


def test_fused_adam_matches_torch(dev):
    from cmlpl_b200.losses import FusedAdam
    g = torch.Generator().manual_seed(4)
    ws = [torch.randn(s, generator=g) for s in ((64, 60, 1, 1), (1024, 103), (9,), (300,))]
    ref = [w.clone().requires_grad_(True) for w in ws]
    mine = [w.clone().to(dev).requires_grad_(True) for w in ws]
    o_ref = torch.optim.Adam(ref, lr=5e-4); o_mine = FusedAdam(mine, lr=5e-4)
    for it in range(4):
        for r, m in zip(ref[:3], mine[:3]):                       # the 4th tensor never gets a grad (skipped)
            gr = torch.randn(r.shape, generator=g) * 10 ** (-it)
            r.grad = gr.clone(); m.grad = gr.to(dev)
        o_ref.step(); o_mine.step()
    for r, m in zip(ref, mine):
        assert rel(m.detach().cpu(), r.detach()) < 1e-6
    assert torch.equal(mine[3].detach().cpu(), ws[3])


def test_mutual_step_matches_oracle_and_fixture(dev, golden_dir):
    """One full 128+128 step: forward, losses, both backward passes, both Adam updates, bank writes."""
    from cmlpl_b200 import train as T
    z = golden.load(os.path.join(golden_dir, "step.npz"))
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    r, ost = replay_step(z, ti)
    inp = ost.extras["inputs"]
    nz, a = inp["noise"], inp["args"]
    args = argparse.Namespace(temperature=a.temperature, thr=a.thr, num_epochs=a.num_epochs, queue_batch=a.queue_batch,
                              alpha=a.alpha, lr=a.lr, labeled_batch_size=128, dropout=0, noise=a.noise)
    st = T.make_state(103, 9, args, dev)
    st.Base.load_state_dict(inp["sd"]); st.Base1.load_state_dict(inp["sd1"])
    for dst, src in zip((st.queue_feats, st.queue_probs, st.queue_feats1, st.queue_probs1), inp["queues"]):
        dst.copy_(src)
    st.extras["keep_grads"] = True
    d = lambda t: t.to(dev)
    XP_b = torch.cat([inp["XP_l"] + nz["xp_l1"] * a.noise, inp["XP_u"] + nz["xp_u1"] * a.noise], 0)
    X_b = torch.cat([inp["X_l"] + nz["x_l1"] * a.noise, inp["X_u"] + nz["x_u1"] * a.noise], 0)
    XP_e = torch.cat([inp["XP_l"] + nz["xp_l2"] * a.noise, inp["XP_u"] + nz["xp_u2"] * a.noise], 0)
    X_e = torch.cat([inp["X_l"] + nz["x_l2"] * a.noise, inp["X_u"] + nz["x_u2"] * a.noise], 0)
    hist, aux = T.mutual_step(st, d(XP_b), d(X_b), d(XP_e), d(X_e), d(inp["Y_l"]), 1, 0, args)
    hist = hist.cpu().numpy()
    # vs the fixture (frozen oracle output) and vs the oracle replayed now
    for want in (z["hist"], r["hist"]):
        assert np.abs(hist - want).max() <= 1e-4 * np.abs(want).max(), (hist, want)
    assert rel(aux["logits"].cpu(), z["logits"]) < 1e-5 and rel(aux["logits1"].cpu(), z["logits1"]) < 1e-5
    assert rel(aux["probs"].cpu(), z["probs"]) < 1e-5 and rel(aux["probs1"].cpu(), z["probs1"]) < 1e-5
    assert np.array_equal(aux["mask"].cpu().numpy(), z["mask"]) and np.array_equal(aux["masks"].cpu().numpy(), z["masks"])
    for name, want in (("total1", z["total1"]), ("lc1", z["lc1"]), ("con1", z["con1"]), ("cls1", z["cls1"])):
        assert abs(float(aux[name]) - float(want)) <= 1e-4 * max(1.0, abs(float(want))), name
    with torch.no_grad():
        flips = relu_flips(inp["sd"], XP_b, X_b, dev), relu_flips(inp["sd1"], XP_e, X_e, dev)
    bars = [1e-4 if f == 0 else 5e-3 for f in flips]
    print("ReLU mask disagreements (net0, net1):", flips)
    for k in O.LIVE_KEYS:
        assert rel(aux["grads"][k].cpu(), z[f"grad.{k}"]) < bars[0], (k, flips)
        assert rel(aux["grads1"][k].cpu(), z[f"grad1.{k}"]) < bars[1], (k, flips)
        new = dict(st.Base.named_parameters())[k].detach().cpu().numpy()
        # Adam's first step moves every weight by ~lr*sign(g): compare where the gradient is not ~0
        gz = np.abs(z[f"grad.{k}"]) > 1e-3 * np.abs(z[f"grad.{k}"]).max()
        assert np.abs(new - z[f"new.{k}"])[gz].max() < (1e-6 if flips[0] == 0 else 5e-5), k
    # memory banks after the step (incl. the queue_ptr1 quirk, train.py:237)
    assert (st.queue_ptr, st.queue_ptr1) == (ost.queue_ptr, ost.queue_ptr1)
    assert rel(st.queue_feats.cpu(), ost.queue_feats) < 1e-5 and rel(st.queue_probs1.cpu(), ost.queue_probs1) < 1e-5


def test_train_cli_end_to_end_synthetic(dev, tmp_path):
    """sample_generation + train + test_whole + CalAccuracy through the CLIs on a tiny synthetic scene."""
    from cmlpl_b200 import sample_generation as SG, synth, train as T
    synth.SHAPES["paviau"] = (48, 44, 103, 9)
    try:
        root = str(tmp_path) + "/"
        SG.main(SG.build_parser().parse_args(["--dataID", "1", "--root", root, "--synthetic"]))
        T.seed_torch()
        out = T.main(T.build_parser().parse_args(["--dataID", "1", "--root", root, "--num_epochs", "2", "--num_unlabel",
                                                  "512", "--print_per_batches", "2"]))
    finally:
        synth.SHAPES["paviau"] = (610, 340, 103, 9)
    h = out["loss_hist"]
    assert h.shape == (8, 5) and np.isfinite(h).all()
    assert h[-1, 2] < h[0, 2]                                   # supervised CE goes down
    assert np.all(h[:4, 3] == 0)                                # thr=1 masks everything in epoch 0 (train.py:148,221)
    assert out["predict_label"].shape == (48 * 44,) and out["predict_label"].dtype == np.int64
    OA, kappa, pa = out["results"][0]
    assert 0.5 < OA <= 1.0 and pa.shape == (9,)
