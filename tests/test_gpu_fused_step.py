"""GPU parity of the FUSED training step (-m gpu): cmlpl_train_step (tcgen05 convolutions, fp16 operands / fp32
accumulate, 15 launches) against the CPU oracle's ref_step (pinned bit-exactly against the reference's train.main) and
the committed step fixture.

Bars (north_star: 1e-3 for reduced-precision operands, stated as |d| <= bar * max|ref| per tensor):
  * logits / probabilities / losses / head gradients: 1e-3;
  * every convolution-backward kernel against torch fp32 convolutions applied to the kernel's OWN saved tensors
    (ReLU masks, fp16 activations, dL/dcat): 1e-3 ("linearised" check -- this is the kernel-correctness gate);
  * convolution gradients end to end against the fp32 oracle: 3e-2.  An fp16-operand forward flips the ReLU mask of
    the few activations that are zero to within 2^-11 (counted and bounded below: < 1e-4 of all mask bits); one flip
    moves a weight gradient -- a sum of ~1e7 signed terms -- by a full term, so this figure measures the flips, not
    the backward kernels.  (The fp32 path has the same effect at its own precision, see scene_harness.relu_flips.)
"""
import argparse
import functools
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from fused_step_harness import HEAD, compare_with_oracle, cube_mode_steps, make_fused
from oracle import cmlpl_oracle as O
from oracle import golden
from scene_harness import rel
from test_oracle_cpu import replay_step

pytestmark = pytest.mark.gpu

def test_fused_step_matches_oracle_and_fixture(dev, golden_dir):
    """The 128+128 step of tests/golden/step.npz (PaviaU shape, B=103, 9 classes, epoch 1, bank smoothing on)."""
    z = golden.load(os.path.join(golden_dir, "step.npz"))
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    r, ost = replay_step(z, ti)
    inp = ost.extras["inputs"]
    nz, a = inp["noise"], inp["args"]
    XP_b = torch.cat([inp["XP_l"] + nz["xp_l1"] * a.noise, inp["XP_u"] + nz["xp_u1"] * a.noise], 0)
    X_b = torch.cat([inp["X_l"] + nz["x_l1"] * a.noise, inp["X_u"] + nz["x_u1"] * a.noise], 0)
    XP_e = torch.cat([inp["XP_l"] + nz["xp_l2"] * a.noise, inp["XP_u"] + nz["xp_u2"] * a.noise], 0)
    X_e = torch.cat([inp["X_l"] + nz["x_l2"] * a.noise, inp["X_u"] + nz["x_u2"] * a.noise], 0)
    fs = make_fused(dev, inp["sd"], inp["sd1"], 103, 9, inp["queues"], thr=a.thr, num_epochs=a.num_epochs, lr=a.lr,
                    temperature=a.temperature, alpha=a.alpha, queue_batch=a.queue_batch, dropout=0.0)
    w_before = [{k: p.detach().clone() for k, p in n.named_parameters()} for n in fs.nets]
    patches = torch.stack([XP_b, XP_e]).to(dev).contiguous()
    spectra = torch.stack([X_b, X_e]).to(dev).contiguous()
    hist = fs.step(inp["Y_l"].to(dev), 1, 0, patches=patches, spectra=spectra)
    # the frozen fixture and the oracle replayed now agree, so one comparison covers both
    assert np.abs(r["hist"] - z["hist"]).max() < 1e-6
    compare_with_oracle(fs, hist, r, ost, w_before, patches, 256)


def test_both_steps_at_the_indian_pines_shape_with_dropout_masks(dev, golden_dir):
    """BASELINE configs[1] shape (B=200, 16 classes) with INJECTED non-null dropout masks (p = 0.8) through the whole
    step: the fp32 path (1e-5 / 1e-4 bars) and the fused tcgen05 path (bars in the module docstring) against the
    oracle's ref_step on the same inputs."""
    from cmlpl_b200 import train as T
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    Xp = ti["cube_pca"]
    B, K, bs = 200, 16, 128
    g = torch.Generator().manual_seed(123)
    R, C = Xp.shape[:2]
    li = torch.randint(0, R * C, (bs,), generator=g).numpy()
    ui = torch.randint(0, R * C, (bs,), generator=g).numpy()
    XP_l = torch.from_numpy(O.extract_patches_at(Xp, 20, li)); XP_u = torch.from_numpy(O.extract_patches_at(Xp, 20, ui))
    X_l = torch.randn(bs, B, generator=g); X_u = torch.randn(bs, B, generator=g)
    Y_l = torch.randint(0, K, (bs,), generator=g)
    torch.manual_seed(77)
    sd, sd1 = O.basenet2_init(B, K), O.basenet2_init(B, K)
    sa = O.StepArgs(num_epochs=20)
    sa.thr = 0.09
    ost = O.make_state(sd, sd1, K, sa)
    queues = [O.normalize(torch.randn(1280, 1024, generator=g).abs()), torch.softmax(torch.randn(1280, K, generator=g) * 2, 1),
              O.normalize(torch.randn(1280, 1024, generator=g).abs()), torch.softmax(torch.randn(1280, K, generator=g) * 2, 1)]
    for dst, src in zip((ost.queue_feats, ost.queue_probs, ost.queue_feats1, ost.queue_probs1), queues):
        dst.copy_(src)
    ost.queue_ptr, ost.queue_ptr1 = 512, 768
    nz = {k: torch.randn(s, generator=g) for k, s in (
        ("xp_l1", XP_l.shape), ("x_l1", X_l.shape), ("xp_l2", XP_l.shape), ("x_l2", X_l.shape),
        ("xp_u1", XP_u.shape), ("x_u1", X_u.shape), ("xp_u2", XP_u.shape), ("x_u2", X_u.shape))}
    p = 0.8
    masks = [(torch.rand(2 * bs, 2624, generator=g) >= p).float() / (1 - p) for _ in range(2)]
    r = O.ref_step(ost, XP_l, X_l, Y_l, XP_u, X_u, nz, epoch=3, batch_index=5, args=sa, drop_masks=tuple(masks))
    assert 0.05 < float(r["mask"].mean()) < 1.0            # the soft-CE term is exercised
    XP_b = torch.cat([XP_l + nz["xp_l1"] * sa.noise, XP_u + nz["xp_u1"] * sa.noise], 0)
    X_b = torch.cat([X_l + nz["x_l1"] * sa.noise, X_u + nz["x_u1"] * sa.noise], 0)
    XP_e = torch.cat([XP_l + nz["xp_l2"] * sa.noise, XP_u + nz["xp_u2"] * sa.noise], 0)
    X_e = torch.cat([X_l + nz["x_l2"] * sa.noise, X_u + nz["x_u2"] * sa.noise], 0)
    d = lambda t: t.to(dev)
    # ---- fp32 path
    args = argparse.Namespace(temperature=sa.temperature, thr=sa.thr, num_epochs=sa.num_epochs, queue_batch=sa.queue_batch,
                              alpha=sa.alpha, lr=sa.lr, labeled_batch_size=128, dropout=0, noise=sa.noise)
    st = T.make_state(B, K, args, dev)
    st.Base.load_state_dict(sd, strict=False); st.Base1.load_state_dict(sd1, strict=False)
    for dst, src in zip((st.queue_feats, st.queue_probs, st.queue_feats1, st.queue_probs1), queues):
        dst.copy_(src)
    st.queue_ptr, st.queue_ptr1 = 512, 768
    st.extras["keep_grads"] = True
    hist, aux = T.mutual_step(st, d(XP_b), d(X_b), d(XP_e), d(X_e), d(Y_l), 3, 5, args, drop_masks=(d(masks[0]), d(masks[1])))
    assert np.abs(hist.cpu().numpy() - r["hist"]).max() <= 1e-4 * np.abs(r["hist"]).max()
    assert rel(aux["logits"], r["logits"]) < 1e-5 and rel(aux["logits1"], r["logits1"]) < 1e-5
    assert np.array_equal(aux["mask"].cpu().numpy(), r["mask"].numpy())
    for k in O.LIVE_KEYS:
        assert rel(aux["grads"][k], r["grads"][k]) < 5e-3 and rel(aux["grads1"][k], r["grads1"][k]) < 5e-3, k
    assert (st.queue_ptr, st.queue_ptr1) == (ost.queue_ptr, ost.queue_ptr1)
    # ---- fused path
    fs = make_fused(dev, sd, sd1, B, K, queues, thr=sa.thr, num_epochs=sa.num_epochs, lr=sa.lr,
                    temperature=sa.temperature, alpha=sa.alpha, queue_batch=sa.queue_batch, dropout=p)
    fs.queue_ptr, fs.queue_ptr1 = 512, 768
    w_before = [{k: q.detach().clone() for k, q in n.named_parameters()} for n in fs.nets]
    patches = torch.stack([XP_b, XP_e]).to(dev).contiguous()
    spectra = torch.stack([X_b, X_e]).to(dev).contiguous()
    hist = fs.step(d(Y_l), 3, 5, patches=patches, spectra=spectra, drop_masks=torch.stack(masks).to(dev))
    compare_with_oracle(fs, hist, r, ost, w_before, patches, 256)


def test_fused_step_cube_mode_philox_and_graph(dev, golden_dir):
    """Inputs gathered from the PCA cube inside the first kernel, noise and dropout from the device Philox stream:
    the gather is exact, the draws have the right moments, are reproducible per (seed, step) and differ between
    steps; a CUDA-graph replay computes the same step as the eager launch sequence."""
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.tools.models import BaseNet2
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    cube = torch.from_numpy(ti["cube_pca"]).to(dev).contiguous()
    spectra = torch.from_numpy(ti["spectra"]).to(dev).contiguous()
    R, C = cube.shape[:2]
    g = torch.Generator().manual_seed(5)
    pix = torch.randint(0, R * C, (256,), generator=g)
    labels = torch.randint(0, 9, (128,), generator=g).to(dev)
    torch.manual_seed(3)
    nets = [BaseNet2(103, 0.8, 9).to(dev) for _ in range(2)]
    sd0 = [{k: v.detach().clone() for k, v in n.state_dict().items()} for n in nets]
    run = functools.partial(cube_mode_steps, nets, sd0, labels, cube, pix, spectra)
    want = torch.from_numpy(O.extract_patches_at(ti["cube_pca"], 20, pix.numpy()))
    clean, _ = run(0.0, False)
    x = clean[0]["x16"]
    assert torch.equal(x[:256, :60].cpu(), want.half().float()) and torch.equal(x[256:, :60].cpu(), want.half().float())
    assert float(x[:, 60:].abs().max()) == 0.0
    assert torch.equal(clean[0]["y"][:256].cpu(), torch.from_numpy(ti["spectra"][pix.numpy()]))
    noisy, _ = run(0.5, False, steps=2)
    zn = (noisy[0]["x16"][:, :60].cpu() - torch.cat([want, want])) / 0.5
    assert abs(float(zn.mean())) < 2e-3 and abs(float(zn.var()) - 1.0) < 1e-2                 # 12.3 M draws
    assert abs(float((zn ** 4).mean()) - 3.0) < 5e-2                                          # Gaussian kurtosis
    zy = (noisy[0]["y"].cpu() - torch.from_numpy(ti["spectra"][pix.numpy()]).repeat(2, 1)) / 0.5
    assert abs(float(zy.mean())) < 2e-2 and abs(float(zy.var()) - 1.0) < 3e-2
    keep = float((noisy[0]["dmask"] > 0).float().mean())
    assert abs(keep - 0.2) < 2e-3 and float(noisy[0]["dmask"].max()) == pytest.approx(5.0)    # inverted dropout, p = 0.8
    # the two nets and two consecutive steps draw different noise; the same (seed, step) reproduces it
    assert not torch.equal(noisy[0]["x16"][:256], noisy[0]["x16"][256:])
    assert not torch.equal(noisy[0]["x16"], noisy[1]["x16"])
    again, _ = run(0.5, False, steps=2)
    assert torch.equal(again[0]["x16"], noisy[0]["x16"]) and torch.equal(again[1]["dmask"], noisy[1]["dmask"])
    other, _ = run(0.5, False, seed=7)
    assert not torch.equal(other[0]["x16"], noisy[0]["x16"])
    # CUDA graph: same logits bit for bit after step 1, same weights after 3 steps up to the order of the fp32 atomics
    eager, _ = run(0.5, False, steps=3)
    graph, fsg = run(0.5, True, steps=3)
    assert torch.equal(eager[0]["logits"], graph[0]["logits"])
    for a, b in zip(eager[2]["w"], graph[2]["w"]):
        assert rel(a, b) < 1e-4
    assert fsg.launches() == 15 and np.isfinite(graph[2]["hist"].cpu().numpy()).all()
    # the host runs many steps ahead of the device: the per-step scalars (Adam bias corrections, bank pointers, Philox
    # offsets) every step READS must be the ones written for that step (ring of pinned blocks, here only 3 deep)
    from cmlpl_b200.fused_step import TrainParams
    for n, s in zip(nets, sd0):
        n.load_state_dict(s)
    fr = FusedMutualStep(nets[0], nets[1], noise=0.5, use_graph=True, thr=0.5, param_slots=3)
    snaps, pix_d = [], pix.to(dev)
    for it in range(40):
        fr.step(labels, 1, it, cube=cube, pix=pix_d, spectra=spectra)
        snaps.append(fr.prm_dev.clone())                      # stream-ordered: what this step's kernels saw
    torch.cuda.synchronize()
    qp = 0
    for it, sn in enumerate(snaps):
        prm = TrainParams.from_buffer_copy(bytes(sn.cpu().numpy()))
        assert prm.offset == it and abs(prm.bc1 - (1 - 0.9 ** (it + 1))) < 1e-6, it
        assert prm.queue_ptr[0] == qp, (it, prm.queue_ptr[0], qp)
        qp = (qp + 256) % 1280


def test_packed_weights_follow_the_optimizers(dev):
    """ADVICE r1: the scene-inference weight pack is cached on parameter versions, and both optimizers update the
    parameters through raw pointers -- eval -> train -> eval must repack."""
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.losses import FusedAdam
    from cmlpl_b200.tools.models import BaseNet2
    torch.manual_seed(0)
    nets = [BaseNet2(103, 0, 9).to(dev) for _ in range(2)]
    before = nets[0].packed_weights(20).clone()
    assert nets[0].packed_weights(20).data_ptr() == nets[0].packed_weights(20).data_ptr()      # cached while unchanged
    opt = FusedAdam(nets[0].parameters(), lr=1e-2)
    for p in (nets[0].conv1.weight, nets[0].classifier.weight):
        p.grad = torch.ones_like(p)
    opt.step()
    mid = nets[0].packed_weights(20).clone()
    assert not torch.equal(before, mid)
    fs = FusedMutualStep(nets[0], nets[1], lr=1e-2)
    g = torch.Generator().manual_seed(1)
    fs.step(torch.randint(0, 9, (128,), generator=g).to(dev), 0, 0, patches=torch.randn(2, 256, 60, 20, 20, generator=g).to(dev),
            spectra=torch.randn(2, 256, 103, generator=g).to(dev))
    after = nets[0].packed_weights(20)
    assert not torch.equal(mid, after)
    from cmlpl_b200 import ops
    fresh = ops.pack_basenet2(dict(nets[0].state_dict()), 103, 9, 20)
    assert torch.equal(after[:2 * 73728], fresh[:2 * 73728])          # conv1 / conv2 regions (the rest has padding gaps)


@pytest.mark.parametrize("M,N", [(128, 1280), (100, 300), (16, 160)])
def test_tcgen05_similarity_gemm(dev, M, N):
    """cmlpl_sim_nt_tc_f32 (fp16 operands on tcgen05, fp32 accumulate) on unit-norm 1024-d features, tails included,
    and the loss entry points in their tensor-core mode against the fp32 mode."""
    from cmlpl_b200 import _lib, ops
    g = torch.Generator().manual_seed(M + N)
    A = F.normalize(torch.randn(M, 1024, generator=g), dim=1).to(dev)
    B = F.normalize(torch.randn(N, 1024, generator=g), dim=1).to(dev)
    C = torch.full((M, N), float("nan"), device=dev)
    _lib.call("cmlpl_sim_nt_tc_f32", A.data_ptr(), B.data_ptr(), M, N, 1024, C.data_ptr(), torch.cuda.current_stream().cuda_stream)
    ref = A.double() @ B.double().t()
    assert float((C.double() - ref).abs().max()) < 1e-3 * float(ref.abs().max())
    z = torch.randn(M, 9, generator=g).to(dev)
    qp = torch.softmax(torch.randn(N, 9, generator=g), 1).to(dev)
    fp32 = ops.bank_smooth(z, A, B, qp, 0.95, 0.3, True, 0.5)
    _lib.call("cmlpl_set_loss_gemm_mode", 1)
    try:
        tc = ops.bank_smooth(z, A, B, qp, 0.95, 0.3, True, 0.5)
    finally:
        _lib.call("cmlpl_set_loss_gemm_mode", 0)
    assert rel(tc[1], fp32[1]) < 1e-3 and torch.equal(tc[0], fp32[0])


def test_fused_step_partial_batch_and_argument_checks(dev, golden_dir):
    """train.py's DataLoaders keep the last partial batch (10 000 samples / 128 -> a 16-row tail): a FusedMutualStep built
    for 128 + 128 runs a 16 + 16 step on the head of its buffers and matches the oracle; bad arguments fail loudly."""
    from cmlpl_b200 import _lib
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    Xp, Xs = ti["cube_pca"], ti["spectra"]
    B, K, bs = 103, 9, 16
    g = torch.Generator().manual_seed(77)
    R, C = Xp.shape[:2]
    li = torch.randint(0, R * C, (bs,), generator=g).numpy(); ui = torch.randint(0, R * C, (bs,), generator=g).numpy()
    XP_l = torch.from_numpy(O.extract_patches_at(Xp, 20, li)); XP_u = torch.from_numpy(O.extract_patches_at(Xp, 20, ui))
    X_l = torch.from_numpy(Xs[li]); X_u = torch.from_numpy(Xs[ui])
    Y_l = torch.randint(0, K, (bs,), generator=g)
    torch.manual_seed(5)
    sd, sd1 = O.basenet2_init(B, K), O.basenet2_init(B, K)
    sa = O.StepArgs(num_epochs=20)
    sa.thr = 0.12
    ost = O.make_state(sd, sd1, K, sa)                                         # 1280-row banks like train.py:138
    queues = [O.normalize(torch.randn(1280, 1024, generator=g).abs()), torch.softmax(torch.randn(1280, K, generator=g) * 2, 1),
              O.normalize(torch.randn(1280, 1024, generator=g).abs()), torch.softmax(torch.randn(1280, K, generator=g) * 2, 1)]
    for dst, src in zip((ost.queue_feats, ost.queue_probs, ost.queue_feats1, ost.queue_probs1), queues):
        dst.copy_(src)
    ost.queue_ptr, ost.queue_ptr1 = 1024, 0
    zero = {k: torch.zeros(s) for k, s in (("xp_l1", XP_l.shape), ("x_l1", X_l.shape), ("xp_l2", XP_l.shape), ("x_l2", X_l.shape),
                                           ("xp_u1", XP_u.shape), ("x_u1", X_u.shape), ("xp_u2", XP_u.shape), ("x_u2", X_u.shape))}
    r = O.ref_step(ost, XP_l, X_l, Y_l, XP_u, X_u, zero, epoch=2, batch_index=78, args=sa)
    fs = make_fused(dev, sd, sd1, B, K, queues, thr=sa.thr, num_epochs=sa.num_epochs, lr=sa.lr, temperature=sa.temperature,
                    alpha=sa.alpha, queue_batch=sa.queue_batch, dropout=0.0, noise=0.0)          # built for 128 + 128
    fs.queue_ptr, fs.queue_ptr1 = 1024, 0
    cube = torch.from_numpy(Xp).to(dev).contiguous()
    spectra = torch.from_numpy(Xs).to(dev).contiguous()
    pix = torch.from_numpy(np.concatenate([li, ui])).to(dev)
    hist = fs.step(Y_l.to(dev), 2, 78, cube=cube, pix=pix, spectra=spectra)
    h = hist.cpu().numpy()
    assert fs.logits.shape == (2, 32, K) and fs.mask.shape == (2, 16)
    assert np.abs(h[:5] - r["hist"]).max() <= 1e-3 * np.abs(r["hist"]).max(), (h[:5], r["hist"])
    assert rel(fs.logits[0], r["logits"]) < 1e-3 and rel(fs.probs[1], r["probs1"]) < 1e-3
    for i, k in enumerate(HEAD):
        assert rel(fs.grads[0][6 + i], r["grads"][k]) < 1e-3, k
    assert (fs.queue_ptr, fs.queue_ptr1) == (ost.queue_ptr, ost.queue_ptr1) == (0, 256)        # literal 256 stride
    assert rel(fs.queue_feats[0][1024:1056], ost.queue_feats[1024:1056]) < 1e-5
    # ---- loud failures
    with pytest.raises(_lib.CmlplError):
        fs.step(torch.zeros(200, dtype=torch.int64, device=dev), 0, 0, cube=cube, pix=torch.zeros(400, dtype=torch.int64, device=dev),
                spectra=spectra)                                                             # larger than the step was built for
    with pytest.raises(_lib.CmlplError):
        fs.step(Y_l.to(dev), 0, 0, cube=cube.cpu(), pix=pix, spectra=spectra)                  # host tensors: no CPU path
    with pytest.raises(_lib.CmlplError):
        fs.step(Y_l.to(dev), 0, 0, cube=cube, pix=pix, spectra=spectra, patches=torch.zeros(2, 32, 60, 20, 20, device=dev))
    fs.queue_ptr = 1260
    with pytest.raises(RuntimeError):
        fs.step(Y_l.to(dev), 0, 0, cube=cube, pix=pix, spectra=spectra)                        # bank write past the queue
