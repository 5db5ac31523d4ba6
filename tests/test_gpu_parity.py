"""GPU parity suite (-m gpu): every CUDA entry point, called through the C ABI, against the CPU
oracle on the same seeded inputs and against the golden vectors the unmodified reference produced.
Bars: bit-exact for gathers / labels-given-logits / counts; |d| <= 1e-5*max|ref| for the fp32
training blocks; |d| <= 1e-3*max|ref| for the fp16-operand (TF32-precision) scene path."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O
from oracle import golden
from scene_harness import rel

pytestmark = pytest.mark.gpu


def g(golden_dir, name):
    return golden.load(os.path.join(golden_dir, name))


# ------------------------------------------------------------------ a1-a3 patch gather (bit-exact)
def test_patch_gather_golden(dev, golden_dir):
    from cmlpl_b200.tools import hyper_tools as H
    z = g(golden_dir, "patches.npz")
    X = z["X"]
    for w in (4, 6, 10):
        assert np.array_equal(H.ExtractPatches(X, w), z[f"even_w{w}"])
    for w in (3, 5, 11):
        assert np.array_equal(H.ExtractPatches_for_base(X, w), z[f"odd_w{w}"])
    for hw in (1, 3, 5):
        assert np.array_equal(H.MirrowCut(X, hw), z[f"mirror_hw{hw}"])
    with pytest.raises(ValueError):
        H.ExtractPatches(X, 5)
    with pytest.raises(ValueError):
        H.ExtractPatches_for_base(X, 4)


@pytest.mark.parametrize("shape,w,odd", [((31, 29, 60), 20, False), ((23, 40, 60), 11, True), ((12, 15, 7), 6, False),
                                         ((10, 10, 60), 20, False)])
def test_patch_gather_random_idx_and_bands(dev, shape, w, odd):
    from cmlpl_b200 import ops
    rng = np.random.default_rng(3)
    X = rng.standard_normal(shape).astype(np.float32)
    R, C, _ = shape
    idx = rng.integers(0, R * C, size=97)
    Xd = torch.from_numpy(X).to(dev)
    got = ops.patch_gather(Xd, w, idx=torch.from_numpy(idx).to(dev), odd_mode=odd)
    assert np.array_equal(got.cpu().numpy(), O.extract_patches_at(X, w, idx, odd))
    # empty request
    assert ops.patch_gather(Xd, w, idx=torch.zeros(0, dtype=torch.int64, device=dev), odd_mode=odd).shape[0] == 0
    # row bands with halo-only slabs reproduce the full gather bit for bit
    full = O.extract_patches_at(X, w, np.arange(R * C), odd)
    for world in (2, 3):
        parts = []
        for rank in range(world):
            r0, r1, s0, s1 = O.band_rows(R, world, rank, w, odd)
            if r1 <= r0:
                continue
            slab = torch.from_numpy(np.ascontiguousarray(X[s0:s1])).to(dev)
            parts.append(ops.patch_gather(slab, w, first=r0 * C, n=(r1 - r0) * C, odd_mode=odd, scene_rows=R,
                                          slab_row0=s0).cpu().numpy())
        assert np.array_equal(np.concatenate(parts), full)


@pytest.mark.parametrize("w", [2, 6, 10, 14, 18, 4, 8, 20])
@pytest.mark.parametrize("feat", [60, 4])
def test_patch_gather_vectorised_path_every_w(dev, w, feat):
    """feat % 4 == 0 takes patch_gather_reg_kernel; w = 2 (mod 4) makes the group count odd (ADVICE r1: the last
    half-filled pair used to be skipped, leaving torch.empty garbage).  Also with fused noise."""
    from cmlpl_b200 import ops
    rng = np.random.default_rng(100 + w)
    X = rng.standard_normal((21, 19, feat)).astype(np.float32)
    idx = rng.integers(0, 21 * 19, size=33)
    Xd = torch.from_numpy(X).to(dev)
    idx_d = torch.from_numpy(idx).to(dev)
    # poison the caching allocator's free blocks so an unwritten element cannot pass by luck
    poison = torch.full((33 * feat * w * w,), float("nan"), device=dev)
    del poison
    got = ops.patch_gather(Xd, w, idx=idx_d)
    ref = O.extract_patches_at(X, w, idx, False)
    assert np.array_equal(got.cpu().numpy(), ref)
    noise = torch.randn(33, feat, w, w)
    poison = torch.full((33 * feat * w * w,), float("nan"), device=dev)
    del poison
    got = ops.patch_gather(Xd, w, idx=idx_d, noise=noise.to(dev), noise_scale=0.5)
    assert torch.equal(got.cpu(), torch.from_numpy(ref) + noise * 0.5)


def test_patch_gather_fused_noise_is_bit_exact(dev):
    from cmlpl_b200 import ops
    rng = np.random.default_rng(4)
    X = rng.standard_normal((25, 22, 60)).astype(np.float32)
    idx = rng.integers(0, 25 * 22, size=16)
    noise = torch.randn(16, 60, 20, 20)
    got = ops.patch_gather(torch.from_numpy(X).to(dev), 20, idx=torch.from_numpy(idx).to(dev), noise=noise.to(dev),
                           noise_scale=0.5)
    ref = torch.from_numpy(O.extract_patches_at(X, 20, idx)) + noise * 0.5        # train.py:157
    assert torch.equal(got.cpu(), ref)


def test_patch_gather_rejects_bad_arguments(dev):
    from cmlpl_b200 import _lib, ops
    X = torch.zeros(8, 8, 4, device=dev)
    with pytest.raises(_lib.CmlplError):
        ops.patch_gather(X, 5, odd_mode=False)
    with pytest.raises(_lib.CmlplError):
        ops.patch_gather(X, 20)                       # window larger than the scene
    with pytest.raises(_lib.CmlplError):
        ops.patch_gather(X.cpu(), 4)


# ------------------------------------------------------------------ fp32 blocks vs torch fp32 (1e-5)
def test_fp32_blocks(dev):
    from cmlpl_b200 import ops
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(5, 64, 10, 10, generator=gen)
    w3 = torch.randn(64, 64, 3, 3, generator=gen) * 0.05
    b3 = torch.randn(64, generator=gen)
    x60 = torch.randn(5, 60, 10, 10, generator=gen)
    w1 = torch.randn(64, 60, 1, 1, generator=gen) * 0.1
    d = lambda t: t.to(dev).contiguous()
    assert rel(ops.conv2d(d(x60), d(w1), d(b3)).cpu(), F.conv2d(x60, w1, b3)) < 1e-5
    ref = F.relu(F.conv2d(x, w3, b3, padding=1) + x)
    assert rel(ops.conv2d(d(x), d(w3), d(b3), res=d(x), relu=True).cpu(), ref) < 1e-5
    # gradients against autograd
    xr = x.clone().requires_grad_(True); wr = w3.clone().requires_grad_(True); br = b3.clone().requires_grad_(True)
    y = F.conv2d(xr, wr, br, padding=1)
    dy = torch.randn(y.shape, generator=gen)
    y.backward(dy)
    assert rel(ops.conv2d_dgrad(d(dy), d(w3)).cpu(), xr.grad) < 1e-5
    dw, db = ops.conv2d_wgrad(d(x), d(dy), 3)
    assert rel(dw.cpu(), wr.grad) < 2e-5 and rel(db.cpu(), br.grad) < 2e-5
    x6 = x60.clone().requires_grad_(True); w1r = w1.clone().requires_grad_(True)
    y1 = F.conv2d(x6, w1r)
    dy1 = torch.randn(y1.shape, generator=gen)
    y1.backward(dy1)
    dw1, _ = ops.conv2d_wgrad(d(x60), d(dy1), 1)
    assert rel(dw1.cpu(), w1r.grad) < 2e-5
    # pooling
    assert rel(ops.avgpool2(d(x)).cpu(), F.avg_pool2d(x, 2, 2)) < 1e-6
    xp = x.clone().requires_grad_(True)
    F.avg_pool2d(xp, 2, 2).backward(dy[:, :, :5, :5])
    assert rel(ops.avgpool2_bwd(d(dy[:, :, :5, :5]), 10, 10).cpu(), xp.grad) < 1e-6
    # linear pieces
    A = torch.randn(37, 103, generator=gen); W = torch.randn(1024, 103, generator=gen) * 0.1; b = torch.randn(1024, generator=gen)
    assert rel(ops.sgemm(d(A), d(W), transB=True, bias=d(b), act=1).cpu(), F.relu(F.linear(A, W, b))) < 1e-5
    G = torch.randn(37, 1024, generator=gen)
    assert rel(ops.sgemm(d(G), d(A), transA=True).cpu(), G.t() @ A) < 1e-5
    assert rel(ops.sgemm(d(G), d(W)).cpu(), G @ W) < 1e-5
    assert rel(ops.colsum(d(G)).cpu(), G.sum(0)) < 1e-5
    assert torch.equal(ops.relu_bwd(d(A), d(A * 2)).cpu(), torch.where(A > 0, A * 2, torch.zeros_like(A)))
    # l2norm forward/backward (models.py:87-90)
    h = torch.rand(9, 1024, generator=gen).requires_grad_(True)
    yn = O.normalize(h)
    dyn = torch.randn(9, 1024, generator=gen)
    yn.backward(dyn)
    y_d, n_d = ops.l2norm(d(h.detach()))
    assert rel(y_d.cpu(), yn.detach()) < 1e-6
    assert rel(ops.l2norm_bwd(y_d, n_d, d(dyn)).cpu(), h.grad) < 1e-5


# ------------------------------------------------------------------ a5/a6 BaseNet2 vs the reference's own outputs
def test_basenet2_module_matches_reference_golden(dev, golden_dir):
    from cmlpl_b200.tools.models import BaseNet2
    z = g(golden_dir, "basenet2.npz")
    torch.manual_seed(1088)
    BaseNet2(num_features=103, dropout=0, num_classes=9)          # golden script creates this one first
    torch.manual_seed(1088)
    net = BaseNet2(num_features=32, dropout=0, num_classes=16)
    for k in O.LIVE_KEYS:                                           # same seed -> same init as the reference
        assert np.array_equal(net.state_dict()[k].numpy(), z[f"sd.{k}"]), k
    net = net.to(dev).train()
    x, y = torch.from_numpy(z["x"]).to(dev), torch.from_numpy(z["y"]).to(dev)
    lo, fe = net(x, y)
    assert rel(lo.detach().cpu(), z["logits"]) < 1e-5
    assert rel(fe.detach().cpu(), z["feat"]) < 1e-5
    loss = F.cross_entropy(lo, (torch.arange(6) % 16).to(dev)) + fe.pow(3).sum() * 0.1
    loss.backward()
    assert abs(float(loss) - float(z["loss"])) < 1e-5
    for k, p in net.named_parameters():
        if k in O.LIVE_KEYS:
            assert rel(p.grad.cpu(), z[f"grad.{k}"]) < 1e-4, k
        else:
            assert p.grad is None                                   # feat_ss* are dead (models.py:122-126)


def test_basenet2_dropout_mask_injection(dev):
    from cmlpl_b200.tools.models import BaseNet2
    torch.manual_seed(3)
    net = BaseNet2(num_features=40, dropout=0.8, num_classes=9).to(dev).train()
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    x = torch.randn(4, 60, 20, 20); y = torch.randn(4, 40)
    mask = F.dropout(torch.ones(4, 2624), 0.8, True)
    lo, _ = net(x.to(dev), y.to(dev), dropout_mask=mask.to(dev))
    ref, _ = O.basenet2_forward(sd, x, y, mask)
    assert rel(lo.detach().cpu(), ref) < 1e-5
    lo2, _ = net(x.to(dev), y.to(dev))                              # own Philox mask: just has to run and differ
    assert lo2.shape == lo.shape


# ------------------------------------------------------------------ a13 scene inference
def _scene(dev, sd, cube, spectra, K, **kw):
    from cmlpl_b200 import ops
    sdd = {k: v.to(dev) for k, v in sd.items()}
    packed = ops.pack_basenet2(sdd, spectra.shape[1], K, 20)
    return ops.scene_infer(torch.from_numpy(cube).to(dev), torch.from_numpy(spectra).to(dev), packed, K, 20, **kw)


def test_scene_inference_trained_net_vs_reference_golden(dev, golden_dir):
    """Label map and logits of the net trained by the reference's own train.main."""
    z = g(golden_dir, "train_infer.npz")
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd.")}
    labels, logits = _scene(dev, sd, z["cube_pca"], z["spectra"], 9, want_logits=True)
    agree = np.mean(labels.cpu().numpy() == z["predict_label"])
    assert agree >= 0.999, agree
    assert rel(logits.cpu(), z["logits_trained"]) < 1e-3              # rtol 1e-3 of max|logit| (fp16 operands)


def test_scene_inference_random_init_vs_oracle(dev):
    rng = np.random.default_rng(11)
    R, C, B, K = 44, 52, 144, 15
    cube = rng.standard_normal((R, C, 60)).astype(np.float32)
    spectra = rng.standard_normal((R * C, B)).astype(np.float32)
    torch.manual_seed(7)
    sd = O.basenet2_init(B, K)
    labels, logits = _scene(dev, sd, cube, spectra, K, want_logits=True)
    lab_ref, log_ref = O.test_whole(sd, cube, spectra, 20, return_logits=True)
    assert rel(logits.cpu(), log_ref) < 1e-3
    lab = labels.cpu().numpy()
    # argmax is exact given the logits (first index on ties, hyper_tools.py:426)
    assert np.array_equal(lab, logits.cpu().numpy().argmax(1))
    # random-init logits are nearly tied: wherever the labels differ the reference's own margin is tiny
    diff = lab != lab_ref
    srt = np.sort(log_ref, 1)
    assert np.all((srt[diff, -1] - srt[diff, -2]) <= 2e-3 * np.abs(log_ref).max())
    assert np.mean(~diff) >= 0.99


@pytest.mark.parametrize("world", [2, 3, 5])
def test_scene_inference_bands_are_bit_identical(dev, world):
    from cmlpl_b200 import ops
    rng = np.random.default_rng(12)
    R, C, B, K = 37, 33, 103, 9
    cube = rng.standard_normal((R, C, 60)).astype(np.float32)
    spectra = rng.standard_normal((R * C, B)).astype(np.float32)
    torch.manual_seed(8)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}
    packed = ops.pack_basenet2(sd, B, K, 20)
    full_l, full_z = ops.scene_infer(torch.from_numpy(cube).to(dev), torch.from_numpy(spectra).to(dev), packed, K, 20,
                                     want_logits=True)
    got_l, got_z = [], []
    for rank in range(world):
        r0, r1, s0, s1 = O.band_rows(R, world, rank, 20)
        slab = torch.from_numpy(np.ascontiguousarray(cube[s0:s1])).to(dev)
        sp = torch.from_numpy(spectra[r0 * C:r1 * C]).to(dev)
        l, zz = ops.scene_infer(slab, sp, packed, K, 20, band_row0=r0, band_rows=r1 - r0, scene_rows=R, slab_row0=s0,
                                want_logits=True)
        got_l.append(l); got_z.append(zz)
    assert torch.equal(torch.cat(got_l), full_l)
    assert torch.equal(torch.cat(got_z), full_z)


def test_scene_inference_rejects_unsupported(dev):
    from cmlpl_b200 import _lib, ops
    sd = {k: v.to(dev) for k, v in O.basenet2_init(16, 4).items()}
    packed = ops.pack_basenet2(sd, 16, 4, 20)
    cube = torch.zeros(30, 30, 60, device=dev); sp = torch.zeros(900, 16, device=dev)
    with pytest.raises(_lib.CmlplError):
        ops.scene_infer(cube, sp, packed, 4, 16)                      # w != 20
    with pytest.raises(_lib.CmlplError):
        ops.scene_infer(cube[:, :, :30].contiguous(), sp, packed, 4, 20)
    with pytest.raises(_lib.CmlplError):
        ops.scene_infer(cube, sp[:100].contiguous(), packed, 4, 20)


# ------------------------------------------------------------------ a14 metrics (bit-exact)
def test_confusion_and_calaccuracy_golden(dev, golden_dir):
    from cmlpl_b200.tools import hyper_tools as H
    z = g(golden_dir, "metrics_losses.npz")
    assert np.array_equal(H.confusion_matrix(z["pred"], z["label"], 9), z["cm"])
    OA, kappa, pa = H.CalAccuracy(z["pred"], z["label"])
    assert OA == z["OA"] and kappa == z["kappa"] and np.array_equal(pa, z["pa"])
    # predictions above max(label) (model has more classes than the test split)
    pred = z["pred"].copy(); pred[::50] = 12
    o = O.cal_accuracy(pred, z["label"]); m = H.CalAccuracy(pred, z["label"])
    assert o[0] == m[0] and o[1] == m[1] and np.array_equal(o[2], m[2])
    big = np.random.default_rng(1).integers(0, 16, size=3_000_000)
    bigp = np.random.default_rng(2).integers(0, 16, size=3_000_000)
    assert np.array_equal(H.confusion_matrix(bigp, big, 16), O.confusion_matrix(bigp, big, 16))


def test_test_whole_generic_loader(dev, golden_dir):
    """test_whole with an arbitrary (XP, X) loader goes batch by batch through model(XP, X)."""
    from cmlpl_b200.tools import hyper_tools as H
    from cmlpl_b200.tools.models import BaseNet2
    z = g(golden_dir, "train_infer.npz")
    net = BaseNet2(num_features=103, dropout=0.8, num_classes=9)
    net.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd.")}, strict=False)
    net = net.to(dev)
    idx = np.arange(300, 700)
    XP = torch.from_numpy(O.extract_patches_at(z["cube_pca"], 20, idx))
    X = torch.from_numpy(z["spectra"][idx])
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(XP, X), batch_size=128)
    out = H.test_whole(net, loader)
    assert out.dtype == np.int64 and np.array_equal(out, z["predict_label"][idx].astype(np.int64))


def test_streamed_scene_equals_plain(dev):
    """Host-buffer entry point (band-wise H2D overlapped with compute) returns the same labels."""
    from cmlpl_b200 import ops
    from cmlpl_b200.tools.hyper_tools import StreamedScene
    rng = np.random.default_rng(13)
    R, C, B, K = 53, 41, 103, 9
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).pin_memory()
    spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).pin_memory()
    torch.manual_seed(9)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}
    packed = ops.pack_basenet2(sd, B, K, 20)
    ref = ops.scene_infer(cube.to(dev), spectra.to(dev), packed, K, 20)
    for nsplit in (1, 3, 4):
        st = StreamedScene(R, C, B, K, 20, nsplit=nsplit)
        for _ in range(2):                                    # second call reuses the buffers
            got = st(packed, cube, spectra)
            torch.cuda.synchronize()
            assert torch.equal(got, ref.cpu())
    # a band of a larger scene (multi-GPU shape): rows 20..40 with its halo slab
    st = StreamedScene(R, C, B, K, 20, nsplit=2, row0=20, rows=20)
    got = st(packed, cube[st.s0:st.s1].contiguous().pin_memory(), spectra[20 * C:40 * C].contiguous().pin_memory())
    torch.cuda.synchronize()
    assert torch.equal(got, ref.cpu()[20 * C:40 * C])


def test_device_preprocessing_matches_reference_numpy(dev):
    """fit (float64 moments on device + host SVD) and apply reproduce PCANorm + featureNormalize
    (tools/hyper_tools.py:8-32,289-292; oracle.preprocess is pinned bit-equal to the reference files)."""
    from cmlpl_b200 import preprocess, synth
    cube_u16, _ = synth.synth_scene(64, 50, 103, 9, seed=5)
    X = cube_u16.reshape(-1, 103)
    ref_cube, ref_spec = O.preprocess(cube_u16, 60)
    raw = torch.from_numpy(X.copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    assert np.abs(pp.mu - X.mean(0)).max() < 1e-9 and np.abs(pp.sigma - X.astype(np.float64).std(0)).max() < 1e-9
    cube, spec = preprocess.apply(raw, pp)
    assert rel(spec.cpu(), ref_spec) < 1e-6
    got = cube.cpu().numpy().reshape(64, 50, 60)
    # the host SVD of (almost) the same matrix gives every component the reference's sign: a net trained on the
    # reference's preprocessing reads the device's unchanged
    sgn = np.sign((got * ref_cube).sum((0, 1)))
    assert np.all(sgn > 0)
    assert rel(got, ref_cube) < 2e-5
    # float32 raw input path
    cube_f, _ = preprocess.apply(raw.float(), pp, want_spectra=False)
    assert rel(cube_f.cpu(), cube.cpu()) < 1e-6


def test_streamed_raw_scene_equals_preprocessed_path(dev):
    from cmlpl_b200 import ops, preprocess, synth
    from cmlpl_b200.tools.hyper_tools import StreamedRawScene
    R, C, B, K = 47, 39, 103, 9
    cube_u16, _ = synth.synth_scene(R, C, B, K, seed=6)
    raw_host = torch.from_numpy(cube_u16.reshape(-1, B).copy()).pin_memory()
    pp = preprocess.fit(raw_host.to(dev), 60)
    cube, spec = preprocess.apply(raw_host.to(dev), pp)
    torch.manual_seed(10)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}
    packed = ops.pack_basenet2(sd, B, K, 20)
    ref = ops.scene_infer(cube.view(R, C, 60), spec, packed, K, 20)
    for nsplit in (1, 3):
        st = StreamedRawScene(pp, R, C, B, K, 20, nsplit=nsplit)
        got = st(packed, raw_host)
        torch.cuda.synchronize()
        assert torch.equal(got, ref.cpu())
    # folded entry point (preprocessing inside conv0 / the fp16 conversion): same labels as its own one-shot call,
    # band splits bit-identical
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    ref_f = ops.scene_infer_raw(raw_host.to(dev), folded, packed, K, C, 20)
    assert (ref_f == ref).float().mean() >= 0.99
    for nsplit in (1, 3):
        st = StreamedRawScene(pp, R, C, B, K, 20, nsplit=nsplit)
        for _ in range(3):                                    # alternating buffer sets
            got = st(packed, raw_host, folded=folded)
            torch.cuda.synchronize()
            assert torch.equal(got, ref_f.cpu())


@pytest.mark.parametrize("B,K,dtype", [(103, 9, "u16"), (200, 16, "f32")])
def test_scene_infer_raw_folded_matches_oracle(dev, B, K, dtype):
    """cmlpl_scene_infer_raw (PCA + z-scores folded into conv0 and into the spectral fp16 conversion) against the
    oracle's float64 preprocessing (hyper_tools.py:285-292) + test_whole on the same raw scene."""
    from cmlpl_b200 import ops, preprocess, synth
    R, C = 41, 37
    cube_u16, _ = synth.synth_scene(R, C, B, K, seed=7)
    ref_cube, ref_spec = O.preprocess(cube_u16, 60)
    raw = torch.from_numpy(cube_u16.reshape(-1, B).copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    cube, _ = preprocess.apply(raw, pp, want_spectra=False)
    # singular vectors are defined up to sign: adopt the oracle's signs before folding
    sgn = np.sign((cube.cpu().numpy().reshape(R, C, 60) * ref_cube).sum((0, 1)))
    pp.U = pp.U * sgn[None, :]
    pp._dev = None
    torch.manual_seed(21)
    sd = O.basenet2_init(B, K)
    sdd = {k: v.to(dev) for k, v in sd.items()}
    packed = ops.pack_basenet2(sdd, B, K, 20)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    raw_in = raw if dtype == "u16" else raw.float()
    labels, logits = ops.scene_infer_raw(raw_in, folded, packed, K, C, 20, want_logits=True)
    lab_ref, log_ref = O.test_whole(sd, ref_cube.astype(np.float32), ref_spec.astype(np.float32), 20, return_logits=True)
    assert rel(logits.cpu(), log_ref) < 1e-3
    lab = labels.cpu().numpy()
    assert np.array_equal(lab, logits.cpu().numpy().argmax(1))
    diff = lab != lab_ref
    srt = np.sort(log_ref, 1)
    assert np.all((srt[diff, -1] - srt[diff, -2]) <= 2e-3 * np.abs(log_ref).max())
    # a band with its halo slab gives the same bits as the full call
    r0, r1, s0, s1 = O.band_rows(R, 3, 1, 20)
    l2, z2 = ops.scene_infer_raw(raw_in[s0 * C:s1 * C].contiguous(), folded, packed, K, C, 20, band_row0=r0,
                                 band_rows=r1 - r0, scene_rows=R, slab_row0=s0, want_logits=True)
    assert torch.equal(l2, labels[r0 * C:r1 * C]) and torch.equal(z2, logits[r0 * C:r1 * C])
