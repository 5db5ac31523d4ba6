"""Scene inference at 17-32 classes (-m gpu): the dense path (conv1 / conv2 once per scene position, pool2_cls and the
fused spectral kernel at a class width of 32, the sum head) on both entry points, against the CPU oracle, against the
per-pixel kernels of path mode 0, in row bands, stage by stage, and on a net trained with the fused step.

Bars as everywhere on the scene path: logits within 1e-3 * max|ref|, labels = argmax of the returned logits, and a
label that differs from the reference only where the reference's top-2 margin is below 2e-3 * max|ref|."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O

pytestmark = pytest.mark.gpu


def rel(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def near_ties_only(lab, lab_ref, log_ref, bar=2e-3):
    """every label that differs from the reference sits on a reference top-2 margin below the bar"""
    lab, lab_ref, log_ref = np.asarray(lab), np.asarray(lab_ref), np.asarray(log_ref, dtype=np.float64)
    diff = lab != lab_ref
    srt = np.sort(log_ref, 1)
    return bool(np.all((srt[diff, -1] - srt[diff, -2]) <= bar * np.abs(log_ref).max()))


class path_mode:
    """cmlpl_set_scene_path_mode for a block (the mode is per host thread; 1 is the default)"""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        from cmlpl_b200 import _lib
        _lib.call("cmlpl_set_scene_path_mode", self.mode)

    def __exit__(self, *exc):
        from cmlpl_b200 import _lib
        _lib.call("cmlpl_set_scene_path_mode", 1)


def _dense_flag(R, C, B, K, w):
    from cmlpl_b200 import _lib
    off = (ctypes.c_size_t * 12)()
    _lib.call("cmlpl_scene_workspace_layout", R, C, B, K, w, off)
    return int(off[11])


def _net(B, K, w, seed, dev):
    """random-init BaseNet2 (w = 11: the 1280-input classifier of the odd-window variant) and its cpu state dict"""
    from cmlpl_b200.tools.models import BaseNet2
    torch.manual_seed(seed)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    return net, {k: v.detach().cpu() for k, v in net.state_dict().items()}


@pytest.mark.parametrize("w,B,K", [(20, 48, 20), (20, 103, 17), (20, 144, 24), (20, 224, 32), (11, 103, 20), (11, 224, 32)])
def test_dense_path_matches_oracle(dev, w, B, K):
    from cmlpl_b200 import ops
    R, C = 23, 29
    assert _dense_flag(R, C, B, K, w) == 1
    rng = np.random.default_rng(B * 100 + K)
    cube = rng.standard_normal((R, C, 60)).astype(np.float32)
    spectra = rng.standard_normal((R * C, B)).astype(np.float32)
    net, sd = _net(B, K, w, B + K, dev)
    lab_ref, log_ref = O.test_whole(sd, cube, spectra, w, odd_mode=(w == 11), return_logits=True)
    labels, logits = ops.scene_infer(torch.from_numpy(cube).to(dev), torch.from_numpy(spectra).to(dev),
                                     net.packed_weights(w), K, w, want_logits=True)
    lab, lg = labels.cpu().numpy(), logits.cpu().numpy()
    assert rel(lg, log_ref) < 1e-3
    assert np.array_equal(lab, lg.argmax(1))
    assert near_ties_only(lab, lab_ref, log_ref)


@pytest.mark.parametrize("K", [20, 32])
def test_cube_path_dense_matches_mode0(dev, K):
    """mode 0 keeps the independent implementation at 17-32 classes: per-pixel patch CNN + CUDA-core heads"""
    from cmlpl_b200 import ops
    R, C, B, w = 45, 61, 103, 20
    gen = torch.Generator(device=dev); gen.manual_seed(K)
    cube = torch.randn((R, C, 60), device=dev, generator=gen)
    spectra = torch.randn((R * C, B), device=dev, generator=gen)
    net, _ = _net(B, K, w, K, dev)
    packed = net.packed_weights(w)
    lab1, log1 = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    with path_mode(0):
        assert _dense_flag(R, C, B, K, w) == 0
        lab0, log0 = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    l1, l0 = log1.cpu().numpy(), log0.cpu().numpy()
    assert rel(l1, l0) < 1e-3
    assert np.array_equal(lab1.cpu().numpy(), l1.argmax(1))
    assert near_ties_only(lab1.cpu().numpy(), lab0.cpu().numpy(), l0)


def _raw_scene(dev, R, C, B, K, seed):
    """synthetic raw scene, its float64 oracle preprocessing, and the device preprocessing with the oracle's PCA signs"""
    from cmlpl_b200 import preprocess, synth
    cube_u16, _ = synth.synth_scene(R, C, B, K, seed=seed)
    ref_cube, ref_spec = O.preprocess(cube_u16, 60)
    raw = torch.from_numpy(cube_u16.reshape(-1, B).copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    cube, _ = preprocess.apply(raw, pp, want_spectra=False)
    sgn = np.sign((cube.cpu().numpy().reshape(R, C, 60) * ref_cube).sum((0, 1)))   # singular vectors: up to sign
    pp.U = pp.U * sgn[None, :]
    pp._dev = None
    return cube_u16, raw, pp, ref_cube.astype(np.float32), ref_spec.astype(np.float32)


@pytest.mark.parametrize("K,dtype", [(20, "u16"), (32, "f32")])
def test_raw_path_dense_and_mode0_match_oracle(dev, K, dtype):
    from cmlpl_b200 import ops
    R, C, B, w = 41, 37, 103, 20
    _, raw, pp, ref_cube, ref_spec = _raw_scene(dev, R, C, B, K, seed=K)
    net, sd = _net(B, K, w, 30 + K, dev)
    packed = net.packed_weights(w)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    raw_in = raw if dtype == "u16" else raw.float()
    lab_ref, log_ref = O.test_whole(sd, ref_cube, ref_spec, w, return_logits=True)
    lab1, log1 = ops.scene_infer_raw(raw_in, folded, packed, K, C, w, want_logits=True)
    with path_mode(0):
        lab0, log0 = ops.scene_infer_raw(raw_in, folded, packed, K, C, w, want_logits=True)
    for lab, lg in ((lab1, log1), (lab0, log0)):
        lab, lg = lab.cpu().numpy(), lg.cpu().numpy()
        assert rel(lg, log_ref) < 1e-3
        assert np.array_equal(lab, lg.argmax(1))
        assert near_ties_only(lab, lab_ref, log_ref)
    assert rel(log1.cpu().numpy(), log0.cpu().numpy()) < 1e-3
    assert near_ties_only(lab1.cpu().numpy(), lab0.cpu().numpy(), log0.cpu().numpy())


def test_row_bands_are_bit_identical_at_32_classes(dev):
    """cube path and raw path: row bands with their halo slabs, single rows included, give the one-call result bit for bit"""
    from cmlpl_b200 import ops
    R, C, B, K, w = 26, 33, 103, 32, 20
    gen = torch.Generator(device=dev); gen.manual_seed(5)
    cube = torch.randn((R, C, 60), device=dev, generator=gen)
    spectra = torch.randn((R * C, B), device=dev, generator=gen)
    net, sd = _net(B, K, w, 5, dev)
    packed = net.packed_weights(w)
    lab, lg = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    bands = [(0, 1), (1, 7), (7, 8), (8, 20), (20, 25), (25, 26)]
    parts = [ops.scene_infer(cube, spectra[a * C:b * C].contiguous(), packed, K, w, band_row0=a, band_rows=b - a, want_logits=True)
             for a, b in bands]
    assert torch.equal(torch.cat([p[0] for p in parts]), lab) and torch.equal(torch.cat([p[1] for p in parts]), lg)
    _, raw, pp, _, _ = _raw_scene(dev, R, C, B, K, seed=6)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    lab_r, lg_r = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True)
    parts = []
    for a, b in bands:
        s0, s1 = max(0, a - 10), min(R, b + 9)
        parts.append(ops.scene_infer_raw(raw[s0 * C:s1 * C].contiguous(), folded, packed, K, C, w, band_row0=a, band_rows=b - a,
                                         scene_rows=R, slab_row0=s0, want_logits=True))
    assert torch.equal(torch.cat([p[0] for p in parts]), lab_r) and torch.equal(torch.cat([p[1] for p in parts]), lg_r)


@pytest.mark.parametrize("K", [24, 32])
def test_pool2_cls_row_maps_match_torch(dev, K):
    """pool2_cls_kernel<32> on the kernel's own half-pooled conv2 maps yq: M[I][y', x'] = sum_J L[I][J][y', x' + 2J]
    with the remaining 2x2 pool of the middle classes, against torch in fp32 on the same fp16 inputs and weights."""
    from cmlpl_b200 import _lib
    R, C, B, w = 37, 45, 103, 20
    rng = np.random.default_rng(K)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    net, _ = _net(B, K, w, K, dev)
    packed = net.packed_weights(w)
    st = torch.cuda.current_stream().cuda_stream
    PR, PC, PR2, PC2 = R + w - 1, C + w - 1, (R + w) // 2, (C + w) // 2
    f0 = torch.empty(8 * PR * PC * 8, dtype=torch.float16, device=dev)
    pmq = torch.full((9, 4, 8, PR2, PC2, 8), float("nan"), dtype=torch.float16, device=dev)
    yq = torch.full((9, 4, 8, PR2, PC2, 8), float("nan"), dtype=torch.float16, device=dev)
    lmap = torch.full((4, 5, 8, PR2, PC2, 4), float("nan"), dtype=torch.float32, device=dev)   # [4][5][NC/4 quads][PR2][PC2][4]
    _lib.call("cmlpl_conv0_map_f16", cube.data_ptr(), R, C, 0, R, w, 0, R, packed.data_ptr(), f0.data_ptr(), st)
    _lib.call("cmlpl_conv1_pool_planes_f16", f0.data_ptr(), C, w, R, packed.data_ptr(), pmq.data_ptr(), st)
    _lib.call("cmlpl_conv2_scene_f16", pmq.data_ptr(), C, w, R, packed.data_ptr(), yq.data_ptr(), st)
    _lib.call("cmlpl_pool2_cls_f16", yq.data_ptr(), C, w, R, B, K, packed.data_ptr(), lmap.data_ptr(), st)
    torch.cuda.synchronize()
    yz = torch.nan_to_num(yq.permute(0, 1, 2, 5, 3, 4).reshape(9, 4, 64, PR2, PC2).float())
    Wc = net.classifier.weight.detach()[:, :1600].reshape(K, 64, 5, 5).half().float()
    for I in range(5):
        Al = 0 if I == 0 else (2 if I == 4 else 1)
        ref = torch.zeros(4, K, PR2, PC2, device=dev)
        for J in range(5):
            Be = 0 if J == 0 else (2 if J == 4 else 1)
            us = [0, 1] if Al == 1 else [0]
            vs = [0, 1] if Be == 1 else [0]
            for u in us:
                for v in vs:
                    sh = F.pad(yz[Al * 3 + Be], (0, 2 * J + 1, 0, 1))[:, :, u:u + PR2, 2 * J + v:2 * J + v + PC2]
                    ref += torch.einsum("kc,pcyx->pkyx", Wc[:, :, I, J], sh) / (len(us) * len(vs))
        got = lmap[:, I].permute(0, 1, 4, 2, 3).reshape(4, 32, PR2, PC2)[:, :K]
        # map I is read at y' = r' + 2I >= 2I, x' = c' <= PC2 - 11 only: compare where every input exists
        g, r = got[:, :, 2 * I:PR2 - 1, :PC2 - 10], ref[:, :, 2 * I:PR2 - 1, :PC2 - 10]
        assert not torch.isnan(g).any(), I
        assert rel(g.cpu(), r.cpu()) < 1e-4, I


def test_trained_20_class_net(dev):
    """Two 20-class peers trained with the fused step on a synthetic 20-class scene: dense labels vs the oracle's
    test_whole, and StreamedRawScene on the raw cube (pinned host rows, two buffer sets) gives the same labels."""
    from cmlpl_b200 import ops, preprocess, synth
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.tools.hyper_tools import StreamedRawScene
    from cmlpl_b200.tools.models import BaseNet2
    R, C, B, K, w = 64, 72, 64, 20, 20                     # the 60 PCA components need >= 60 bands
    cube_u16, gt = synth.synth_scene(R, C, B, K, seed=20)
    raw_host = torch.from_numpy(cube_u16.reshape(-1, B).copy()).pin_memory()
    pp = preprocess.fit(raw_host.to(dev), 60)
    cube, spec = preprocess.apply(raw_host.to(dev), pp)
    cube = cube.view(R, C, 60).contiguous()
    torch.manual_seed(20)
    nets = [BaseNet2(B, 0, K).to(dev) for _ in range(2)]
    fs = FusedMutualStep(nets[0], nets[1], bs=128, btu=128, lr=1e-3)
    flat = gt.reshape(-1)
    lab_pix = np.nonzero(flat > 0)[0]
    g = np.random.default_rng(20)
    for it in range(300):
        pl = g.choice(lab_pix, 128, replace=False)
        pu = g.choice(R * C, 128, replace=False)
        fs.step(torch.from_numpy(flat[pl].astype(np.int64) - 1).to(dev), it // 30, it % 30, cube=cube,
                pix=torch.from_numpy(np.concatenate([pl, pu]).astype(np.int64)).to(dev), spectra=spec)
    torch.cuda.synchronize()
    net = nets[0].eval()
    packed = net.packed_weights(w)
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    assert _dense_flag(R, C, B, K, w) == 1
    labels = ops.scene_infer(cube, spec, packed, K, w)
    lab_ref = O.test_whole(sd, cube.cpu().numpy(), spec.cpu().numpy(), w)
    lab = labels.cpu().numpy()
    assert float(np.mean(lab == lab_ref)) >= 0.999
    # the net has learnt the scene (not a degenerate constant map)
    assert float(np.mean(lab[flat > 0] == flat[flat > 0] - 1)) > 0.25
    for nsplit in (1, 3):
        st = StreamedRawScene(pp, R, C, B, K, w, nsplit=nsplit)
        for _ in range(2):
            got = st(packed, raw_host)
            torch.cuda.synchronize()
            assert torch.equal(got, labels.cpu())


def test_more_than_32_classes_is_an_error(dev):
    from cmlpl_b200 import _lib, ops, preprocess
    R, C, B, K, w = 12, 14, 103, 33, 20
    cube = torch.randn((R, C, 60), device=dev)
    spectra = torch.randn((R * C, B), device=dev)
    torch.manual_seed(33)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}
    packed = ops.pack_basenet2(sd, B, K, w)
    assert _dense_flag(R, C, B, K, w) == 0
    with pytest.raises(_lib.CmlplError):
        ops.scene_infer(cube, spectra, packed, K, w)
    raw = torch.from_numpy(np.random.default_rng(33).integers(0, 4000, (R * C, B)).astype(np.uint16)).to(dev)
    pp = preprocess.fit(raw, 60)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    with pytest.raises(_lib.CmlplError):
        ops.scene_infer_raw(raw, folded, packed, K, C, w)
    st = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros(1 << 20, dtype=torch.float32, device=dev)
    lab = torch.zeros(R * C, dtype=torch.uint8, device=dev)
    with pytest.raises(_lib.CmlplError):
        _lib.call("cmlpl_pool2_cls_f16", buf.data_ptr(), C, w, R, B, K, packed.data_ptr(), buf.data_ptr(), st)
    with pytest.raises(_lib.CmlplError):
        _lib.call("cmlpl_head_sum_lmap", buf.data_ptr(), buf.data_ptr(), C, R, B, K, w, packed.data_ptr(), lab.data_ptr(), None, st)
