"""BASELINE configs[4] as written: 11x11 patches.  The reference's BaseNet2 is hard-wired to w = 20
(tools/models.py:127), so the odd-window variant is a documented extension: windows follow
ExtractPatches_for_base (hyper_tools.py:300-317: 5 / 5 halo), pooling keeps torch's floor semantics (11 -> 5 -> 2)
and the classifier takes 64*2*2 + 1024 = 1280 inputs.  The CPU oracle restates exactly that (its forward is
size-agnostic); the scene path runs patch_cnn_kernel<11> per pixel.  Bars as for w = 20: logits 1e-3 * max|ref|,
labels 99 % on a random-init net (near-tied logits; every disagreement must sit inside the logit error)."""
import numpy as np
import pytest
import torch

from oracle import cmlpl_oracle as O
from scene_harness import rel

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape,B,K", [((23, 31), 224, 16), ((12, 40), 103, 9)])
def test_scene_inference_w11_matches_oracle(dev, shape, B, K):
    from cmlpl_b200 import ops
    from cmlpl_b200.tools.models import BaseNet2
    R, C = shape
    rng = np.random.default_rng(11)
    cube = rng.standard_normal((R, C, 60)).astype(np.float32)
    spectra = rng.standard_normal((R * C, B)).astype(np.float32)
    torch.manual_seed(1088)
    net = BaseNet2(B, 0, K, w=11).to(dev).eval()
    assert net.classifier.in_features == 1280
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    lab_ref, log_ref = O.test_whole(sd, cube, spectra, 11, odd_mode=True, return_logits=True)
    packed = net.packed_weights(11)
    cube_d, spec_d = torch.from_numpy(cube).to(dev), torch.from_numpy(spectra).to(dev)
    labels, logits = ops.scene_infer(cube_d, spec_d, packed, K, 11, want_logits=True)
    assert rel(logits.cpu().numpy(), log_ref) < 1e-3
    got = labels.cpu().numpy()
    agree = float(np.mean(got == lab_ref))
    assert agree >= 0.99, agree
    bad = np.nonzero(got != lab_ref)[0]
    tol = 2e-3 * np.abs(log_ref).max()
    for i in bad:                                   # only near-ties may flip
        assert log_ref[i].max() - log_ref[i, got[i]] < tol
    # row bands with 5/5 halo slabs reproduce the one-band result bit for bit
    for world in (2, 3):
        parts = []
        for rank in range(world):
            r0, r1, s0, s1 = O.band_rows(R, world, rank, 11, True)
            if r1 <= r0:
                continue
            parts.append(ops.scene_infer(cube_d[s0:s1].contiguous(), spec_d[r0 * C:r1 * C].contiguous(), packed, K, 11,
                                         band_row0=r0, band_rows=r1 - r0, scene_rows=R, slab_row0=s0))
        assert torch.equal(torch.cat(parts), labels)


def test_batch_forward_backward_w11(dev):
    """The fp32 batch-mode path (training blocks) with the 1280-input classifier, against torch."""
    from cmlpl_b200.tools.models import BaseNet2
    torch.manual_seed(3)
    net = BaseNet2(50, 0, 7, w=11).to(dev).train()
    x = torch.randn(6, 60, 11, 11, device=dev); y = torch.randn(6, 50, device=dev)
    lo, fe = net(x, y)
    (lo.square().sum() + fe.sum()).backward()
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in net.state_dict().items()}
    lo_r, fe_r = O.basenet2_forward(sd, x.cpu(), y.cpu())
    (lo_r.square().sum() + fe_r.sum()).backward()
    assert rel(lo.detach().cpu(), lo_r.detach()) < 1e-5
    for k in O.LIVE_KEYS:
        assert rel(dict(net.named_parameters())[k].grad.cpu(), sd[k].grad) < 1e-4, k


@pytest.mark.parametrize("w,shape,B,K", [(11, (29, 37), 224, 16), (11, (18, 52), 103, 9), (20, (33, 41), 144, 15),
                                         (20, (37, 45), 103, 9), (20, (37, 45), 200, 16)])
def test_compute_sharing_path_matches_per_pixel_path(dev, w, shape, B, K):
    """cmlpl_scene_infer's default kernels (conv1 / conv2 evaluated once per scene position in border classes, pooled
    cells as class-partial maps) against the per-pixel kernels (cmlpl_set_scene_path_mode(0): patch_cnn_kernel<w> on every
    pixel's own window) on the same conv0 map -- two independent evaluations of tools/models.py:133-150.  For w = 11 the
    shared kernels run with the 2x2 pooled cells of the 1280-input classifier.  Logits within 5e-4 * max, labels the
    argmax of the logits, labels equal wherever the per-pixel logits are not tied to within that and on > 99.5 % of
    the pixels."""
    from cmlpl_b200 import _lib, ops
    from cmlpl_b200.tools.models import BaseNet2
    R, C = shape
    rng = np.random.default_rng(w + B)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
    torch.manual_seed(w + B)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    packed = net.packed_weights(w)
    lab_d, log_d = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    _lib.call("cmlpl_set_scene_path_mode", 0)
    try:
        lab_p, log_p = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    finally:
        _lib.call("cmlpl_set_scene_path_mode", 1)
    log_d, log_p, lab_d, lab_p = log_d.cpu().numpy(), log_p.cpu().numpy(), lab_d.cpu().numpy(), lab_p.cpu().numpy()
    assert rel(log_d, log_p) < 5e-4
    assert np.array_equal(lab_d, log_d.argmax(1))
    tol = 1e-3 * np.abs(log_p).max()
    top2 = np.sort(log_p, axis=1)[:, -2:]
    clear = (top2[:, 1] - top2[:, 0]) > tol
    assert np.array_equal(lab_d[clear], lab_p[clear])
    assert clear.mean() > 0.9
    assert np.mean(lab_d == lab_p) > 0.995
