"""Edge cases of the scene path on GPU (-m gpu): tiny / ragged scenes, odd pixel counts, single-row
bands, class/band counts that take the CUDA-core head, a Houston-shaped scene checked on sampled rows."""
import numpy as np
import pytest
import torch

from oracle import cmlpl_oracle as O

pytestmark = pytest.mark.gpu


def rel(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _run(dev, R, C, B, K, seed, **kw):
    from cmlpl_b200 import ops
    rng = np.random.default_rng(seed)
    cube = rng.standard_normal((R, C, 60)).astype(np.float32)
    spectra = rng.standard_normal((R * C, B)).astype(np.float32)
    torch.manual_seed(seed)
    sd = O.basenet2_init(B, K)
    packed = ops.pack_basenet2({k: v.to(dev) for k, v in sd.items()}, B, K, 20)
    labels, logits = ops.scene_infer(torch.from_numpy(cube).to(dev), torch.from_numpy(spectra).to(dev), packed, K, 20,
                                     want_logits=True, **kw)
    return sd, cube, spectra, labels.cpu().numpy(), logits.cpu().numpy()


@pytest.mark.parametrize("R,C", [(10, 10), (11, 13), (10, 31), (33, 10)])
def test_tiny_and_odd_scenes(dev, R, C):
    """Smallest scenes the mirror padding allows (w/2 <= min dim), odd pixel counts (pair tail)."""
    sd, cube, spectra, lab, logits = _run(dev, R, C, 103, 9, seed=R * 100 + C)
    lab_ref, log_ref = O.test_whole(sd, cube, spectra, 20, return_logits=True)
    assert rel(logits, log_ref) < 1e-3
    assert np.array_equal(lab, logits.argmax(1))
    assert np.mean(lab == lab_ref) >= 0.97


def test_single_row_bands_are_bit_identical(dev):
    from cmlpl_b200 import ops
    R, C, B, K = 14, 21, 103, 9
    rng = np.random.default_rng(2)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
    torch.manual_seed(2)
    packed = ops.pack_basenet2({k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}, B, K, 20)
    full = ops.scene_infer(cube, spectra, packed, K, 20)
    rows = [ops.scene_infer(cube, spectra[r * C:(r + 1) * C].contiguous(), packed, K, 20, band_row0=r, band_rows=1)
            for r in range(R)]
    assert torch.equal(torch.cat(rows), full)


@pytest.mark.parametrize("B,K", [(224, 16), (240, 16), (103, 20), (40, 3)])
def test_cuda_core_head_and_unusual_widths(dev, B, K):
    """> 224 bands or > 16 classes take the all-per-pixel kernel + CUDA-core head; 224 bands (AVIRIS-NG, BASELINE.json
    configs[4]) is the widest spectrum of the tensor-core path (spectral_logits_kernel, 28 k-chunks); small B/K too."""
    sd, cube, spectra, lab, logits = _run(dev, 24, 26, B, K, seed=B + K)
    lab_ref, log_ref = O.test_whole(sd, cube, spectra, 20, return_logits=True)
    assert rel(logits, log_ref) < 1e-3
    assert np.array_equal(lab, logits.argmax(1))


def test_houston_shaped_scene_sampled_rows(dev):
    """BASELINE.json configs[3] shape (349 x 1905 x 144, 15 classes): whole scene on GPU, oracle on sampled rows."""
    R, C, B, K = 349, 1905, 144, 15
    sd, cube, spectra, lab, logits = _run(dev, R, C, B, K, seed=4)
    assert lab.shape == (R * C,) and np.array_equal(lab, logits.argmax(1))
    for r in (0, 173, 348):                                  # first, middle, last row (mirror at both edges)
        cols = np.arange(0, C, 37)
        idx = r * C + cols
        XP = O.extract_patches_at(cube, 20, idx)
        with torch.no_grad():
            ref, _ = O.basenet2_forward(sd, torch.from_numpy(XP), torch.from_numpy(spectra[idx]))
        assert rel(logits[idx], ref.numpy()) < 1e-3, r


def test_confusion_and_gather_empty_inputs(dev):
    from cmlpl_b200 import ops
    cm = ops.confusion(torch.zeros(0, dtype=torch.uint8, device=dev), torch.zeros(0, dtype=torch.int64, device=dev), 5)
    assert int(cm.sum()) == 0
    lab = torch.tensor([0, 1, 2, 250], dtype=torch.uint8, device=dev)
    tru = torch.tensor([0, -1, 2, 3], dtype=torch.int64, device=dev)           # -1 (unlabelled) and out-of-range ignored
    cm = ops.confusion(lab, tru, 4).cpu().numpy()
    assert cm.sum() == 2 and cm[0, 0] == 1 and cm[2, 2] == 1


def test_full_size_scene_properties(dev):
    """BASELINE.json's headline shape (610 x 340 x 103, 9 classes) at full size, through size-independent properties:
    labels are the argmax of the returned logits, an uneven 4-band walk with read-only halos reproduces the one-shot
    label map bit for bit, a second run is bit-identical (no race in the persistent kernels), and a stride of sampled
    pixels agrees with the CPU oracle."""
    from cmlpl_b200 import ops
    R, C, B, K, w = 610, 340, 103, 9, 20
    gen = torch.Generator(device=dev); gen.manual_seed(7)
    cube = torch.randn((R, C, 60), device=dev, generator=gen)
    spectra = torch.randn((R * C, B), device=dev, generator=gen)
    torch.manual_seed(7)
    sd = O.basenet2_init(B, K)
    packed = ops.pack_basenet2({k: v.to(dev) for k, v in sd.items()}, B, K, w)
    lab, logits = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    assert torch.equal(lab, logits.argmax(1).to(torch.uint8))
    assert torch.equal(lab, ops.scene_infer(cube, spectra, packed, K, w))
    parts, r0 = [], 0
    for rows in (97, 200, 13, 300):
        parts.append(ops.scene_infer(cube, spectra[r0 * C:(r0 + rows) * C], packed, K, w, band_row0=r0, band_rows=rows,
                                     scene_rows=R))
        r0 += rows
    assert r0 == R and torch.equal(torch.cat(parts), lab)
    idx = np.arange(0, R * C, 6007)
    cube_h = cube.cpu().numpy()
    with torch.no_grad():
        ref, _ = O.basenet2_forward(sd, torch.from_numpy(O.extract_patches_at(cube_h, w, idx)), spectra[torch.from_numpy(idx).to(dev)].cpu())
    assert rel(logits[torch.from_numpy(idx).to(dev)].cpu().numpy(), ref.numpy()) < 1e-3


def test_wide_spectrum_scene_in_row_bands(dev):
    """224 bands / 16 classes (the AVIRIS-NG-scale shape of BASELINE.json configs[4], reduced to 300 x 257 pixels): the
    row-band walk an 8192 x 8192 scene needs gives the one-shot label map bit for bit."""
    from cmlpl_b200 import ops
    R, C, B, K, w = 300, 257, 224, 16, 20
    gen = torch.Generator(device=dev); gen.manual_seed(9)
    cube = torch.randn((R, C, 60), device=dev, generator=gen)
    spectra = torch.randn((R * C, B), device=dev, generator=gen)
    torch.manual_seed(9)
    packed = ops.pack_basenet2({k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}, B, K, w)
    full = ops.scene_infer(cube, spectra, packed, K, w)
    ws = ops.scene_workspace(64, C, B, K, w, dev)
    parts = [ops.scene_infer(cube, spectra[a * C:min(a + 64, R) * C], packed, K, w, band_row0=a, band_rows=min(64, R - a),
                             scene_rows=R, workspace=ws) for a in range(0, R, 64)]
    assert torch.equal(torch.cat(parts), full)


@pytest.mark.parametrize("B,K,dtype", [(103, 9, "u16"), (200, 16, "f32")])
def test_raw_path_mid_size_matches_preprocessed_path(dev, B, K, dtype):
    """cmlpl_scene_infer_raw on a scene large enough that every persistent kernel walks several tiles per CTA
    (220 x 180 pixels): logits within 2e-3 of the path that materialises the PCA cube / z-scored spectra first, the
    same labels wherever the margin allows, band walk bit-identical."""
    from cmlpl_b200 import ops, preprocess, synth
    R, C = 220, 180
    cube_u16, _ = synth.synth_scene(R, C, B, K, seed=12)
    raw = torch.from_numpy(cube_u16.reshape(-1, B).copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    cube, spec = preprocess.apply(raw, pp)
    torch.manual_seed(12)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}
    packed = ops.pack_basenet2(sd, B, K, 20)
    lab_a, log_a = ops.scene_infer(cube.view(R, C, 60), spec, packed, K, 20, want_logits=True)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    raw_in = raw if dtype == "u16" else raw.float()
    lab_b, log_b = ops.scene_infer_raw(raw_in, folded, packed, K, C, 20, want_logits=True)
    assert rel(log_b.cpu().numpy(), log_a.cpu().numpy()) < 2e-3
    assert torch.equal(lab_b, log_b.argmax(1).to(torch.uint8))
    assert float((lab_a == lab_b).float().mean()) > 0.99
    parts = []
    for a in range(0, R, 64):
        b = min(a + 64, R)
        s0, s1 = max(0, a - 10), min(R, b + 9)
        parts.append(ops.scene_infer_raw(raw_in[s0 * C:s1 * C].contiguous(), folded, packed, K, C, 20, band_row0=a,
                                         band_rows=b - a, scene_rows=R, slab_row0=s0))
    assert torch.equal(torch.cat(parts), lab_b)


def test_scene_infer_from_two_streams_interleaved(dev):
    """cmlpl_scene_infer forks its spectral branch onto the library's per-device side stream (api.cu::side_stream).  Two
    caller streams that issue scenes alternately share that side stream and its events; every result must still be
    the one a lone call produces (bit-identical: the kernels are deterministic), and work queued on a caller stream
    after the call must see the labels."""
    from cmlpl_b200 import ops
    K, w = 9, 20
    scenes = []
    for i, (R, C, B) in enumerate([(61, 83, 103), (47, 120, 103)]):
        rng = np.random.default_rng(40 + i)
        cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
        spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
        torch.manual_seed(40 + i)
        packed = ops.pack_basenet2({k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}, B, K, w)
        ref = ops.scene_infer(cube, spectra, packed, K, w).clone()
        scenes.append(dict(cube=cube, spectra=spectra, packed=packed, ref=ref, R=R, C=C, B=B,
                           ws=ops.scene_workspace(R, C, B, K, w, dev), labels=torch.empty(R * C, dtype=torch.uint8, device=dev),
                           copy=torch.empty(R * C, dtype=torch.uint8, device=dev), stream=torch.cuda.Stream(device=dev)))
    torch.cuda.synchronize()
    for it in range(25):
        for s in scenes:
            with torch.cuda.stream(s["stream"]):
                s["labels"].fill_(255)
                ops.scene_infer(s["cube"], s["spectra"], s["packed"], K, w, workspace=s["ws"], labels=s["labels"])
                s["copy"].copy_(s["labels"])                  # queued behind the call on the caller's stream
        if it % 8 == 7:
            torch.cuda.synchronize()
            for s in scenes:
                assert torch.equal(s["copy"], s["ref"]), it
    torch.cuda.synchronize()
    for s in scenes:
        assert torch.equal(s["copy"], s["ref"]) and torch.equal(s["labels"], s["ref"])


@pytest.mark.parametrize("case", ["band_outside_the_scene", "slab_misses_the_halo", "cube_not_16_byte_aligned"])
def test_rejected_scene_call_leaves_workspace_and_labels_untouched(dev, case):
    """A dense-path call that is rejected enqueues nothing, on the caller's stream or on the side stream: after a
    device-wide synchronize (which waits on the side stream too) the workspace still holds its sentinel bytes and the
    labels still read 255."""
    from cmlpl_b200 import _lib, ops
    R, C, B, K, w, rows = 40, 50, 103, 9, 20, 10
    rng = np.random.default_rng(77)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    spectra = torch.from_numpy(rng.standard_normal((rows * C, B)).astype(np.float32)).to(dev)
    torch.manual_seed(77)
    packed = ops.pack_basenet2({k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}, B, K, w)
    ws = ops.scene_workspace(rows, C, B, K, w, dev).fill_(0xA5)
    labels = torch.full((rows * C,), 255, dtype=torch.uint8, device=dev)
    kw = dict(band_rows=rows, scene_rows=R, workspace=ws, labels=labels)
    if case == "band_outside_the_scene":
        kw["band_row0"], match = R - 5, "band outside the scene"
    elif case == "slab_misses_the_halo":
        cube, kw["slab_row0"], match = cube[5:], 5, "do not cover the band's halo"     # rows 0..9 need scene row 0
    else:
        flat = torch.empty(R * C * 60 + 4, device=dev)
        cube = flat[1:1 + R * C * 60].view(R, C, 60).copy_(cube)                       # 4 bytes past a 16-byte boundary
        match = "cube must be 16-byte aligned"
    torch.cuda.synchronize()
    with pytest.raises(_lib.CmlplError, match=match):
        ops.scene_infer(cube, spectra, packed, K, w, **kw)
    torch.cuda.synchronize()
    assert bool((ws == 0xA5).all()) and bool((labels == 255).all())
