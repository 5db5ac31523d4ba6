"""Band selection on the GPU.  The oracle of every call with a band list is the same call without one on the cube that
holds only the listed bands, ``raw.index_select(band_axis, bands).contiguous()``: the kernels read the same samples in
the same K order, so the validity mask, its counts, the apply outputs, the conv0 map (workspace offset 0), the labels and
the logits are bit-identical.  The fit's mean and Gram are float64 sums whose atomic accumulation order is not fixed from
run to run (nor between two calls of the same entry point), so they match to 1e-12 and its pixel count exactly.

The dropped bands are poisoned (NaN / Inf and extremes in float32, the fill value, zeros and the type's extremes in the
integer types): no output may change, and no pixel may turn no-data."""
import numpy as np
import pytest
import torch

from scene_harness import as_layout, path_mode, scene_net

pytestmark = pytest.mark.gpu

TORCH = {"u16": torch.uint16, "i16": torch.int16, "f32": torch.float32}
AXIS = {"bip": 2, "bil": 1, "bsq": 0}           # band axis of as_layout's [rows, cols, B] -> layout tensors (BIP: 1 of 2-D)
FILL = {"u16": 65535, "i16": -9999, "f32": -1.0}          # never a value of the synthetic scenes
HYPERION_GOOD = np.array([b for b in range(242) if not (b < 8 or 57 <= b < 77 or 224 <= b < 242)], dtype=np.int32)
WIDE = np.array(sorted(set(range(0, 425, 2)) | set(range(1, 175, 2))), dtype=np.int32)       # 300 of 425
# the layouts and sample types, each layout with two types and each type with two layouts
COMBOS = [("bip", "u16"), ("bil", "i16"), ("bsq", "f32"), ("bip", "f32"), ("bil", "u16"), ("bsq", "i16")]


def _cube(R, C, B, sample, bands, seed, holes=0):
    """A synthetic [R, C, B] raw cube of the sample type whose unlisted bands are poisoned; ``holes`` pixels have the
    fill value in one listed band."""
    from cmlpl_b200 import synth
    u16, _ = synth.synth_scene(R, C, B, 9, seed=seed)
    cube = {"u16": u16, "i16": (u16.astype(np.int32) - 4000).astype(np.int16),
            "f32": u16.astype(np.float32) * np.float32(1e-4)}[sample]
    drop = np.setdiff1d(np.arange(B), bands)
    rng = np.random.default_rng(seed)
    if sample == "f32":
        poison = np.array([np.nan, np.inf, -np.inf, 3e38, -3e38, 0.0, FILL[sample]], dtype=np.float32)
    else:
        info = np.iinfo(cube.dtype)
        poison = np.array([FILL[sample], 0, info.min, info.max], dtype=cube.dtype)
    cube[:, :, drop] = rng.choice(poison, size=(R, C, drop.size))
    cube[:, :, drop[::3]] = poison[0]                  # some dropped bands are fill / NaN everywhere
    if holes:
        idx = rng.choice(R * C, holes, replace=False)
        cube.reshape(-1, B)[idx, bands[rng.integers(0, bands.size, holes)]] = FILL[sample]
    return cube


def _both(cube, layout, bands, dev):
    """(the raw cube in the layout, the oracle: the same holding only the listed bands)"""
    raw = as_layout(cube, layout, dev)
    sel = torch.from_numpy(bands.astype(np.int64)).to(dev)
    return raw, raw.index_select(1 if layout == "bip" else AXIS[layout], sel).contiguous()


def _fit_pair(raw, compact, layout, bands, fill, rows, cols):
    """The mask and the fit with a list, and without on the compacted cube; checks mask, counts and moments."""
    from cmlpl_b200 import preprocess
    v, n, miss = preprocess.valid_mask(raw, fill, layout, cols=cols, bands=bands)
    v0, n0, miss0 = preprocess.valid_mask(compact, fill, layout, cols=cols)
    assert torch.equal(v, v0) and n == n0 and np.array_equal(miss, miss0)
    mask_all = preprocess.valid_mask(raw, fill, layout, cols=cols)[1]
    assert mask_all == 0 and n > 0                      # the poison alone would mark every pixel no-data
    raw_f = raw.view(rows, cols, -1) if layout == "bip" else raw
    cmp_f = compact.view(rows, cols, -1) if layout == "bip" else compact
    pp = preprocess.fit(raw_f, interleave=layout, valid=v, bands=bands)
    pp0 = preprocess.fit(cmp_f, interleave=layout, valid=v0)
    assert list(pp.bands) == list(bands) and pp.raw_bands == raw_f.shape[AXIS[layout]]
    for a, b in ((pp.mu, pp0.mu), (pp.sigma, pp0.sigma)):
        assert np.abs(a - b).max() <= 1e-12 * np.abs(b).max()
    return v, pp, pp0


@pytest.mark.parametrize("layout,sample", COMBOS)
def test_mask_fit_and_apply_read_only_the_listed_bands(dev, layout, sample):
    from cmlpl_b200 import preprocess
    R, C, bands = 37, 41, HYPERION_GOOD
    cube = _cube(R, C, 242, sample, bands, seed=7, holes=50)
    raw, compact = _both(cube, layout, bands, dev)
    v, pp, pp0 = _fit_pair(raw, compact, layout, bands, FILL[sample], R, C)
    assert int(v.sum()) >= R * C - 50
    # apply (BIP): the compacted fit's parameters with and without the list
    pp0.bands, pp0.raw_bands = None, len(bands)
    pps = preprocess.Preproc(pp0.mu, pp0.sigma, pp0.U, pp0.pca_mu, pp0.pca_sigma, bands=bands, raw_bands=242)
    rb, cb = _both(cube, "bip", bands, dev)
    for valid in (None, v.view(-1)):
        got = preprocess.apply(rb, pps, valid=valid, bands=bands)
        want = preprocess.apply(cb, pp0, valid=valid)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
        assert got[1].shape == (R * C, len(bands))


def _scene_pair(dev, layout, sample, B, bands, K, w, masked, mode=1, R=40, C=48, seed=11):
    """One scene call with the list and one on the compacted cube, same folded parameters and explicit workspaces:
    labels, logits and the conv0 map must be equal bit for bit."""
    from cmlpl_b200 import ops, preprocess
    cube = _cube(R, C, B, sample, bands, seed=seed, holes=30 if masked else 0)
    raw, compact = _both(cube, layout, bands, dev)
    v = preprocess.valid_mask(raw, FILL[sample], layout, cols=C, bands=bands)[0] if masked else None
    raw_f = compact.view(R, C, -1) if layout == "bip" else compact
    pp0 = preprocess.fit(raw_f, interleave=layout, valid=v)
    net, _ = scene_net(len(bands), K, w, seed, dev)
    folded0 = pp0.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    folded = dict(folded0, bands=bands, raw_bands=B)
    packed = net.packed_weights(w)
    out = []
    with path_mode(mode):
        for f, x in ((folded, raw), (folded0, compact)):
            ws = ops.scene_workspace(R, C, len(bands), K, w, dev).zero_()
            lab, log = ops.scene_infer_raw(x, f, packed, K, C, w, want_logits=True, workspace=ws, interleave=layout, valid=v)
            out.append((lab, log, ws[:(R + w - 1) * (C + w - 1) * 128]))
    torch.cuda.synchronize()
    (l1, g1, f1), (l0, g0, f0) = out
    assert torch.equal(f1, f0), "conv0 map"
    assert torch.equal(l1, l0) and torch.equal(g1, g0)
    assert torch.isfinite(g1).all()
    if masked:
        assert int((l1 == ops.NODATA_LABEL).sum()) == int((v == 0).sum()) > 0
    return l1


@pytest.mark.parametrize("layout,sample", COMBOS)
@pytest.mark.parametrize("w", [20, 11])
def test_dense_path_196_of_242(dev, layout, sample, w):
    _scene_pair(dev, layout, sample, 242, HYPERION_GOOD, 16, w, masked=(layout, sample) in COMBOS[::2])


@pytest.mark.parametrize("layout,sample", COMBOS[:3])
@pytest.mark.parametrize("masked", [False, True])
def test_k_sliced_conv0_and_cuda_core_head_300_of_425(dev, layout, sample, masked):
    _scene_pair(dev, layout, sample, 425, WIDE, 22, 20, masked, R=24, C=36)


@pytest.mark.parametrize("layout,sample", COMBOS[3:])
@pytest.mark.parametrize("K", [9, 22])
def test_path_mode_0(dev, layout, sample, K):
    _scene_pair(dev, layout, sample, 242, HYPERION_GOOD, K, 11 if K == 22 else 20, masked=K == 9, mode=0)


@pytest.mark.parametrize("layout,sample", COMBOS[:3])
def test_identity_list_equals_the_entry_points_without_a_list(dev, layout, sample):
    """bands = 0..B-1 runs the same kernels' list instantiation; every output equals the existing entry points'."""
    from cmlpl_b200 import ops, preprocess
    R, C, B, K, w = 33, 40, 103, 9, 20
    bands = np.arange(B, dtype=np.int32)
    cube = _cube(R, C, B, sample, bands, seed=5, holes=20)
    raw = as_layout(cube, layout, dev)
    v, n, miss = preprocess.valid_mask(raw, FILL[sample], layout, cols=C, bands=bands)
    v0, n0, miss0 = preprocess.valid_mask(raw, FILL[sample], layout, cols=C)
    assert torch.equal(v, v0) and n == n0 and np.array_equal(miss, miss0)
    raw_f = raw.view(R, C, B) if layout == "bip" else raw
    pp0 = preprocess.fit(raw_f, interleave=layout, valid=v0)
    pp = preprocess.fit(raw_f, interleave=layout, valid=v0, bands=bands)
    assert np.abs(pp.mu - pp0.mu).max() <= 1e-12 * np.abs(pp0.mu).max()
    net, _ = scene_net(B, K, w, 3, dev)
    folded0 = pp0.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    packed = net.packed_weights(w)
    for valid in (None, v0):
        a = ops.scene_infer_raw(raw, dict(folded0, bands=bands, raw_bands=B), packed, K, C, w, want_logits=True,
                                interleave=layout, valid=valid)
        b = ops.scene_infer_raw(raw, folded0, packed, K, C, w, want_logits=True, interleave=layout, valid=valid)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    if layout == "bip":
        pps = preprocess.Preproc(pp0.mu, pp0.sigma, pp0.U, pp0.pca_mu, pp0.pca_sigma, bands=bands, raw_bands=B)
        for valid in (None, v0.view(-1)):
            a, b = preprocess.apply(raw, pps, valid=valid), preprocess.apply(raw, pp0, valid=valid)
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_hyperion_like_scene_with_zero_filled_bands(dev):
    """Hyperion L1R carries uncalibrated bands as zeros.  dead_bands finds exactly them; a fit over all bands with fill 0
    has no valid pixel, and one that lists a dead band is refused by name; fit(bands=good) + scene_infer_raw meets the
    label bar of the dense path against the per-pixel path."""
    from cmlpl_b200 import _lib, ops, preprocess, synth
    from scene_harness import near_ties_only
    R, C, B, K, w = 64, 72, 242, 12, 20
    u16, _ = synth.synth_scene(R, C, B, K, seed=21)
    dead = np.setdiff1d(np.arange(B), HYPERION_GOOD)
    u16[:, :, dead] = 0
    for layout in ("bil", "bsq"):
        raw = as_layout(u16, layout, dev)
        assert np.array_equal(preprocess.dead_bands(raw, fill=0, interleave=layout), dead)
        assert np.array_equal(preprocess.dead_bands(raw, interleave=layout), dead)       # zero variance without a fill
    raw = as_layout(u16, "bil", dev)
    with pytest.raises(_lib.CmlplError, match="bands missing in every pixel"):
        preprocess.fit(raw, interleave="bil", fill=0)
    with pytest.raises(_lib.CmlplError, match=r"zero variance .*: \[0\]"):
        preprocess.fit(raw, interleave="bil", bands=[0, *HYPERION_GOOD.tolist()])
    pp = preprocess.fit(raw, interleave="bil", bands=HYPERION_GOOD)
    net, _ = scene_net(len(HYPERION_GOOD), K, w, 21, dev)
    folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    assert torch.isfinite(folded["inv_sigma"]).all()
    packed = net.packed_weights(w)
    lab, log = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True, interleave="bil")
    with path_mode(0):
        lab0, log0 = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True, interleave="bil")
    log, log0 = log.cpu().numpy(), log0.cpu().numpy()
    assert np.abs(log - log0).max() <= 1e-3 * np.abs(log0).max()
    assert near_ties_only(lab.cpu().numpy(), lab0.cpu().numpy(), log0)


@pytest.mark.parametrize("layout,sample", COMBOS[:3])
@pytest.mark.parametrize("masked", [False, True])
def test_streamed_raw_scene_with_a_band_list(dev, layout, sample, masked):
    """StreamedRawScene takes the list from its Preproc and equals the one-shot call; a BSQ cube moves only the listed
    planes (nsel / B of the bytes)."""
    from cmlpl_b200 import ops, preprocess
    from cmlpl_b200.tools.hyper_tools import StreamedRawScene
    R, C, B, K, w = 44, 40, 242, 9, 20
    bands = HYPERION_GOOD
    cube = _cube(R, C, B, sample, bands, seed=31, holes=25 if masked else 0)
    raw = as_layout(cube, layout, dev)
    fill = FILL[sample] if masked else None
    v = preprocess.valid_mask(raw, fill, layout, cols=C, bands=bands)[0] if masked else None
    pp = preprocess.fit(raw.view(R, C, B) if layout == "bip" else raw, interleave=layout, valid=v, bands=bands)
    net, _ = scene_net(len(bands), K, w, 31, dev)
    folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    packed = net.packed_weights(w)
    one = ops.scene_infer_raw(raw, folded, packed, K, C, w, interleave=layout, valid=v)
    host = torch.from_numpy(np.ascontiguousarray(raw.cpu().numpy())).pin_memory()
    full = host.numel() * host.element_size()
    for nsplit in (1, 3):
        st = StreamedRawScene(pp, R, C, B, K, w, nsplit=nsplit, raw_dtype=TORCH[sample], interleave=layout, fill=fill)
        for _ in range(3):
            st(packed, host, folded=folded)
            assert torch.equal(st.wait().to(dev), one), nsplit
        assert st.h2d_bytes == (full * len(bands) // B if layout == "bsq" else full)
