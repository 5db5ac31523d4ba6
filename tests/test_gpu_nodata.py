"""No-data pixels on the GPU (-m gpu): the validity mask, the masked fit and apply, and cmlpl_scene_infer_raw_masked,
against the float64 definitions of test_nodata_cpu.py.

  1. mask: cmlpl_valid_mask_u8 equals numpy exactly (mask bytes, n_valid, band_missing) in every sample type and
     interleave; fills u16 0, i16 -32768, f32 -9999 and f32 NaN-only;
  2. fit: against numpy float64 on X[valid] with the bars of test_gpu_sensor_scenes.py::test_fit_on_sensor_scenes;
     an all-fill band raises an error that names it;
  3. apply: first-order bounds on valid rows, exact imputed values on no-data rows;
  4. labels and logits against the oracle (impute, test_whole, 255) across the raw entry point's paths;
  5. locality: a pixel whose window holds no no-data pixel gets bit-identical logits with and without the mask;
  6. an all-valid mask is bit-identical to the unmasked call;
  7. row bands and StreamedRawScene(fill=...) are bit-identical to one masked call;
  8. the reference-trained hard scene with a corner wedge cut to fill."""
import numpy as np
import pytest
import torch

from oracle import cmlpl_oracle as O
from test_gpu_many_classes import near_ties_only, path_mode, rel
from test_gpu_raw_layouts import as_layout
from test_nodata_cpu import (NODATA, masked_params, nodata_pattern, scene_oracle, valid_mask,
                             window_touches, with_nodata)
from test_sensor_scenes_cpu import apply_bound

pytestmark = pytest.mark.gpu

TORCH = {"u16": torch.uint16, "f32": torch.float32, "i16": torch.int16}
FILL = {"u16": 0, "i16": -32768, "f32": None}


def _pp(d):
    from cmlpl_b200 import preprocess
    return preprocess.Preproc(mu=d["mu"], sigma=d["sigma"], U=d["U"], pca_mu=d["pca_mu"], pca_sigma=d["pca_sigma"])


def _dirty_scene(R, C, B, K, sample, kind, seed, fill="default"):
    cube, _ = O.sensor_scene(R, C, B, K, 8.0, seed=seed, sample=sample, dc=20000.0 if sample == "u16" else 0.0)
    fill = FILL[sample] if fill == "default" else fill
    nd = nodata_pattern(R, C, kind, seed)
    dirty = with_nodata(cube, nd, fill, seed)
    valid, n, _ = valid_mask(dirty, fill)
    assert np.array_equal(valid == 0, nd)
    return dirty, valid, fill


# ------------------------------------------------------------------------------------------------------------ 1. mask
@pytest.mark.parametrize("sample,fill", [("u16", 0), ("i16", -32768), ("f32", -9999.0), ("f32", None)])
def test_mask_matches_numpy(dev, sample, fill):
    from cmlpl_b200 import preprocess
    R, C = 41, 53
    for B in (103, 270):
        cube, _ = O.sensor_scene(R, C, B, 9, 8.0, seed=B, sample=sample, dc=20000.0 if sample == "u16" else 0.0)
        for kind in ("wedge", "lines", "pixels"):
            dirty = with_nodata(cube, nodata_pattern(R, C, kind, B), fill, B)
            if sample == "f32" and fill is not None:
                dirty[3, 4, 7] = np.nan                  # non-finite samples are missing whatever the fill
            want = valid_mask(dirty, fill)
            for il in ("bip", "bil", "bsq"):
                got = preprocess.valid_mask(as_layout(dirty, il, dev), fill, il, cols=C if il == "bip" else None)
                assert np.array_equal(got[0].cpu().numpy().reshape(R, C), want[0]), (B, kind, il)
                assert got[1] == want[1] and np.array_equal(got[2], want[2]), (B, kind, il)


# ------------------------------------------------------------------------------------------------------------- 2. fit
@pytest.mark.parametrize("B,K,sample,layout,kind", [(103, 9, "u16", "bil", "wedge"), (224, 16, "i16", "bsq", "lines"),
                                                    (270, 22, "f32", "bil", "edge"), (512, 16, "u16", "bsq", "pixels")])
def test_masked_fit_matches_numpy_on_the_valid_pixels(dev, B, K, sample, layout, kind):
    """Mean and Gram within 1e-12 of the largest entry of numpy float64 on X[valid] (BIP and a band-major layout);
    n_valid exact; every U component with the oracle's sign and within the Davis-Kahan bound; pca_sigma within 1e-8."""
    from cmlpl_b200 import _lib, preprocess
    R, C = 60, 70
    dirty, valid, fill = _dirty_scene(R, C, B, K, sample, kind, B + K)
    X = dirty.reshape(-1, B)[valid.reshape(-1) != 0].astype(np.float64)
    mu = X.mean(0)
    gram = (X - mu).T @ (X - mu)
    ref = masked_params(dirty, valid)
    for il in ("bip", layout):
        raw = as_layout(dirty, il, dev)
        v = torch.from_numpy(valid).to(dev)
        mean = torch.empty(B, dtype=torch.float64, device=dev)
        g = torch.empty(B, B, dtype=torch.float64, device=dev)
        cnt = torch.empty(1, dtype=torch.int64, device=dev)
        rows, cols = (R * C, 1) if il == "bip" else (R, C)
        _lib.call("cmlpl_preprocess_fit_masked_f64", raw.data_ptr(), preprocess._dtype_code(raw) | preprocess.INTERLEAVE[il],
                  rows, cols, B, v.data_ptr(), mean.data_ptr(), g.data_ptr(), cnt.data_ptr(),
                  torch.cuda.current_stream().cuda_stream)
        g = g.cpu().numpy()
        g = np.triu(g) + np.triu(g, 1).T
        err_m, err_g = np.abs(mean.cpu().numpy() - mu).max() / np.abs(mu).max(), np.abs(g - gram).max() / np.abs(gram).max()
        print("B = %d, %s, %s, %s: n_valid %d of %d, mean %.1e, Gram %.1e" % (B, sample, il, kind, int(cnt.item()), R * C,
                                                                            err_m, err_g))
        assert int(cnt.item()) == X.shape[0]
        assert err_m <= 1e-12 and err_g <= 1e-12
    pp = preprocess.fit(as_layout(dirty, layout, dev), 60, interleave=layout, valid=torch.from_numpy(valid).to(dev))
    n = X.shape[0]
    dG = np.linalg.norm(g / (n - 1) - np.cov((X - mu).T), 2)
    ev = np.linalg.eigvalsh(np.cov((X - mu).T))[::-1]
    gap = np.minimum(np.abs(ev[:60] - np.r_[np.inf, ev[:59]]), np.abs(ev[:60] - ev[1:61]))
    bar = 8 * (dG / gap) ** 2 + B * 2.0 ** -52
    cos = np.sum(pp.U * ref["U"], 0)
    assert np.all(cos > 0) and np.all(1 - np.abs(cos) <= bar)
    assert rel(pp.mu, ref["mu"]) < 1e-12 and rel(pp.sigma, ref["sigma"]) < 1e-12
    assert np.abs(pp.pca_sigma / ref["pca_sigma"] - 1).max() < 1e-8


def test_an_all_fill_band_is_named(dev):
    from cmlpl_b200 import _lib, preprocess
    R, C, B = 20, 30, 103
    cube, _ = O.sensor_scene(R, C, B, 9, 8.0, seed=5, sample="i16")
    cube[:, :, 41] = -32768
    v, n, miss = preprocess.valid_mask(as_layout(cube, "bil", dev), -32768, "bil")
    assert n == 0 and miss[41] == R * C and miss.sum() == R * C
    with pytest.raises(_lib.CmlplError, match=r"0 valid pixels of 600.*bands missing in every pixel: \[41\]"):
        preprocess.fit(as_layout(cube, "bil", dev), 60, interleave="bil", fill=-32768)


# ----------------------------------------------------------------------------------------------------------- 3. apply
@pytest.mark.parametrize("B,sample", [(103, "u16"), (224, "i16"), (270, "f32")])
def test_masked_apply(dev, B, sample):
    """Valid rows within the first-order bounds of test_gpu_sensor_scenes.py::test_apply_on_sensor_scenes; no-data rows
    exactly the imputed values: spectra 0, PCA cube -shift."""
    from cmlpl_b200 import preprocess
    R, C = 64, 50
    dirty, valid, fill = _dirty_scene(R, C, B, 9, sample, "wedge", B)
    raw = as_layout(dirty, "bip", dev)
    vd = torch.from_numpy(valid).to(dev)
    pp = preprocess.fit(raw, 60, valid=vd)
    got, spec = preprocess.apply(raw, pp, valid=vd)
    got, spec = got.cpu().numpy(), spec.cpu().numpy()
    d = pp.device_params(dev)
    nd = valid.reshape(-1) == 0
    assert np.all(spec[nd] == 0) and np.array_equal(got[nd], np.broadcast_to(-d["shift"].cpu().numpy(), (nd.sum(), 60)))
    X = dirty.reshape(-1, B)[~nd].astype(np.float64)
    mu32 = d["mu"].cpu().numpy().astype(np.float64)
    u = 2.0 ** -24
    ref_s = (X - pp.mu) / pp.sigma
    bar_s = (np.abs(mu32 - pp.mu) + 2 * u * np.abs(X - pp.mu)) / pp.sigma + 2 * u * np.abs(ref_s)
    assert np.all(np.abs(spec[~nd] - ref_s) <= bar_s)
    sh = pp.pca_mu / pp.pca_sigma
    ref = (X - pp.mu) @ (pp.U / pp.pca_sigma[None]) - sh
    assert np.all(np.abs(got[~nd] - ref) <= apply_bound(X, mu32, pp.mu, d["Us"].cpu().numpy(), sh))


# ------------------------------------------------------------------------------------------ 4-6. the masked entry point
#          B    K   w  mode sample layout kind
CASES = [(103, 9, 20, 1, "u16", "bip", "wedge"),       # dense path, tensor-core spectral branch
         (103, 22, 20, 1, "i16", "bil", "lines"),      # dense path, 17-32 classes
         (103, 9, 11, 1, "f32", "bsq", "edge"),        # dense path, 11 x 11 windows, NaN / Inf
         (103, 22, 20, 0, "u16", "bsq", "pixels"),     # path mode 0: per-pixel kernels + classify, 17-32 classes
         (200, 9, 11, 0, "f32", "bip", "wedge"),       # path mode 0 at <= 16 classes
         (240, 16, 20, 1, "u16", "bsq", "edge"),       # conv0_tc (band-major) + CUDA-core head (RawBandZA)
         (240, 9, 20, 1, "f32", "bip", "lines"),       # conv0_tc + CUDA-core head (RawZA)
         (270, 22, 20, 1, "i16", "bip", "wedge"),      # K-sliced conv0 + CUDA-core head
         (300, 9, 11, 1, "u16", "bil", "edge")]        # K-sliced band-major conv0, w = 11


def _net(B, K, w, seed, dev):
    from cmlpl_b200.tools.models import BaseNet2
    torch.manual_seed(seed)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    return net, {k: v.detach().cpu() for k, v in net.state_dict().items()}


@pytest.mark.parametrize("B,K,w,mode,sample,layout,kind", CASES)
def test_masked_scene_against_the_oracle(dev, B, K, w, mode, sample, layout, kind):
    """4: against the oracle (impute, test_whole, 255): logits within 1e-3 of the largest (no-data pixels: those of the
    imputed pixel), >= 99.9 % of the valid pixels' labels identical and every difference a near tie, every no-data
    pixel 255.  5: with the same folded parameters and no mask, every pixel whose window holds no no-data pixel has
    bit-identical logits.  6: an all-valid mask is bit-identical to the unmasked call."""
    from cmlpl_b200 import ops
    R, C = 60, 70
    dirty, valid, fill = _dirty_scene(R, C, B, K, sample, kind, B + K + w)
    ref_pp = masked_params(dirty, valid)
    net, sd = _net(B, K, w, B * 7 + K, dev)
    lab_ref, log_ref = scene_oracle(sd, dirty, valid, ref_pp, w)
    raw = as_layout(dirty, layout, dev)
    vd = torch.from_numpy(valid).to(dev)
    with path_mode(mode):
        packed = net.packed_weights(w)
        folded = _pp(ref_pp).folded_conv0(net.conv0.weight, net.conv0.bias, dev)
        lab, lg = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True, interleave=layout, valid=vd)
        lab_u, lg_u = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True, interleave=layout)
        ones = torch.ones_like(vd)
        lab_1, lg_1 = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True, interleave=layout, valid=ones)
        torch.cuda.synchronize()
    lab, lg = lab.cpu().numpy().astype(np.int64), lg.cpu().numpy()
    ok = valid.reshape(-1) != 0
    agree = float(np.mean(lab[ok] == lab_ref[ok]))
    far = ~window_touches(valid == 0, w).reshape(-1)
    print("B = %d, K = %d, w = %d, mode %d, %s %s, %s: %d no-data pixels, %d untouched; logit error %.1e; label agreement "
          "on valid pixels %.5f" % (B, K, w, mode, sample, layout, kind, (~ok).sum(), far.sum(), rel(lg, log_ref), agree))
    assert np.all(lab[~ok] == NODATA)
    assert rel(lg, log_ref) < 1e-3
    assert np.array_equal(lab[ok], lg[ok].argmax(1))
    assert agree >= 0.999 and near_ties_only(lab[ok], lab_ref[ok], log_ref[ok])
    # 5. locality
    assert far.sum() > 0
    assert np.array_equal(lg[far], lg_u.cpu().numpy()[far]) and np.array_equal(lab[far], lab_u.cpu().numpy()[far])
    # 6. no-op mask
    assert torch.equal(lab_1, lab_u) and torch.equal(lg_1, lg_u)


# ------------------------------------------------------------------------------------------------------- 7. row bands
@pytest.mark.parametrize("B,K,w,layout,sample", [(103, 9, 20, "bsq", "u16"), (270, 22, 11, "bil", "f32"),
                                                 (103, 20, 20, "bip", "i16")])
def test_row_bands_and_streamed_scene(dev, B, K, w, layout, sample):
    """Row bands, each from its own halo slab and the slab's own mask, are bit-identical to one call; so is
    StreamedRawScene(fill=...), which builds the mask on the device from the rows it copied."""
    from cmlpl_b200 import ops
    from cmlpl_b200.tools.hyper_tools import StreamedRawScene
    R, C = 60, 37
    dirty, valid, fill = _dirty_scene(R, C, B, K, sample, "edge", B + w)
    dirty[R - 1, 5:9] = with_nodata(dirty[R - 1:, 5:9], np.ones((1, 4), bool), fill)[0]      # the bottom edge too
    valid = valid_mask(dirty, fill)[0]
    net, _ = _net(B, K, w, B + K, dev)
    folded = _pp(masked_params(dirty, valid)).folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    packed = net.packed_weights(w)
    one = ops.scene_infer_raw(as_layout(dirty, layout, dev), folded, packed, K, C, w, want_logits=True, interleave=layout,
                              valid=torch.from_numpy(valid).to(dev))
    lo, hi = w // 2, w - w // 2 - 1
    for a, b in [(0, 7), (7, 31), (31, 60)]:
        s0, s1 = max(0, a - lo), min(R, b + hi)
        got = ops.scene_infer_raw(as_layout(dirty[s0:s1], layout, dev), folded, packed, K, C, w, band_row0=a,
                                  band_rows=b - a, scene_rows=R, slab_row0=s0, want_logits=True, interleave=layout,
                                  valid=torch.from_numpy(np.ascontiguousarray(valid[s0:s1])).to(dev))
        assert torch.equal(got[0], one[0][a * C:b * C]) and torch.equal(got[1], one[1][a * C:b * C]), (a, b)
    row0, rows = 12, 40
    s0, s1 = max(0, row0 - lo), min(R, row0 + rows + hi)
    for nsplit in (1, 3):
        st = StreamedRawScene(None, R, C, B, K, w, nsplit=nsplit, row0=row0, rows=rows, raw_dtype=TORCH[sample],
                              interleave=layout, fill=float("nan") if fill is None else fill)
        host = {"bip": dirty[s0:s1].reshape(-1, B), "bil": dirty[s0:s1].transpose(0, 2, 1),
                "bsq": dirty[s0:s1].transpose(2, 0, 1)}[layout]
        host = torch.from_numpy(np.ascontiguousarray(host)).pin_memory()
        for _ in range(3):                                  # both buffer sets, then the first one again
            st(packed, host, folded=folded)
            assert torch.equal(st.wait().to(dev), one[0][row0 * C:(row0 + rows) * C]), nsplit


# ------------------------------------------------------------------------------------------------ 8. trained network
def test_trained_net_on_the_hard_scene_with_a_wedge(dev, golden_dir):
    """The reference-trained hard scene (tests/golden/hard_scene.npz) with a corner wedge cut to fill (0): under the same
    folded parameters, every valid pixel whose window does not reach the wedge keeps its unmasked label, and every
    wedge pixel is 255."""
    import os
    from cmlpl_b200 import ops
    from cmlpl_b200.tools.models import BaseNet2
    z = np.load(os.path.join(golden_dir, "hard_scene.npz"))
    R, C, B, K = (int(v) for v in z["shape"])
    cube, _ = O.synth_cube_hard(R, C, B, K, seed=int(z["seed"]), spread=float(z["spread"]), sigma=float(z["sigma"]))
    net = BaseNet2(B, 0, K).to(dev).eval()
    net.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}, strict=False)
    pp = {"mu": z["mu"], "sigma": z["sigma_x"], "U": z["U"], "pca_mu": z["pca_mu"], "pca_sigma": z["pca_sigma"]}
    folded = _pp(pp).folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    r, c = np.mgrid[0:R, 0:C]
    wedge = r + c < 0.45 * (R + C) / 2                       # the top-left corner
    dirty = cube.copy()
    dirty[wedge] = 0
    packed = net.packed_weights(20)
    lab_u = ops.scene_infer_raw(torch.from_numpy(cube.reshape(-1, B)).to(dev), folded, packed, K, C, 20).cpu().numpy()
    from cmlpl_b200 import preprocess
    raw = torch.from_numpy(dirty.reshape(-1, B)).to(dev)
    vd, n, _ = preprocess.valid_mask(raw, 0, cols=C)
    assert n == R * C - wedge.sum()
    lab = ops.scene_infer_raw(raw, folded, packed, K, C, 20, valid=vd).cpu().numpy()
    far = ~window_touches(wedge, 20).reshape(-1)
    print("hard scene with a %.1f %% wedge: %d pixels outside its window reach, label agreement there %.5f"
          % (100 * wedge.mean(), far.sum(), float(np.mean(lab[far] == lab_u[far]))))
    assert np.all(lab[wedge.reshape(-1)] == NODATA)
    assert far.sum() > R * C // 2 and np.array_equal(lab[far], lab_u[far])
