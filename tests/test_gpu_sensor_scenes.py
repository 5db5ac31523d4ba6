"""Device preprocessing and the raw-cube entry point on sensor-like scenes (-m gpu): ``oracle.sensor_scene`` cubes,
whose band covariance has lambda_1 / lambda_60 of 1e5 to 1e8, so the trailing z-scored PCA components are small
differences of large band values.  Everything is compared with the oracle's float64 preprocessing
(``preprocess_params`` / ``apply_preprocess`` / ``test_whole``); the bars are the error bounds of
test_sensor_scenes_cpu.py, evaluated from each case's own operands, and every case prints its error, its bar and
their ratio.

  1. fit: mean and Gram to 1e-12 of numpy float64; U against the oracle's: the same sign for every one of the 60
     components, and 1 - |cos| within the perturbation bound of the Gram difference; pca_sigma to 1e-8;
  2. apply: spectra and the PCA cube per pixel and component within their first-order f32 bounds;
  3. the conv0 map of the three raw conv0 variants within half an fp16 ulp plus the hi / lo cancellation term;
  4. scene_infer_raw and StreamedRawScene (apply -> scene_infer) with the device fit, unchanged, against test_whole;
  5. a net trained by sample_generation + train on a sensor-like scene, deployed on the raw uint16 cube;
  6. a PaviaU-size sensor-like scene, fitted on all its pixels."""
import numpy as np
import pytest
import torch

import dense_refs as D
from oracle import cmlpl_oracle as O
from scene_harness import as_layout, fit_moments, near_ties_only, path_mode, rel
from test_sensor_scenes_cpu import apply_bound

pytestmark = pytest.mark.gpu

CODE = {"u16": 0, "f32": 1, "i16": 2}
TORCH = {"u16": torch.uint16, "f32": torch.float32, "i16": torch.int16}


def _scene(R, C, B, K, nd, sample, dc=0.0, seed=None):
    cube, gt = O.sensor_scene(R, C, B, K, nd, seed=B + K if seed is None else seed, sample=sample, dc=dc)
    return cube, gt, O.preprocess_params(cube, 60)


def _pp_dict(pp):
    return {"mu": pp.mu, "sigma": pp.sigma, "U": pp.U, "pca_mu": pp.pca_mu, "pca_sigma": pp.pca_sigma}


# ------------------------------------------------------------------------------------------------------------ 1. fit
@pytest.mark.parametrize("B,K,nd,sample,dc,layout", [(103, 9, 1.0, "u16", 20000.0, "bil"), (224, 16, 8.0, "i16", 0.0, "bsq"),
                                                     (270, 22, 1.0, "f32", 0.0, "bil"), (512, 16, 8.0, "u16", 20000.0, "bsq")])
def test_fit_on_sensor_scenes(dev, B, K, nd, sample, dc, layout):
    """Mean and Gram within 1e-12 of the largest entry (float64 atomics reorder the sums), through the BIP path and a
    band-major layout.  U: every component has the oracle's sign, and 1 - |cos| <= 8 (||dG||_2 / gap_k)^2 + B * 2^-52,
    Davis-Kahan with dG the difference between the covariance the device fit decomposes and np.cov (with a factor 4 on
    the angle) plus the host SVD's own orthogonality level.  pca_sigma within 1e-8."""
    from cmlpl_b200 import preprocess
    R, C = 60, 70
    cube, _, ref = _scene(R, C, B, K, nd, sample, dc)
    X = cube.reshape(-1, B).astype(np.float64)
    mu = X.mean(0)
    gram = (X - mu).T @ (X - mu)
    for il in ("bip", layout):
        m, g = fit_moments(as_layout(cube, il, dev), CODE[sample] | preprocess.INTERLEAVE[il], R if il != "bip" else R * C,
                           C if il != "bip" else None, B)
        err_m, err_g = np.abs(m - mu).max() / np.abs(mu).max(), np.abs(g - gram).max() / np.abs(gram).max()
        print("B = %d, %s, %s: mean %.1e, Gram %.1e of the largest entry" % (B, sample, il, err_m, err_g))
        assert err_m <= 1e-12 and err_g <= 1e-12
    pp = preprocess.fit(as_layout(cube, layout, dev), 60, interleave=layout)
    dG = np.linalg.norm(g / (R * C - 1) - np.cov((X - mu).T), 2)
    ev = np.linalg.eigvalsh(np.cov((X - mu).T))[::-1]
    gap = np.minimum(np.abs(ev[:60] - np.r_[np.inf, ev[:59]]), np.abs(ev[:60] - ev[1:61]))
    bar = 8 * (dG / gap) ** 2 + B * 2.0 ** -52
    cos = np.sum(pp.U * ref["U"], 0)
    print("B = %d, %s, %.0f DN: lambda_1/lambda_60 %.1e, ||dG|| / lambda_1 %.1e; worst 1 - |cos| %.1e (bar %.1e, "
          "largest ratio %.2f); signs flipped: %d" % (B, sample, nd, ev[0] / ev[59], dG / ev[0], (1 - np.abs(cos)).max(),
                                                      bar[np.argmax(1 - np.abs(cos))], ((1 - np.abs(cos)) / bar).max(),
                                                      int((cos < 0).sum())))
    assert np.all(cos > 0), "a component of the device U has the opposite sign of the reference's"
    assert np.all(1 - np.abs(cos) <= bar)
    assert rel(pp.mu, ref["mu"]) < 1e-12 and rel(pp.sigma, ref["sigma"]) < 1e-12
    assert np.abs(pp.pca_sigma / ref["pca_sigma"] - 1).max() < 1e-8


# ---------------------------------------------------------------------------------------------------------- 2. apply
@pytest.mark.parametrize("B,K,nd,sample,dc", [(103, 9, 8.0, "u16", 20000.0), (103, 9, 0.5, "u16", 20000.0),
                                              (224, 16, 1.0, "i16", 0.0), (270, 22, 1.0, "f32", 0.0)])
def test_apply_on_sensor_scenes(dev, B, K, nd, sample, dc):
    """preprocess.apply with the device fit against float64 with the same parameters.  Spectra: |err| <= (|mu32 - mu| +
    2u |x - mu|) / sigma + u |ref| per element (the band means' f32 rounding, the centring and the scaling; no
    cancellation) and 1e-6 of the largest entry.  PCA cube: apply_bound per pixel and component."""
    from cmlpl_b200 import preprocess
    cube, _, _ = _scene(64, 50, B, K, nd, sample, dc)
    X = cube.reshape(-1, B).astype(np.float64)
    raw = torch.from_numpy(cube.reshape(-1, B).copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    got, spec = preprocess.apply(raw, pp)
    d = pp.device_params(dev)
    mu32 = d["mu"].cpu().numpy().astype(np.float64)
    u = 2.0 ** -24
    ref_s = (X - pp.mu) / pp.sigma
    bar_s = (np.abs(mu32 - pp.mu) + 2 * u * np.abs(X - pp.mu)) / pp.sigma + 2 * u * np.abs(ref_s)
    err_s = np.abs(spec.cpu().numpy() - ref_s)
    Us, sh = pp.U / pp.pca_sigma[None], pp.pca_mu / pp.pca_sigma
    ref = (X - pp.mu) @ Us - sh
    bound = apply_bound(X, mu32, pp.mu, d["Us"].cpu().numpy(), sh)
    err = np.abs(got.cpu().numpy() - ref)
    r = err / bound
    print("B = %d, %s, %.1f DN: spectra err / bar %.3f (%.1e of max); PCA cube: worst error %.2e (trailing 30 "
          "components %.2e), its bar %.2e, largest err / bar %.3f" % (B, sample, nd, (err_s / bar_s).max(),
                                                                      rel(spec.cpu(), ref_s), err.max(), err[:, 30:].max(),
                                                                      bound.flat[np.argmax(r)], r.max()))
    assert np.all(err_s <= bar_s) and rel(spec.cpu(), ref_s) < 1e-6
    assert np.all(err <= bound)


# ------------------------------------------------------------------------------------------------- 3. conv0 map
@pytest.mark.parametrize("B,nd,sample,dc,layout", [(103, 1.0, "u16", 20000.0, "bip"), (224, 1.0, "u16", 0.0, "bsq"),
                                                   (270, 8.0, "i16", 0.0, "bil"), (512, 1.0, "f32", 0.0, "bip")])
def test_raw_conv0_map_on_sensor_scenes(dev, B, nd, sample, dc, layout):
    """The conv0 map (workspace offset 0, chunk-planar fp16 [8][R+w-1][C+w-1][8]) of conv0_tc_kernel (103 / 224 bands
    BIP), its band-major instantiation (224 BSQ), and the K-sliced kernel (270 BIL, 512 BIP), against the folded 1x1 conv
    in float64 on the mirror-padded scene: per position and channel within conv0_bar (half an fp16 ulp + the hi / lo
    cancellation term), and 1e-3 of the largest entry overall."""
    q, e = D.raw_conv0_map_check(dev, 23, 31, B, 9, 20, nd, sample, dc, layout)
    print("B = %d, %s, %s, %.0f DN: conv0 map error / max|F0| %.1e; worst error / bar %.3f" % (B, sample, layout, nd, e, q))
    assert q <= 1.0
    assert e < 1e-3


# --------------------------------------------------------------------------------------- 4. raw entry point, oracle
#          B    K   w   noise sample  dc       path
RAW_CASES = [(103, 9, 20, 8.0, "u16", 20000.0, 1),     # dense path, tensor-core spectral head
             (103, 9, 11, 1.0, "u16", 0.0, 1),         # dense path, 11 x 11 windows
             (224, 16, 20, 1.0, "i16", 0.0, 1),        # dense path at 224 bands
             (103, 22, 20, 8.0, "u16", 0.0, 0),        # path mode 0 (per-pixel kernels), 17-32 classes
             (270, 32, 20, 1.0, "f32", 0.0, 1),        # K-sliced conv0, CUDA-core head
             (512, 16, 11, 8.0, "i16", 0.0, 1)]        # K-sliced conv0 at 512 bands, CUDA-core head, w = 11


@pytest.mark.parametrize("B,K,w,nd,sample,dc,mode", RAW_CASES)
def test_raw_entry_point_on_sensor_scenes(dev, B, K, w, nd, sample, dc, mode):
    """The device fit as it comes (no sign alignment), folded into conv0 (scene_infer_raw) and applied by
    StreamedRawScene(pp) (preprocess.apply -> scene_infer), against test_whole on the oracle's float64 preprocessing:
    logits within 1e-3 of the largest, labels = argmax of the logits, label differences only at near ties."""
    from cmlpl_b200 import ops, preprocess
    from cmlpl_b200.tools.hyper_tools import StreamedRawScene
    from cmlpl_b200.tools.models import BaseNet2
    R, C = 29, 37
    cube, _, ref_pp = _scene(R, C, B, K, nd, sample, dc)
    Xp, Xs = O.apply_preprocess(cube, ref_pp)
    raw = torch.from_numpy(cube.reshape(-1, B).copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    torch.manual_seed(B * 7 + K)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    lab_ref, log_ref = O.test_whole(sd, Xp.astype(np.float32), Xs.astype(np.float32), w, odd_mode=(w == 11),
                                    return_logits=True)
    with path_mode(mode):
        packed = net.packed_weights(w)
        folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
        lab, lg = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True)
        cube_d, spec_d = preprocess.apply(raw, pp)
        lab_a, lg_a = ops.scene_infer(cube_d.view(R, C, 60), spec_d, packed, K, w, want_logits=True)
        st = StreamedRawScene(pp, R, C, B, K, w, nsplit=2, raw_dtype=TORCH[sample])
        lab_s = st(packed, torch.from_numpy(cube.reshape(-1, B).copy()).pin_memory())
        torch.cuda.synchronize()
    for name, l, z in (("raw", lab, lg), ("apply", lab_a, lg_a)):
        l, z = l.cpu().numpy(), z.cpu().numpy()
        print("B = %d, K = %d, w = %d, %.0f DN, %s, path mode %d, %s: logit error %.1e of the largest (bar 1e-3), "
              "label agreement %.5f" % (B, K, w, nd, sample, mode, name, rel(z, log_ref), float(np.mean(l == lab_ref))))
        assert rel(z, log_ref) < 1e-3
        assert np.array_equal(l, z.argmax(1))
        assert near_ties_only(l, lab_ref, log_ref)
    assert torch.equal(lab_s.cpu(), lab_a.cpu())


# ------------------------------------------------------------------------------------------- 5. deployment, trained
def test_trained_net_deployed_on_the_raw_cube(dev, tmp_path, monkeypatch):
    """sample_generation (host float64 preprocessing) + train for 2 epochs on a 150 x 140 x 103 sensor-like scene; then
    the deployment path: preprocess.fit on the device from the raw uint16 cube and folded_conv0 of the trained weights.
    >= 99.9 % of its labels equal train.main's own label map and the oracle's test_whole, differences only at near ties;
    OA and kappa through CalAccuracy within the label disagreement."""
    from cmlpl_b200 import ops, preprocess, sample_generation as SG, train as T
    from cmlpl_b200.tools import hyper_tools as H
    R, C, B, K = 150, 140, 103, 9
    cube, gt = O.sensor_scene(R, C, B, K, 4.0, seed=1503, sample="u16", dc=1000.0)
    monkeypatch.setattr(SG, "load_scene", lambda *a, **k: (cube, gt))
    root = str(tmp_path) + "/"
    SG.main(SG.build_parser().parse_args(["--dataID", "1", "--root", root]))
    T.seed_torch()
    out = T.main(T.build_parser().parse_args(["--dataID", "1", "--root", root, "--num_epochs", "2", "--num_unlabel",
                                              "2048", "--print_per_batches", "5"]))
    net = out["state"].Base.eval()
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    d = root + H.DATASETS[1][0] + "/"
    lab_ref, log_ref = O.test_whole(sd, np.load(d + "XPCA.npy"), np.load(d + "X.npy").astype(np.float32), 20,
                                    return_logits=True)
    raw = torch.from_numpy(cube.reshape(-1, B).copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    lab, lg = ops.scene_infer_raw(raw, pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev), net.packed_weights(20), K,
                                  C, 20, want_logits=True)
    lab, lg = lab.cpu().numpy(), lg.cpu().numpy()
    own = np.asarray(out["predict_label"])
    a_own, a_ref = float(np.mean(lab == own)), float(np.mean(lab == lab_ref))
    te = np.load(d + "test_array.npy")
    Y = np.load(d + "Y.npy").astype(np.int64) - 1
    OA, kappa, _ = H.CalAccuracy(lab[te], Y[te])
    OA_t, kappa_t, _ = out["results"][0]
    dis = float(np.mean(lab[te] != own[te]))
    print("trained net, raw uint16 cube + device fit: label agreement with train.main %.5f, with the oracle %.5f; logit "
          "error %.1e; OA %.4f vs %.4f, kappa %.4f vs %.4f" % (a_own, a_ref, rel(lg, log_ref), OA, OA_t, kappa, kappa_t))
    assert OA_t > 1.0 / K
    assert a_own >= 0.999 and a_ref >= 0.999
    assert rel(lg, log_ref) < 1e-3 and near_ties_only(lab, lab_ref, log_ref)
    # a fraction d of changed labels moves OA by at most d and the chance agreement p_e by at most 2d, so kappa =
    # (OA - p_e) / (1 - p_e) by at most 3d / (1 - p_e - 2d)^2
    n = te.size
    pe = float(np.bincount(Y[te], minlength=K) @ np.bincount(lab[te], minlength=K)) / n ** 2
    assert abs(OA - OA_t) <= dis + 1e-12 and abs(kappa - kappa_t) <= 3 * dis / (1 - pe - 2 * dis) ** 2 + 1e-12


# ---------------------------------------------------------------------------------------------- 6. full size
def test_full_size_sensor_scene(dev):
    """610 x 340 x 103 (PaviaU's shape), 2 DN: fit on all 207 400 pixels, then the raw entry point; a pixel every 6007
    against the oracle's float64 preprocessing + BaseNet2 forward (1e-3 of the largest logit); labels = argmax."""
    from cmlpl_b200 import ops, preprocess
    R, C, B, K, w = 610, 340, 103, 9, 20
    cube, _, ref_pp = _scene(R, C, B, K, 2.0, "u16", 0.0, seed=610)
    raw = torch.from_numpy(cube.reshape(-1, B)).to(dev)
    pp = preprocess.fit(raw, 60)
    assert np.all(np.sum(pp.U * ref_pp["U"], 0) > 0)
    torch.manual_seed(610)
    sd = O.basenet2_init(B, K)
    packed = ops.pack_basenet2({k: v.to(dev) for k, v in sd.items()}, B, K, w)
    lab, lg = ops.scene_infer_raw(raw, pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev), packed, K, C, w,
                                  want_logits=True)
    idx = np.arange(0, R * C, 6007)
    Xp, Xs = O.apply_preprocess(cube, ref_pp)
    with torch.no_grad():
        ref, _ = O.basenet2_forward(sd, torch.from_numpy(O.extract_patches_at(Xp.astype(np.float32), w, idx)),
                                    torch.from_numpy(Xs[idx].astype(np.float32)))
    got = lg.cpu().numpy()[idx]
    print("full-size sensor-like scene: logit error at %d sampled pixels %.1e of the largest" % (idx.size,
                                                                                                  rel(got, ref.numpy())))
    assert rel(got, ref.numpy()) < 1e-3
    assert torch.equal(lab, lg.argmax(1).to(torch.uint8))
