"""Label-map parity where it is NOT trivial (VERDICT r1 item 3): tests/golden/hard_scene.npz holds what the UNMODIFIED
reference produced on a 150 x 140 x 103 synthetic scene whose classes overlap (oracle/make_golden.py::gold_hard: the
reference's own sample_generation.main + train.main, 3 epochs; its OA on the scene is ~0.93, so thousands of pixels sit
near a decision boundary).  The scene is regenerated from its seed; preprocessing uses the stored float64 parameters.
Bars: >= 99.9 % identical labels for cmlpl_scene_infer AND for the raw-cube entry point cmlpl_scene_infer_raw
(the headline end-to-end path); logits 1e-3 * max|ref|; OA / kappa through CalAccuracy within the label disagreement."""
import os

import numpy as np
import pytest
import torch

from oracle import cmlpl_oracle as O
from scene_harness import rel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hard(golden_dir):
    z = np.load(os.path.join(golden_dir, "hard_scene.npz"))
    R, C, B, K = (int(v) for v in z["shape"])
    cube, gt = O.synth_cube_hard(R, C, B, K, seed=int(z["seed"]), spread=float(z["spread"]), sigma=float(z["sigma"]))
    chk = np.array([int(cube.astype(np.int64).sum()), int((cube.astype(np.int64) ** 2).sum() % (1 << 61))])
    assert np.array_equal(chk, z["cube_checksum"]), "the regenerated scene differs from the one the reference saw"
    pp = {"mu": z["mu"], "sigma": z["sigma_x"], "U": z["U"], "pca_mu": z["pca_mu"], "pca_sigma": z["pca_sigma"]}
    Xp, Xs = O.apply_preprocess(cube, pp)
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    return dict(z=z, R=R, C=C, B=B, K=K, cube=cube, gt=gt, pp=pp, Xp=Xp.astype(np.float32), Xs=Xs.astype(np.float32), sd=sd)


def make_net(h, dev):
    from cmlpl_b200.tools.models import BaseNet2
    net = BaseNet2(h["B"], 0, h["K"]).to(dev).eval()
    net.load_state_dict(h["sd"], strict=False)
    return net


def test_trained_net_label_map_on_a_hard_scene(dev, hard):
    from cmlpl_b200.tools import hyper_tools as H
    h, z = hard, hard["z"]
    assert h["R"] * h["C"] >= 20000 and 0.8 <= float(z["OA"]) <= 0.95       # not a trivially separable scene
    net = make_net(h, dev)
    cube_d, spec_d = torch.from_numpy(h["Xp"]).to(dev), torch.from_numpy(h["Xs"]).to(dev)
    labels, logits = H.scene_labels(net, cube_d, spec_d, 20, want_logits=True)
    got = labels.cpu().numpy()
    agree = float(np.mean(got == z["predict_label"]))
    print("hard scene: label agreement with the reference's own label map = %.5f (reference OA %.4f)" % (agree, float(z["OA"])))
    assert agree >= 0.999
    band = z["band"]
    assert rel(logits.cpu().numpy()[band], z["logits_band"]) < 1e-3
    # OA / kappa through the device confusion matrix: exactly CalAccuracy of OUR labels, and close to the reference's
    te = z["test_array"]
    Y = z["Y"].astype(np.int64) - 1
    OA, kappa, pa = H.CalAccuracy(got[te], Y[te])
    OA_o, kappa_o, pa_o = O.cal_accuracy(got[te], Y[te])
    assert OA == OA_o and kappa == kappa_o and np.array_equal(pa, pa_o)
    assert abs(OA - float(z["OA"])) <= (1 - agree) + 1e-12 and abs(kappa - float(z["Kappa"])) < 2e-3


def test_raw_cube_entry_point_on_the_hard_scene(dev, hard):
    """cmlpl_scene_infer_raw (uint16 cube in, preprocessing folded into conv0 / the fp16 conversion of the spectra):
    the path bench.py's end-to-end number goes through, against the reference's label map."""
    from cmlpl_b200 import ops, preprocess
    h, z = hard, hard["z"]
    net = make_net(h, dev)
    pp = preprocess.Preproc(mu=h["pp"]["mu"], sigma=h["pp"]["sigma"], U=h["pp"]["U"], pca_mu=h["pp"]["pca_mu"],
                            pca_sigma=h["pp"]["pca_sigma"])
    folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    raw = torch.from_numpy(h["cube"].reshape(-1, h["B"])).to(dev)
    labels, logits = ops.scene_infer_raw(raw, folded, net.packed_weights(20), h["K"], h["C"], 20, want_logits=True)
    agree = float(np.mean(labels.cpu().numpy() == z["predict_label"]))
    print("hard scene, raw entry point: label agreement = %.5f" % agree)
    assert agree >= 0.999
    assert rel(logits.cpu().numpy()[z["band"]], z["logits_band"]) < 1e-3
    # the device fit reproduces the stored parameters: subspace, scales and the sign of every component
    fit = preprocess.fit(raw, 60)
    assert rel(fit.mu, h["pp"]["mu"]) < 1e-9 and rel(fit.sigma, h["pp"]["sigma"]) < 1e-9
    cos = np.sum(fit.U * h["pp"]["U"], 0)
    assert np.all(cos > 0) and rel(cos, np.ones(60)) < 1e-6
    assert rel(fit.pca_sigma, h["pp"]["pca_sigma"]) < 1e-8


def test_fp16_operand_range(dev, hard):
    """Activations driven toward fp16's range limit: conv0 scaled by 100 (a0 ~ 1e3, conv sums ~ 1e3..1e4, still far
    below 65504) must keep the 1e-3 logit bar and the labels; a scale that would overflow fp16 is reported as
    non-finite logits instead of silently wrong labels."""
    from cmlpl_b200.tools import hyper_tools as H
    h = hard
    rows = (60, 66)
    C = h["C"]
    sl = slice(rows[0] * C, rows[1] * C)
    cube_d = torch.from_numpy(h["Xp"]).to(dev)
    spec_band = torch.from_numpy(h["Xs"][sl]).to(dev)
    for scale, finite in ((100.0, True), (3.0e4, False)):
        sd = {k: v.clone() for k, v in h["sd"].items()}
        sd["conv0.weight"] *= scale; sd["conv0.bias"] *= scale
        net = make_net(dict(h, sd=sd), dev)
        lab, logits = H.scene_labels(net, cube_d, spec_band, 20, band=rows, want_logits=True)
        lg = logits.cpu().numpy()
        if not finite:
            assert not np.isfinite(lg).all()
            continue
        lab_ref, log_ref = O.test_whole(sd, h["Xp"], h["Xs"], 20, rows=rows, return_logits=True)
        assert np.isfinite(lg).all() and rel(lg, log_ref) < 1e-3
        assert float(np.mean(lab.cpu().numpy() == lab_ref)) >= 0.999


def test_paviau_size_row_band_with_the_trained_net(dev, hard):
    """VERDICT r1 item 3b: a scene of the headline size (610 x 340 x 103: the hard scene tiled 5 x 3 and cropped, so the
    spectra stay in the distribution of the net the reference trained and the tile seams add new neighbourhoods; stored
    preprocessing) inferred in ONE call; a 60-row band of it (20 400 pixels, across a seam) through the CPU oracle's
    test_whole (hyper_tools.py:416-437 per pixel).  >= 99.9 % identical labels, logits 1e-3 * max|ref|, both for the
    preprocessed entry point and for the raw-cube one."""
    from cmlpl_b200 import ops, preprocess
    h, z = hard, hard["z"]
    R, C, B, K, w = 610, 340, h["B"], h["K"], 20
    cube = np.ascontiguousarray(np.tile(h["cube"], (5, 3, 1))[:R, :C])
    Xp, Xs = O.apply_preprocess(cube, h["pp"])
    Xp, Xs = Xp.astype(np.float32), Xs.astype(np.float32)
    net = make_net(h, dev)
    packed = net.packed_weights(w)
    r0, r1 = 275, 335                                              # 60 rows x 340 columns = 20 400 pixels
    lab_ref, log_ref = O.test_whole(h["sd"], Xp, Xs, w, rows=(r0, r1), return_logits=True)
    lab, logits = ops.scene_infer(torch.from_numpy(Xp).to(dev), torch.from_numpy(Xs).to(dev), packed, K, w, want_logits=True)
    sl = slice(r0 * C, r1 * C)
    agree = float(np.mean(lab.cpu().numpy()[sl] == lab_ref))
    print("PaviaU-size band: label agreement %.5f over %d pixels" % (agree, (r1 - r0) * C))
    assert len(np.unique(lab_ref)) >= 6                            # the band is not a one-class region
    assert (r1 - r0) * C >= 20000 and agree >= 0.999
    assert rel(logits.cpu().numpy()[sl], log_ref) < 1e-3
    tol = 2e-3 * np.abs(log_ref).max()                             # only near-ties of the reference may flip
    for i in np.nonzero(lab.cpu().numpy()[sl] != lab_ref)[0]:
        assert log_ref[i].max() - log_ref[i, lab.cpu().numpy()[sl][i]] < tol
    # the raw-cube entry point on the same scene (preprocessing folded into the first kernels)
    pp = preprocess.Preproc(mu=h["pp"]["mu"], sigma=h["pp"]["sigma"], U=h["pp"]["U"], pca_mu=h["pp"]["pca_mu"],
                            pca_sigma=h["pp"]["pca_sigma"])
    folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    raw = torch.from_numpy(np.ascontiguousarray(cube.reshape(R * C, B))).to(dev)
    lab_raw, log_raw = ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True)
    agree_raw = float(np.mean(lab_raw.cpu().numpy()[sl] == lab_ref))
    print("PaviaU-size band, raw entry point: label agreement %.5f" % agree_raw)
    assert agree_raw >= 0.999
    assert rel(log_raw.cpu().numpy()[sl], log_ref) < 1e-3
