"""CPU suite: the oracle against the committed golden vectors (which were produced by the
unmodified reference, oracle/make_golden.py), host logic, and the C-ABI surface."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import cmlpl_oracle as O
from oracle import golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _g(golden_dir, name):
    return golden.load(os.path.join(golden_dir, name))


def test_patches_match_reference_golden(golden_dir):
    z = _g(golden_dir, "patches.npz")
    X = z["X"]
    for w in (4, 6, 10):
        assert np.array_equal(O.extract_patches(X, w), z[f"even_w{w}"])
        assert np.array_equal(O.extract_patches_loop(X, w), z[f"even_w{w}"])
    for w in (3, 5, 11):
        assert np.array_equal(O.extract_patches_for_base(X, w), z[f"odd_w{w}"])
    for hw in (1, 3, 5):
        assert np.array_equal(O.mirrow_cut(X, hw), z[f"mirror_hw{hw}"])
    with pytest.raises(ValueError):
        O.extract_patches(X, 5)           # the reference raises for odd w (hyper_tools.py:240)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_band_sharding_reproduces_full_gather(golden_dir, world):
    z = _g(golden_dir, "patches.npz")
    X = z["X"]
    R, C = X.shape[:2]
    for w, odd, key in ((6, False, "even_w6"), (5, True, "odd_w5")):
        got = []
        for rank in range(world):
            r0, r1, s0, s1 = O.band_rows(R, world, rank, w, odd)
            if r1 > r0:
                got.append(O.extract_patches_at(X[s0:s1], w, np.arange(r0 * C, r1 * C), odd, scene_rows=R, row0=s0))
        assert np.array_equal(np.concatenate(got), z[key])


def test_basenet2_matches_reference_golden(golden_dir):
    z = _g(golden_dir, "basenet2.npz")
    sd = {k[3:]: torch.from_numpy(z[k]).requires_grad_(True) for k in z if k.startswith("sd.")}
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    lo, fe = O.basenet2_forward(sd, x, y)
    assert np.abs(lo.detach().numpy() - z["logits"]).max() <= 1e-5 * np.abs(z["logits"]).max()
    assert np.abs(fe.detach().numpy() - z["feat"]).max() <= 1e-5
    loss = torch.nn.functional.cross_entropy(lo, torch.arange(6) % 16) + fe.pow(3).sum() * 0.1
    loss.backward()
    assert abs(float(loss) - float(z["loss"])) < 1e-5
    for k in O.LIVE_KEYS:
        g = z[f"grad.{k}"]
        assert np.abs(sd[k].grad.numpy() - g).max() <= 1e-4 * np.abs(g).max() + 1e-7, k


def test_init_order_matches_reference(golden_dir):
    z = _g(golden_dir, "basenet2.npz")
    torch.manual_seed(1088)
    O.basenet2_init(103, 9)                      # first net of the golden script ("paviau")
    torch.manual_seed(1088)
    sd = O.basenet2_init(32, 16)
    for k in O.LIVE_KEYS:
        assert np.array_equal(sd[k].numpy(), z[f"sd.{k}"]), k


def test_metrics_and_losses_match_reference_golden(golden_dir):
    z = _g(golden_dir, "metrics_losses.npz")
    OA, kappa, pa = O.cal_accuracy(z["pred"], z["label"])
    assert OA == z["OA"] and kappa == z["kappa"] and np.array_equal(pa, z["pa"])
    cm = O.confusion_matrix(z["pred"], z["label"], 9)
    assert np.array_equal(cm, z["cm"])
    o2 = O.accuracy_from_confusion(cm)
    assert o2[0] == z["OA"] and o2[1] == z["kappa"] and np.array_equal(o2[2], z["pa"])
    l = O.nt_xent(torch.from_numpy(z["ntx_i"]), torch.from_numpy(z["ntx_j"]), 0.5)
    assert abs(float(l) - float(z["ntx_loss"])) < 1e-5
    tgt = torch.from_numpy(z["us_target"]).clone()
    l = O.compute_unsupervised_loss(torch.from_numpy(z["us_predict"]), tgt, 80, torch.from_numpy(z["us_teacher"]))
    assert abs(float(l) - float(z["us_loss"])) < 1e-5
    assert np.array_equal(tgt.numpy(), z["us_target_after"])


def test_trained_inference_matches_reference_golden(golden_dir):
    """test_whole + CalAccuracy on the nets the reference's train.main produced."""
    z = _g(golden_dir, "train_infer.npz")
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z if k.startswith("sd.")}
    rows = (10, 14)                                # a band keeps the CPU suite fast
    C = 36
    lab, logits = O.test_whole(sd, z["cube_pca"], z["spectra"], 20, rows=rows, return_logits=True)
    sl = slice(rows[0] * C, rows[1] * C)
    assert np.array_equal(lab, z["predict_label"][sl].astype(np.int64))
    assert np.abs(logits - z["logits_trained"][sl]).max() <= 1e-4 * np.abs(z["logits_trained"]).max()
    te = z["test_array"]
    OA, kappa, pa = O.cal_accuracy(z["predict_label"].astype(np.int64)[te], (z["Y"].astype(np.int64) - 1)[te])
    assert abs(OA - float(z["OA"])) < 1e-12 and abs(kappa - float(z["Kappa"])) < 1e-12
    s = O.make_splits(z["Y"], 5)
    assert np.array_equal(s[0], z["train_array"]) and np.array_equal(s[1], te)
    assert np.array_equal(s[2], z["unlabel_array"])


def test_step_fixture_replays(golden_dir):
    """ref_step (pinned bit-exactly against train.main by make_golden.py) reproduces its fixture."""
    z = _g(golden_dir, "step.npz")
    ti = _g(golden_dir, "train_infer.npz")
    r, st = replay_step(z, ti)
    assert np.abs(r["hist"] - z["hist"]).max() < 1e-4
    assert np.abs(r["logits"].numpy() - z["logits"]).max() <= 1e-4 * np.abs(z["logits"]).max()
    for k in ("conv1.weight", "classifier.weight", "feat_spe.bias"):
        g = z[f"grad.{k}"]
        assert np.abs(r["grads"][k].numpy() - g).max() <= 1e-3 * np.abs(g).max() + 1e-8, k


def replay_step(z, ti):
    """Regenerate the inputs of tests/golden/step.npz (same recipe as make_golden.gold_step)."""
    Xp, Xs, Y = ti["cube_pca"], ti["spectra"], ti["Y"].astype(np.int64) - 1
    K, B = 9, 103
    torch.manual_seed(2024)
    sd, sd1 = O.basenet2_init(B, K), O.basenet2_init(B, K)
    sa = O.StepArgs(num_epochs=20)
    st = O.make_state(sd, sd1, K, sa)
    g = torch.Generator().manual_seed(99)
    li = ti["train_array"][torch.randint(0, len(ti["train_array"]), (128,), generator=g).numpy()]
    ui = ti["unlabel_array"][torch.randint(0, len(ti["unlabel_array"]), (128,), generator=g).numpy()]
    assert np.array_equal(li, z["li"]) and np.array_equal(ui, z["ui"])
    st.queue_feats.copy_(O.normalize(torch.randn(1280, 1024, generator=g).abs()))
    st.queue_probs.copy_(torch.softmax(torch.randn(1280, K, generator=g) * 2, 1))
    st.queue_feats1.copy_(O.normalize(torch.randn(1280, 1024, generator=g).abs()))
    st.queue_probs1.copy_(torch.softmax(torch.randn(1280, K, generator=g) * 2, 1))
    XP_l = torch.from_numpy(O.extract_patches_at(Xp, 20, li)); X_l = torch.from_numpy(Xs[li])
    XP_u = torch.from_numpy(O.extract_patches_at(Xp, 20, ui)); X_u = torch.from_numpy(Xs[ui])
    Y_l = torch.from_numpy(Y[li])
    nz = {k: torch.randn(s, generator=g) for k, s in (
        ("xp_l1", XP_l.shape), ("x_l1", X_l.shape), ("xp_l2", XP_l.shape), ("x_l2", X_l.shape),
        ("xp_u1", XP_u.shape), ("x_u1", X_u.shape), ("xp_u2", XP_u.shape), ("x_u2", X_u.shape))}
    sa.thr = 0.1445
    inputs = dict(XP_l=XP_l, X_l=X_l, Y_l=Y_l, XP_u=XP_u, X_u=X_u, noise=nz, args=sa, sd=sd, sd1=sd1)
    inputs["queues"] = [q.clone() for q in (st.queue_feats, st.queue_probs, st.queue_feats1, st.queue_probs1)]
    st.extras["inputs"] = inputs
    r = O.ref_step(st, XP_l, X_l, Y_l, XP_u, X_u, nz, epoch=1, batch_index=0, args=sa)
    return r, st


# ---------------------------------------------------------------- C-ABI surface (no GPU needed)
def _header_symbols():
    src = open(os.path.join(ROOT, "include", "cmlpl.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(cmlpl_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from cmlpl_b200 import _lib

    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/cmlpl.h but not exported"
    assert set(syms) == set(_lib.SIGNATURES), set(syms) ^ set(_lib.SIGNATURES)
    assert lib.cmlpl_version() >= 100
    assert lib.cmlpl_packed_bytes(103, 9, 20) > 2 * 73728
    assert lib.cmlpl_scene_workspace_bytes(10, 10, 103, 9, 20) > 0


def test_no_product_import_of_oracle():
    """The product package must never import the oracle (or torch CPU fallbacks through it)."""
    pkg = os.path.join(ROOT, "cmlpl_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.replace("the oracle", ""), f"{f} mentions oracle"


def test_product_fails_loudly_without_gpu():
    from cmlpl_b200 import _lib

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.CmlplError):
        _lib.require_device()
    from cmlpl_b200.tools import hyper_tools as H
    with pytest.raises(_lib.CmlplError):
        H.ExtractPatches(np.zeros((8, 8, 4)), 4)
