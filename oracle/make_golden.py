"""Pin the oracle against the UNMODIFIED reference and write tests/golden/*.npz.

Run in the build container only (needs /root/reference):
    python oracle/make_golden.py
Every fixture holds the inputs (or the seeds that regenerate them) and the outputs the
*reference's own code* produced; the script also asserts the oracle restatement agrees
with the reference before anything is written.  TEST INFRASTRUCTURE ONLY.
"""
import argparse
import os
import sys
import tempfile

import numpy as np
import scipy.io as sio
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shims  # noqa: E402

ref_shims.install()
from oracle import cmlpl_oracle as O  # noqa: E402
from oracle import golden  # noqa: E402

from tools import hyper_tools as RH  # noqa: E402  (reference)
from tools import models as RM  # noqa: E402  (reference)
import hsi_loader as RL  # noqa: E402  (reference)
import loss_helper as RLH  # noqa: E402  (reference)

GOLD = os.path.join(ROOT, "tests", "golden")


def close(a, b, rtol, what):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    err = np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)
    assert err <= rtol, f"{what}: rel err {err:.3e} > {rtol}"
    return err


def gold_patches():
    rng = np.random.default_rng(1088)
    X = rng.standard_normal((13, 11, 6))            # float64 like X_PCA
    out = {"X": X}
    for w in (4, 6, 10):                             # even: ExtractPatches (hw <= min dim)
        ref = RH.ExtractPatches(X, w)
        assert ref.dtype == np.float32
        assert np.array_equal(ref, O.extract_patches(X, w))
        assert np.array_equal(ref, O.extract_patches_loop(X, w))
        out[f"even_w{w}"] = np.ascontiguousarray(ref)
    for w in (3, 5, 11):                             # odd: ExtractPatches_for_base
        ref = RH.ExtractPatches_for_base(X, w)
        assert np.array_equal(ref, O.extract_patches_for_base(X, w))
        assert np.array_equal(ref, O.extract_patches_loop(X, w, odd_mode=True))
        out[f"odd_w{w}"] = np.ascontiguousarray(ref)
    for hw in (1, 3, 5):
        m = RH.MirrowCut(X, hw)
        assert np.array_equal(m, O.mirrow_cut(X, hw))
        out[f"mirror_hw{hw}"] = m
    # odd w through the even entry point raises in the reference
    try:
        RH.ExtractPatches(X, 5)
        raise AssertionError("reference accepted odd w")
    except ValueError:
        pass
    # band sharding reproduces the full gather (SURVEY 8e)
    full = RH.ExtractPatches(X, 6)
    for world in (2, 3, 4):
        got = []
        for rank in range(world):
            r0, r1, s0, s1 = O.band_rows(13, world, rank, 6)
            idx = np.arange(r0 * 11, r1 * 11)
            got.append(O.extract_patches_at(X[s0:s1], 6, idx, scene_rows=13, row0=s0))
        assert np.array_equal(np.concatenate(got), full)
    np.savez_compressed(os.path.join(GOLD, "patches.npz"), **out)
    print("patches.npz ok")


def gold_basenet2():
    out = {}
    for tag, (B, C) in {"paviau": (103, 9), "small": (32, 16)}.items():
        torch.manual_seed(1088)
        net = RM.BaseNet2(num_features=B, dropout=0, num_classes=C)
        torch.manual_seed(1088)
        sd = O.basenet2_init(B, C)
        rsd = net.state_dict()
        assert list(rsd.keys()) == list(sd.keys()) or set(rsd.keys()) == set(sd.keys())
        for k in rsd:
            assert torch.equal(rsd[k], sd[k]), f"init mismatch {k}"
        g = torch.Generator().manual_seed(7)
        x = torch.randn(6, 60, 20, 20, generator=g)
        y = torch.randn(6, B, generator=g)
        net.eval()
        with torch.no_grad():
            lo, fe = net(x, y)
            lo2, fe2 = O.basenet2_forward(sd, x, y)
        close(lo2, lo, 1e-6, "logits")
        close(fe2, fe, 1e-6, "feat")
        if tag == "small":
            for k, v in rsd.items():
                if k in O.LIVE_KEYS:
                    out[f"sd.{k}"] = v.numpy()
            out["x"], out["y"] = x.numpy(), y.numpy()
            out["logits"], out["feat"] = lo.numpy(), fe.numpy()
            # gradients of a scalar through the reference module
            net.train()
            net.zero_grad()
            lo, fe = net(x, y)
            tgt = torch.arange(6) % C
            loss = torch.nn.functional.cross_entropy(lo, tgt) + fe.pow(3).sum() * 0.1
            loss.backward()
            out["loss"] = loss.detach().numpy()
            for k, p in net.named_parameters():
                if k in O.LIVE_KEYS:
                    out[f"grad.{k}"] = p.grad.numpy()
    golden.save(os.path.join(GOLD, "basenet2.npz"), out)
    print("basenet2.npz ok")


def gold_metrics_losses():
    rng = np.random.default_rng(3)
    label = rng.integers(0, 9, size=5000)
    pred = np.where(rng.random(5000) < 0.8, label, rng.integers(0, 9, size=5000))
    OA, kappa, pa = RH.CalAccuracy(pred, label)
    o = O.cal_accuracy(pred, label)
    assert OA == o[0] and kappa == o[1] and np.array_equal(pa, o[2])
    cm = O.confusion_matrix(pred, label, 9)
    o2 = O.accuracy_from_confusion(cm)
    assert OA == o2[0] and kappa == o2[1] and np.array_equal(pa, o2[2])
    out = {"label": label, "pred": pred, "OA": OA, "kappa": kappa, "pa": pa, "cm": cm}

    g = torch.Generator().manual_seed(11)
    ei, ej = torch.randn(24, 40, generator=g), torch.randn(24, 40, generator=g)
    ref = RM.ContrastiveLoss(24, device="cpu", temperature=0.5)(ei, ej)
    close(O.nt_xent(ei, ej, 0.5), ref, 1e-6, "nt_xent")
    out.update(ntx_i=ei.numpy(), ntx_j=ej.numpy(), ntx_loss=ref.numpy())

    predict = torch.randn(200, 16, generator=g)
    teacher = torch.randn(200, 16, generator=g) * 3
    target = torch.randint(0, 16, (200,), generator=g)
    target[::13] = 255
    t_ref, t_or = target.clone(), target.clone()
    l_ref = RLH.compute_unsupervised_loss(predict, t_ref, 80, teacher)
    l_or = O.compute_unsupervised_loss(predict, t_or, 80, teacher)
    close(l_or, l_ref, 1e-6, "unsup")
    assert torch.equal(t_ref, t_or)
    out.update(us_predict=predict.numpy(), us_teacher=teacher.numpy(), us_target=target.numpy(),
               us_target_after=t_ref.numpy(), us_loss=l_ref.numpy())
    np.savez_compressed(os.path.join(GOLD, "metrics_losses.npz"), **out)
    print("metrics_losses.npz ok")


def gold_train(num_epochs=2, num_unlabel=512):
    """Run the unmodified sample_generation.main + train.main on a tiny PaviaU-keyed
    scene and check the oracle's ref_step / test_whole against what they produced."""
    R, C, B, K = 40, 36, 103, 9
    cube, gt = O.synth_cube(R, C, B, K, seed=1088)
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp(prefix="cmlpl_gold_")
    os.makedirs(os.path.join(tmp, "dataset"))
    sio.savemat(os.path.join(tmp, "dataset", "PaviaU.mat"), {"paviaU": cube})
    sio.savemat(os.path.join(tmp, "dataset", "PaviaU_gt.mat"), {"paviaU_gt": gt})
    os.chdir(tmp)
    try:
        import sample_generation as RS  # reference
        RS.main(argparse.Namespace(dataID=1, num_label=5, w=20, n_PC=60))
        d = os.path.join(tmp, "dataset", "PaviaU")
        XP = np.load(os.path.join(d, "XP.npy"))
        X = np.load(os.path.join(d, "X.npy"))
        Y = np.load(os.path.join(d, "Y.npy"))
        tr = np.load(os.path.join(d, "train_array.npy"))
        te = np.load(os.path.join(d, "test_array.npy"))
        un = np.load(os.path.join(d, "unlabel_array.npy"))
        # oracle preprocessing + splits reproduce the files
        Xp, Xs = O.preprocess(cube, 60)
        assert np.array_equal(Xs, X)
        assert np.array_equal(O.extract_patches(Xp, 20), XP)
        s = O.make_splits(Y, 5)
        assert np.array_equal(s[0], tr) and np.array_equal(s[1], te) and np.array_equal(s[2], un)

        import train as RT  # reference (seed_torch() runs at import, train.py:58)
        RT.DrawResult = lambda *a, **k: np.zeros((2, 2, 3))
        ns = argparse.Namespace(
            dataID=1, num_label=5, save_path_prefix="./", labeled_batch_size=128,
            unlabeled_batch_size=128, val_batch_size=512, num_workers=0, lr=5e-4,
            num_epochs=num_epochs, print_per_batches=2, num_unlabel=num_unlabel, thr=1,
            alpha=0.95, queue_batch=17, temperature=0.3, teacher_alpha=0.95, dropout=0.8,
            noise=0.5, m=5)
        RT.seed_torch()
        _, loc = ref_shims.capture_locals(
            RT.main, ns, names=("loss_hist", "Base", "Base1", "predict_label", "predict_label1",
                                "OA", "Kappa", "producerA", "queue_feats", "queue_probs1"))
        ref_hist = loc["loss_hist"].copy()

        # ---- replay with the oracle restatement, drawing RNG in the reference's order
        RT.seed_torch()
        from torch.utils import data
        lab = data.DataLoader(RL.HSIDataSet(1, setindex="label", max_iters=num_unlabel),
                              batch_size=128, shuffle=True, num_workers=0, worker_init_fn=RT.seed_worker)
        unl = data.DataLoader(RL.HSIDataSet(1, setindex="unlabel", max_iters=num_unlabel, num_unlabel=num_unlabel),
                              batch_size=128, shuffle=True, num_workers=0, worker_init_fn=RT.seed_worker)
        sd = O.basenet2_init(B, K)
        sd1 = O.basenet2_init(B, K)
        sa = O.StepArgs(num_epochs=num_epochs)
        st = O.make_state(sd, sd1, K, sa)
        p = 0.8
        hist = []
        first = None
        for epoch in range(num_epochs):
            for bi, ((XP_l, X_l, Y_l), (XP_u, X_u, _)) in enumerate(zip(lab, unl)):
                nz = {}
                nz["xp_l1"] = torch.randn(XP_l.size()); nz["x_l1"] = torch.randn(X_l.size())
                nz["xp_l2"] = torch.randn(XP_l.size()); nz["x_l2"] = torch.randn(X_l.size())
                nz["xp_u1"] = torch.randn(XP_u.size()); nz["x_u1"] = torch.randn(X_u.size())
                m0 = torch.nn.functional.dropout(torch.ones(256, 2624), p, True)
                nz["xp_u2"] = torch.randn(XP_u.size()); nz["x_u2"] = torch.randn(X_u.size())
                m1 = torch.nn.functional.dropout(torch.ones(256, 2624), p, True)
                r = O.ref_step(st, XP_l, X_l, Y_l, XP_u, X_u, nz, epoch, bi, sa, (m0, m1))
                hist.append(r["hist"])
        hist = np.array(hist)
        err = np.abs(hist - ref_hist).max()
        print("train replay: max |loss_hist diff| =", err)
        assert err < 2e-4, (hist, ref_hist)
        for k, v in loc["Base"].state_dict().items():
            close(st.sd[k].detach(), v, 2e-4, f"final weight {k}")
        # inference + metrics on the trained nets
        fsd = {k: v.detach() for k, v in st.sd.items()}
        pl = O.test_whole(fsd, Xp, Xs, 20)
        agree = np.mean(pl == loc["predict_label"])
        print("test_whole agreement oracle vs reference:", agree)
        assert agree >= 0.999
        OA, kappa, pa = O.cal_accuracy(loc["predict_label"][te], (Y.astype(np.int64) - 1)[te])
        # train.py:324 rebinds OA to mean(oa)*100 before main returns
        assert abs(OA * 100 - loc["OA"]) < 1e-9 and abs(kappa - loc["Kappa"]) < 1e-12
        ref_sd = {k: v.detach().numpy() for k, v in loc["Base"].state_dict().items() if k in O.LIVE_KEYS}
        lab_ref, logit_ref = O.test_whole({k: torch.from_numpy(v) for k, v in ref_sd.items()},
                                          Xp, Xs, 20, return_logits=True)
        assert np.mean(lab_ref == loc["predict_label"]) >= 0.9995
        golden.save(
            os.path.join(GOLD, "train_infer.npz"),
            dict(cube_pca=Xp.astype(np.float32), spectra=Xs.astype(np.float32), Y=Y, train_array=tr,
                 test_array=te, unlabel_array=un, loss_hist=ref_hist,
                 predict_label=loc["predict_label"].astype(np.uint8),
                 logits_trained=logit_ref.astype(np.float32),
                 OA=loc["OA"] / 100.0, Kappa=loc["Kappa"], producerA=loc["producerA"],
                 **{f"sd.{k}": v for k, v in ref_sd.items()}))
        print("train_infer.npz ok  (OA=%.4f kappa=%.4f)" % (loc["OA"] / 100.0, loc["Kappa"]))
    finally:
        os.chdir(cwd)


def gold_hard(R=150, C=140, spread=50.0, sigma=200.0, num_epochs=3, num_unlabel=2048, write=True):
    """A >= 20 k-pixel scene that the reference does NOT classify perfectly (VERDICT r1 item 3a): run the unmodified
    sample_generation.main + train.main on it and keep the trained weights, the reference's label map and the
    preprocessing parameters.  The scene itself is regenerated from its seed by the tests."""
    B, K = 103, 9
    cube, gt = O.synth_cube_hard(R, C, B, K, seed=1088, spread=spread, sigma=sigma)
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp(prefix="cmlpl_gold_hard_")
    os.makedirs(os.path.join(tmp, "dataset"))
    sio.savemat(os.path.join(tmp, "dataset", "PaviaU.mat"), {"paviaU": cube})
    sio.savemat(os.path.join(tmp, "dataset", "PaviaU_gt.mat"), {"paviaU_gt": gt})
    os.chdir(tmp)
    try:
        import sample_generation as RS
        RS.main(argparse.Namespace(dataID=1, num_label=5, w=20, n_PC=60))
        d = os.path.join(tmp, "dataset", "PaviaU")
        X = np.load(os.path.join(d, "X.npy"))
        Y = np.load(os.path.join(d, "Y.npy"))
        te = np.load(os.path.join(d, "test_array.npy"))
        pp = O.preprocess_params(cube, 60)
        Xp, Xs = O.apply_preprocess(cube, pp)
        close(Xs, X, 1e-12, "explicit z-score vs the reference's X.npy")
        XPr = np.load(os.path.join(d, "XP.npy"), mmap_mode="r")
        idx = np.array([0, 77, C * 40 + 3, R * C - 1])
        close(O.extract_patches_at(Xp, 20, idx), np.asarray(XPr[idx]), 1e-5, "explicit PCA cube vs the reference's XP.npy")
        import train as RT
        RT.DrawResult = lambda *a, **k: np.zeros((2, 2, 3))
        ns = argparse.Namespace(
            dataID=1, num_label=5, save_path_prefix="./", labeled_batch_size=128, unlabeled_batch_size=128,
            val_batch_size=512, num_workers=0, lr=5e-4, num_epochs=num_epochs, print_per_batches=4,
            num_unlabel=num_unlabel, thr=1, alpha=0.95, queue_batch=17, temperature=0.3, teacher_alpha=0.95,
            dropout=0.8, noise=0.5, m=5)
        RT.seed_torch()
        _, loc = ref_shims.capture_locals(RT.main, ns, names=("Base", "predict_label", "OA", "Kappa", "producerA"))
        ref_sd = {k: v.detach().numpy() for k, v in loc["Base"].state_dict().items() if k in O.LIVE_KEYS}
        OA, kappa, pa = O.cal_accuracy(loc["predict_label"][te], (Y.astype(np.int64) - 1)[te])
        print("hard scene: reference OA = %.4f kappa = %.4f" % (OA, kappa))
        fsd = {k: torch.from_numpy(v) for k, v in ref_sd.items()}
        band = np.arange(60 * C, 64 * C)                       # a row band for the fixture's logits
        lab, logit = O.test_whole(fsd, Xp, Xs, 20, return_logits=True)
        agree = float(np.mean(lab == loc["predict_label"]))
        print("oracle test_whole vs reference on the hard scene:", agree)
        assert agree >= 0.999
        if write:
            np.savez_compressed(
                os.path.join(GOLD, "hard_scene.npz"),
                shape=np.array([R, C, B, K]), spread=spread, sigma=sigma, seed=1088,
                mu=pp["mu"], sigma_x=pp["sigma"], U=pp["U"], pca_mu=pp["pca_mu"], pca_sigma=pp["pca_sigma"],
                predict_label=loc["predict_label"].astype(np.uint8), OA=OA, Kappa=kappa, producerA=pa,
                test_array=te, Y=Y, band=band, logits_band=logit[band].astype(np.float32),
                cube_checksum=np.array([int(cube.astype(np.int64).sum()), int((cube.astype(np.int64) ** 2).sum() % (1 << 61))]),
                **{f"sd.{k}": v for k, v in ref_sd.items()})
            print("hard_scene.npz ok")
        return OA
    finally:
        os.chdir(cwd)


def gold_loader():
    """hsi_loader.HSIDataSet of the reference on the files its own sample_generation.main wrote for the 40x36 scene:
    lengths, the tiled label / spectrum order of every split and full items (VERDICT r1 item 3c)."""
    R, C, B, K = 40, 36, 103, 9
    cube, gt = O.synth_cube(R, C, B, K, seed=1088)
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp(prefix="cmlpl_gold_loader_")
    os.makedirs(os.path.join(tmp, "dataset"))
    sio.savemat(os.path.join(tmp, "dataset", "PaviaU.mat"), {"paviaU": cube})
    sio.savemat(os.path.join(tmp, "dataset", "PaviaU_gt.mat"), {"paviaU_gt": gt})
    os.chdir(tmp)
    out = {}
    try:
        import sample_generation as RS
        RS.main(argparse.Namespace(dataID=1, num_label=5, w=20, n_PC=60))
        d = os.path.join(tmp, "dataset", "PaviaU")
        for f in ("train_array", "test_array", "unlabel_array", "Y"):
            out[f] = np.load(os.path.join(d, f + ".npy"))
        out["X"] = np.load(os.path.join(d, "X.npy"))                       # f64 [N, B], the file contract
        cases = {"label_tiled": dict(setindex="label", max_iters=137), "label_plain": dict(setindex="label"),
                 "unlabel_head": dict(setindex="unlabel", max_iters=300, num_unlabel=200),      # tiled to 300 rows
                 "unlabel_short": dict(setindex="unlabel", max_iters=96, num_unlabel=200),      # head of the split only
                 "unlabel_plain": dict(setindex="unlabel", num_unlabel=50),
                 "test": dict(setindex="test"), "wholeset": dict(setindex="wholeset")}
        for name, kw in cases.items():
            ds = RL.HSIDataSet(1, **kw)
            n = len(ds)
            out[f"{name}.len"] = np.array(n)
            picks = sorted({0, 1, n // 2, n - 1})
            out[f"{name}.picks"] = np.array(picks)
            # order of the whole split through cheap per-item signatures
            sig = np.array([ds[i][1][:4] for i in range(n)])
            out[f"{name}.spec_sig"] = sig
            if kw["setindex"] != "wholeset":
                out[f"{name}.labels"] = np.array([int(ds[i][2]) for i in range(n)])
            for j, i in enumerate(picks[:2]):
                item = ds[i]
                out[f"{name}.item{j}.xp"] = item[0]
                out[f"{name}.item{j}.x"] = item[1]
                assert item[0].dtype == np.float32 and item[1].dtype == np.float32
                if len(item) == 3:
                    assert item[2].dtype == np.int64 or item[2].dtype == int
            out[f"{name}.arity"] = np.array(len(ds[0]))
        golden.save(os.path.join(GOLD, "loader.npz"), out)
        print("loader.npz ok:", {k: int(v) for k, v in out.items() if k.endswith(".len")})
    finally:
        os.chdir(cwd)


def _reference_function(path, name):
    """Compile ONE function of a reference script that cannot be imported as a module (trian_CCT.py imports names the
    repository does not ship): its unmodified source text, executed in a namespace holding torch and F."""
    import ast
    import torch.nn.functional as F_
    src = open(path).read()
    node = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == name)
    ns = {"torch": torch, "F": F_}
    exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    return ns[name]


def gold_ablation():
    """f4: softmax_js_loss of trian_CCT.py:76-84 (the reference's own function object) and the CPS cross-supervision
    losses of trian_CPS.py:232-247 (restated inline: the script has no function boundary there)."""
    js = _reference_function(os.path.join(ref_shims.REFERENCE_ROOT, "trian_CCT.py"), "softmax_js_loss")
    g = torch.Generator().manual_seed(31)
    out = {}
    for tag, (n, C) in {"a": (37, 9), "b": (128, 16)}.items():
        z = (torch.randn(n, C, generator=g) * 2).requires_grad_(True)
        t = torch.softmax(torch.randn(n, C, generator=g) * 3, 1)
        if tag == "a":
            t[0] = 0.0; t[0, 3] = 1.0                      # exact zeros in the target (xlogy branch of F.kl_div)
        loss = js(z, t)
        loss.backward()
        out.update({f"js_{tag}_z": z.detach().numpy(), f"js_{tag}_t": t.numpy(), f"js_{tag}_loss": loss.detach().numpy(),
                    f"js_{tag}_grad": z.grad.numpy()})
    # CPS
    bs, n, C = 24, 56, 9
    ob = (torch.randn(n, C, generator=g)).requires_grad_(True); oe = (torch.randn(n, C, generator=g)).requires_grad_(True)
    Y = torch.randint(0, C, (bs,), generator=g)
    ce = torch.nn.CrossEntropyLoss()
    cls, cls1 = ce(ob[:bs], Y), ce(oe[:bs], Y)
    p1, p2 = torch.max(ob[bs:], 1)[1], torch.max(oe[bs:], 1)[1]
    con, con1 = ce(ob[bs:], p2.detach()).mean(), ce(oe[bs:], p1.detach()).mean()
    tot, tot1 = cls + 0.1 * con, cls1 + 0.1 * con1
    tot.backward(); tot1.backward()
    out.update(cps_ob=ob.detach().numpy(), cps_oe=oe.detach().numpy(), cps_Y=Y.numpy(), cps_total=tot.detach().numpy(),
               cps_total1=tot1.detach().numpy(), cps_con=con.detach().numpy(), cps_con1=con1.detach().numpy(),
               cps_gb=ob.grad.numpy(), cps_ge=oe.grad.numpy())
    np.savez_compressed(os.path.join(GOLD, "ablation.npz"), **out)
    print("ablation.npz ok")


def gold_step():
    """One full-size (128+128) mutual-learning step through the oracle, with every input
    regenerable from the fixture (cube + indices + seeds).  The oracle's ref_step was
    pinned against train.main by gold_train(); this fixture freezes its outputs."""
    z = golden.load(os.path.join(GOLD, "train_infer.npz"))
    Xp, Xs, Y = z["cube_pca"], z["spectra"], z["Y"].astype(np.int64) - 1
    tr, un = z["train_array"], z["unlabel_array"]
    K, B = 9, 103
    torch.manual_seed(2024)
    sd, sd1 = O.basenet2_init(B, K), O.basenet2_init(B, K)
    sa = O.StepArgs(num_epochs=20)
    st = O.make_state(sd, sd1, K, sa)
    g = torch.Generator().manual_seed(99)
    li = tr[torch.randint(0, len(tr), (128,), generator=g).numpy()]
    ui = un[torch.randint(0, len(un), (128,), generator=g).numpy()]
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
    sa.thr = 0.1445   # so that the mask is not all-zero and the soft-CE term is exercised
    r = O.ref_step(st, XP_l, X_l, Y_l, XP_u, X_u, nz, epoch=1, batch_index=0, args=sa)
    out = {"li": li, "ui": ui, "hist": r["hist"], "total1": r["total1"], "lc1": r["lc1"],
           "con1": r["con1"], "cls1": r["cls1"], "logits": r["logits"].numpy(),
           "logits1": r["logits1"].numpy(), "mask": r["mask"].numpy(), "masks": r["masks"].numpy(),
           "probs": r["probs"].numpy(), "probs1": r["probs1"].numpy()}
    for k in O.LIVE_KEYS:
        out[f"grad.{k}"] = r["grads"][k].numpy()
        out[f"grad1.{k}"] = r["grads1"][k].numpy()
        out[f"new.{k}"] = st.sd[k].detach().numpy()
    golden.save(os.path.join(GOLD, "step.npz"), out)
    print("step.npz ok, hist =", r["hist"])


def gold_loss_helper():
    """Outputs of the reference's loss_helper callables (loss_helper.py) on seeded inputs."""
    g = torch.Generator().manual_seed(21)
    out = {}
    # segmentation-style criteria on [b, 19, h, w]
    pred = torch.randn(2, 19, 12, 10, generator=g)
    aux = torch.randn(2, 19, 12, 10, generator=g)
    tgt = torch.randint(0, 19, (2, 12, 10), generator=g)
    tgt[0, :3] = 255
    out.update(seg_pred=pred.numpy(), seg_aux=aux.numpy(), seg_tgt=tgt.numpy())
    out["crit_plain"] = RLH.Criterion(0)(pred, tgt).numpy()
    out["crit_aux"] = RLH.Criterion(0.4)((pred, aux), tgt).numpy()
    out["crit_weight"] = RLH.Criterion(0.4, use_weight=True)((pred, aux), tgt).numpy()
    out["ohem_tensor"] = RLH.OhemCrossEntropy2dTensor(255, 0.7, 40)(pred, tgt.clone()).numpy()
    out["ohem_tensor_w"] = RLH.OhemCrossEntropy2dTensor(255, 0.05, 30, use_weight=True)(pred, tgt.clone()).numpy()
    out["crit_ohem"] = RLH.CriterionOhem(0.4, thresh=0.7, min_kept=50)((pred, aux), tgt.clone()).numpy()
    cfg = {"criterion": {"type": "ohem", "kwargs": {"thresh": 0.7, "min_kept": 50}}, "net": {"aux_loss": {"loss_weight": 0.4}},
           "dataset": {"ignore_label": 255}}
    out["get_criterion"] = RLH.get_criterion(cfg)((pred, aux), tgt.clone()).numpy()
    torch.Tensor.get_device = lambda self: "cpu"
    out["ohem_host"] = RLH.OhemCrossEntropy2d(255, 0.7, 160, factor=2)(pred, tgt.clone()).numpy()
    out["rce"] = RLH.compute_rce_loss(pred, tgt.clone()).numpy()
    # dequeue_and_enqueue
    q, ptr = [torch.zeros(0, 8)], torch.zeros(1, dtype=torch.long)
    hist = []
    for n in (5, 9, 4):
        keys = torch.randn(n, 8, generator=g)
        RLH.dequeue_and_enqueue(keys, q, ptr, 12)
        hist.append((q[0].clone().numpy(), int(ptr[0])))
    out["dq_final"] = hist[-1][0]; out["dq_ptrs"] = np.array([h[1] for h in hist]); out["dq_mid"] = hist[1][0]
    # compute_contra_memobank_loss: 6 classes, 24 labelled + 24 unlabelled, 32-d representations
    C, nl, nu, D = 6, 24, 24, 32
    rep = torch.randn(nl + nu, D, generator=g); rep_t = torch.randn(nl + nu, D, generator=g)
    yl = torch.randint(0, C, (nl,), generator=g); yu = torch.randint(0, C, (nu,), generator=g)
    label_l = torch.nn.functional.one_hot(yl, C).float(); label_u = torch.nn.functional.one_hot(yu, C).float()
    prob_l = torch.softmax(torch.randn(nl, C, generator=g) * 2, 1); prob_u = torch.softmax(torch.randn(nu, C, generator=g) * 2, 1)
    low_mask = (torch.rand(nl + nu, 1, generator=g) > 0.3).float(); high_mask = (torch.rand(nl + nu, 1, generator=g) > 0.3).float()
    def banks():
        gg = torch.Generator().manual_seed(5)
        return [[torch.randn(7, D, generator=gg)] for _ in range(C)], [torch.zeros(1, dtype=torch.long) for _ in range(C)]
    mb, ptrs = banks()
    torch.manual_seed(77)
    rr = rep.clone().requires_grad_(True)
    keys, loss = RLH.compute_contra_memobank_loss(rr, label_l, label_u, prob_l, prob_u, low_mask, high_mask, mb, ptrs,
                                                  [30] * C, rep_t)
    loss.backward()
    out.update(mb_rep=rep.numpy(), mb_rep_t=rep_t.numpy(), mb_label_l=label_l.numpy(), mb_label_u=label_u.numpy(),
               mb_prob_l=prob_l.numpy(), mb_prob_u=prob_u.numpy(), mb_low=low_mask.numpy(), mb_high=high_mask.numpy(),
               mb_loss=loss.detach().numpy(), mb_keys=np.array(keys), mb_grad=rr.grad.numpy(),
               mb_bank_sizes=np.array([b[0].shape[0] for b in mb]))
    mb, ptrs = banks()
    torch.manual_seed(78)
    proto, keys, loss = RLH.compute_contra_memobank_loss(rep, label_l, label_u, prob_l, prob_u, low_mask, high_mask, mb,
                                                         ptrs, [30] * C, rep_t, momentum_prototype=torch.ones(C, 256, 1, D) * 0.1, i_iter=5)
    out.update(mb_loss_mom=loss.numpy(), mb_proto_sum=proto.sum((1, 2, 3)).numpy())
    np.savez_compressed(os.path.join(GOLD, "loss_helper.npz"), **out)
    print("loss_helper.npz ok")


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
    which = sys.argv[1:] or ["patches", "basenet2", "metrics", "train", "step", "loss_helper", "ablation", "loader", "hard"]
    if "patches" in which:
        gold_patches()
    if "basenet2" in which:
        gold_basenet2()
    if "metrics" in which:
        gold_metrics_losses()
    if "train" in which:
        gold_train()
    if "step" in which:
        gold_step()
    if "loss_helper" in which:
        gold_loss_helper()
    if "ablation" in which:
        gold_ablation()
    if "loader" in which:
        gold_loader()
    if "hard" in which:
        gold_hard()
