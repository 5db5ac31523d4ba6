"""CPU restatement of the CMLPL hot path (oracle).  TEST INFRASTRUCTURE ONLY.

Parity status: the reference ships no tests / golden vectors (SURVEY.md section 4),
so this oracle is pinned by *executing the reference itself* in the build
container: ``oracle/make_golden.py`` imports ``/root/reference`` (three shims),
runs its functions on seeded synthetic inputs, checks every function below
against them and commits the outputs under ``tests/golden/``.  The CPU tests
re-check this file against those fixtures on every run.

All ``file:line`` citations are relative to ``/root/reference``.
Numerics: float64 where the reference uses numpy float64, torch CPU float32
where the reference uses torch (CPU fp32 is the exact ground truth; the
reference's GPU path under torch 1.8 would have used TF32).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np
import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------
# a1 / a2 / a3: mirror padding and per-pixel patch extraction
# --------------------------------------------------------------------------


def mirror_index(o: np.ndarray | int, n: int):
    """Map an unpadded coordinate ``o`` (may be <0 or >=n) to its source index.

    tools/hyper_tools.py:35-55 (MirrowCut) tiles flipped copies 3x3 and crops,
    which equals ``np.pad(..., mode='symmetric')``: o<0 -> -o-1, o>=n -> 2n-1-o.
    Valid for the single reflection the reference supports (hw <= n).
    """
    o = np.asarray(o)
    return np.where(o < 0, -o - 1, np.where(o >= n, 2 * n - 1 - o, o))


def mirrow_cut(X: np.ndarray, hw: int) -> np.ndarray:
    """tools/hyper_tools.py:35-55.  Output is float64 like the reference's zeros()."""
    return np.pad(np.asarray(X, dtype=np.float64), ((hw, hw), (hw, hw), (0, 0)), mode="symmetric")


def window_bounds(w: int, odd_mode: bool):
    """Offsets (lo, hi) such that the window of pixel r is rows r+lo .. r+hi-1.

    even (ExtractPatches, hyper_tools.py:227,239): hw=w//2, rows r-hw .. r+hw-1
    odd  (ExtractPatches_for_base, hyper_tools.py:301,313): hw=(w-1)//2, r-hw .. r+hw
    """
    if odd_mode:
        hw = (w - 1) // 2
        return -hw, hw + 1
    hw = w // 2
    return -hw, hw


def extract_patches_loop(X: np.ndarray, w: int, odd_mode: bool = False) -> np.ndarray:
    """The reference algorithm as written (per-pixel Python loop); this is the form
    that is *timed* as the CPU baseline.  hyper_tools.py:226-243 / :300-317."""
    hw = int((w - 1) / 2) if odd_mode else int(w / 2)
    row, col, nf = X.shape
    K = row * col
    Xm = mirrow_cut(X, hw)
    XP = np.zeros((K, w, w, nf), dtype=np.float32)
    ext = 1 if odd_mode else 0
    for i in range(1, K + 1):
        index_row = int(np.ceil(i * 1.0 / col))
        index_col = i - (index_row - 1) * col + hw - 1
        index_row += hw - 1
        XP[i - 1] = Xm[index_row - hw:index_row + hw + ext, index_col - hw:index_col + hw + ext, :]
    return np.ascontiguousarray(np.moveaxis(XP, 3, 1)).astype(np.float32)


def extract_patches_at(X: np.ndarray, w: int, idx: np.ndarray, odd_mode: bool = False,
                       scene_rows: int | None = None, row0: int = 0) -> np.ndarray:
    """Vectorised gather of the patches of raster indices ``idx`` -> f32 [n, F, w, w].

    Same values as ``extract_patches_loop(X, w)[idx]`` (the f64->f32 cast commutes
    with the gather).  ``X`` may be a row slab ``[row0, row0+X.shape[0])`` of a scene
    with ``scene_rows`` rows (band sharding, SURVEY section 8e): mirroring is applied
    at true scene edges only and every source row must lie inside the slab.
    """
    if not odd_mode and w % 2:
        raise ValueError("ExtractPatches (hyper_tools.py:226) only supports even w")
    if odd_mode and w % 2 == 0:
        raise ValueError("ExtractPatches_for_base (hyper_tools.py:300) only supports odd w")
    R = X.shape[0] if scene_rows is None else scene_rows
    C = X.shape[1]
    idx = np.asarray(idx, dtype=np.int64)
    lo, hi = window_bounds(w, odd_mode)
    r = idx // C
    c = idx % C
    rr = mirror_index(r[:, None] + np.arange(lo, hi)[None, :], R) - row0   # [n, w]
    cc = mirror_index(c[:, None] + np.arange(lo, hi)[None, :], C)          # [n, w]
    assert rr.min() >= 0 and rr.max() < X.shape[0], "slab does not cover the halo"
    Xf = np.asarray(X, dtype=np.float32)
    out = Xf[rr[:, :, None], cc[:, None, :], :]                             # [n, w, w, F]
    return np.ascontiguousarray(np.moveaxis(out, 3, 1))


def extract_patches(X: np.ndarray, w: int) -> np.ndarray:
    """hyper_tools.py:226-243, vectorised."""
    return extract_patches_at(X, w, np.arange(X.shape[0] * X.shape[1]), odd_mode=False)


def extract_patches_for_base(X: np.ndarray, w: int) -> np.ndarray:
    """hyper_tools.py:300-317, vectorised."""
    return extract_patches_at(X, w, np.arange(X.shape[0] * X.shape[1]), odd_mode=True)


def band_rows(R: int, world: int, rank: int, w: int, odd_mode: bool = False):
    """Row band of ``rank`` and the slab of cube rows (halo included) it must hold."""
    per = -(-R // world)
    r0 = min(rank * per, R)
    r1 = min(r0 + per, R)
    lo, hi = window_bounds(w, odd_mode)
    if r1 <= r0:
        return r0, r1, r0, r0
    rows = mirror_index(np.arange(r0 + lo, r1 - 1 + hi), R)
    return r0, r1, int(rows.min()), int(rows.max()) + 1


# --------------------------------------------------------------------------
# preprocessing shared by both sides (hyper_tools.py:8-32) and synthetic data
# --------------------------------------------------------------------------


def feature_normalize(X: np.ndarray, type: int = 1) -> np.ndarray:
    """hyper_tools.py:8-22."""
    if type == 1:
        Xn = X - np.mean(X, 0)
        return Xn / np.std(Xn, 0)
    mn, mx = np.min(X, 0), np.max(X, 0)
    return (X - mn) / (mx - mn)


def pca_norm(X: np.ndarray, num_PC: int) -> np.ndarray:
    """hyper_tools.py:25-32."""
    Xn = X - np.mean(X, 0)
    U, _, _ = np.linalg.svd(np.cov(Xn.T))
    return Xn @ U[:, :num_PC]


def synth_cube(R: int, C: int, B: int, K: int, seed: int = 1088, block: int = 8):
    """Synthetic scene of SURVEY section 8(d): blocky class map + noisy class prototypes."""
    rng = np.random.default_rng(seed)
    gb = rng.integers(0, K + 1, size=(-(-R // block), -(-C // block)))
    gt = np.kron(gb, np.ones((block, block), dtype=np.int64))[:R, :C]
    flat = gt.reshape(-1)
    # guarantee every class is populated: stamp class k on a few pixels
    for k in range(1, K + 1):
        if (flat == k).sum() < 32:
            flat[rng.choice(flat.size, 32, replace=False)] = k
    gt = flat.reshape(R, C)
    P = rng.uniform(0, 4000, size=(K + 1, B))
    cube = P[gt] + rng.normal(0, 200, size=(R, C, B))
    return np.clip(cube, 0, 8000).astype(np.uint16), gt.astype(np.uint8)


def synth_cube_hard(R: int, C: int, B: int, K: int, seed: int = 1088, spread: float = 50.0, sigma: float = 200.0,
                    block: int = 8):
    """A scene whose classes are NOT trivially separable (parity stress, VERDICT r1 item 3a): every class prototype
    is one common spectrum plus a small class offset (``spread`` DN per band) under the same sensor noise, so a
    net trained on 5 labels per class lands well below 100 % and many pixels sit near a decision boundary."""
    rng = np.random.default_rng(seed)
    gb = rng.integers(0, K + 1, size=(-(-R // block), -(-C // block)))
    gt = np.kron(gb, np.ones((block, block), dtype=np.int64))[:R, :C]
    base = rng.uniform(1000, 3000, size=(1, B))
    P = base + spread * rng.standard_normal((K + 1, B))
    cube = P[gt] + rng.normal(0, sigma, size=(R, C, B))
    return np.clip(cube, 0, 8000).astype(np.uint16), gt.astype(np.uint8)


def sensor_scene(R: int, C: int, B: int, K: int, noise_dn: float = 8.0, seed: int = 1088, sample: str = "u16",
                 dc: float = 0.0, block: int = 8):
    """A scene conditioned like a real sensor's (PaviaU, AVIRIS, WHU-Hi) rather than like ``synth_cube``: every pixel is a
    smooth mixture of K + 1 endmember spectra under a per-pixel illumination, plus ``noise_dn`` DN of sensor noise.  The
    signal spans K + 1 dimensions and the noise floor is a few DN, so lambda_1 / lambda_60 of the band covariance is 1e5 to
    1e8 (``synth_cube``: 1e3) and the trailing z-scored PCA components are small differences of large band values.

    * endmembers: an offset plus four Gaussians over the band index (widths 5-30 % of the band range), 200-8000 DN;
    * class map: blocky as in ``synth_cube``; abundances are the pixel's own class (weight 0.75-1) plus a share of the
      classes half a block away in each direction;
    * illumination: uniform in [0.7, 1.3] per pixel;
    * ``sample``: "u16" (rounded, + ``dc`` DN, e.g. a 20 000 DN offset that makes the band means large next to their
      standard deviations), "i16" (dark-subtracted: minus a dark level per band of about half the band's mean, so many
      values are negative) or "f32" (reflectance-like: DN / 10 000, noise ``noise_dn`` / 10 000, not rounded).
    -> (cube [R, C, B] of the sample type, gt uint8 [R, C] with 0 = unlabelled)."""
    rng = np.random.default_rng(seed)
    gb = rng.integers(0, K + 1, size=(-(-R // block), -(-C // block)))
    gt = np.kron(gb, np.ones((block, block), dtype=np.int64))[:R, :C]
    flat = gt.reshape(-1)
    for k in range(1, K + 1):
        if (flat == k).sum() < 32:
            flat[rng.choice(flat.size, 32, replace=False)] = k
    gt = flat.reshape(R, C)
    t = np.arange(B) / max(B - 1, 1)
    E = np.empty((K + 1, B))
    for k in range(K + 1):
        e = rng.uniform(200, 1200) + sum(rng.uniform(500, 2500) * np.exp(-0.5 * ((t - rng.uniform(-0.1, 1.1))
                                                                                  / rng.uniform(0.05, 0.3)) ** 2)
                                         for _ in range(4))
        E[k] = np.clip(e, 200, 8000)
    onehot = (gt[..., None] == np.arange(K + 1)).astype(np.float64)
    h = max(block // 2, 1)
    nb = sum(onehot[mirror_index(np.arange(R) + dr, R)][:, mirror_index(np.arange(C) + dc_, C)]
             for dr, dc_ in ((-h, 0), (h, 0), (0, -h), (0, h))) / 4.0
    own = rng.uniform(0.75, 1.0, size=(R, C, 1))
    A = own * onehot + (1 - own) * nb
    cube = rng.uniform(0.7, 1.3, size=(R, C, 1)) * (A @ E) + rng.normal(0, noise_dn, size=(R, C, B))
    if sample == "u16":
        cube = np.clip(np.rint(cube + dc), 0, 65535).astype(np.uint16)
    elif sample == "i16":
        dark = 0.5 * E.mean(0) * rng.uniform(0.8, 1.2, size=B)
        cube = np.clip(np.rint(cube - dark), -32768, 32767).astype(np.int16)
    elif sample == "f32":
        cube = (cube / 1e4).astype(np.float32)
    else:
        raise ValueError(f"sample must be u16, i16 or f32, got {sample!r}")
    return cube, gt.astype(np.uint8)


def preprocess_params(cube_u16: np.ndarray, n_PC: int = 60):
    """The affine maps behind hyper_tools.py:285-292 as explicit float64 parameters:
    spectra = (X - mu) / sigma;  cubePCA = ((X - mu) @ U - pca_mu) / pca_sigma."""
    R, C, B = cube_u16.shape
    X = cube_u16.reshape(R * C, B).astype(np.float64)
    mu = X.mean(0)
    Xc = X - mu
    sigma = Xc.std(0)
    U = np.linalg.svd(np.cov(Xc.T))[0][:, :n_PC]
    proj = Xc @ U
    return {"mu": mu, "sigma": sigma, "U": U, "pca_mu": proj.mean(0), "pca_sigma": (proj - proj.mean(0)).std(0)}


def apply_preprocess(cube_u16: np.ndarray, pp: dict):
    R, C, B = cube_u16.shape
    Xc = cube_u16.reshape(R * C, B).astype(np.float64) - pp["mu"]
    cube = ((Xc @ pp["U"]) - pp["pca_mu"]) / pp["pca_sigma"]
    return cube.reshape(R, C, -1), Xc / pp["sigma"]


def preprocess(cube_u16: np.ndarray, n_PC: int = 60):
    """hyper_tools.py:285-292: returns (cubePCA f64 [R,C,n_PC], spectra f64 [N,B])."""
    R, C, B = cube_u16.shape
    X = cube_u16.reshape(R * C, B)
    Xp = feature_normalize(pca_norm(X, n_PC), 1).reshape(R, C, n_PC)
    return Xp, feature_normalize(X, 1)


def make_splits(Y: np.ndarray, num_label: int):
    """sample_generation.py:43-65 (numpy legacy seeds 2 and 0)."""
    n_class = int(Y.max())
    np.random.seed(2)
    whole = np.where(Y > 0)[0]
    np.random.shuffle(whole)
    train, test = [], []
    for i in range(1, n_class + 1):
        index = np.where(Y == i)[0]
        np.random.seed(0)
        perm = np.random.permutation(index.shape[0])
        train.append(index[perm[:num_label]])
        test.append(index[perm[num_label:]])
    train = np.concatenate(train)
    test = np.concatenate(test)
    unlabel = np.array(list(set(whole) - set(train)))
    return train, test, unlabel


# --------------------------------------------------------------------------
# a5 / a6: BaseNet2 (tools/models.py:97-152) as pure functions of a state dict
# --------------------------------------------------------------------------

LIVE_KEYS = ("conv0.weight", "conv0.bias", "conv1.weight", "conv1.bias", "conv2.weight",
             "conv2.bias", "feat_spe.weight", "feat_spe.bias", "classifier.weight",
             "classifier.bias")


def _conv_init(out_c, in_c, k):
    w = torch.empty(out_c, in_c, k, k)
    torch.nn.init.kaiming_uniform_(w, a=math.sqrt(5))
    bound = 1 / math.sqrt(in_c * k * k)
    b = torch.empty(out_c).uniform_(-bound, bound)
    return w, b


def _lin_init(out_f, in_f):
    w = torch.empty(out_f, in_f)
    torch.nn.init.kaiming_uniform_(w, a=math.sqrt(5))
    bound = 1 / math.sqrt(in_f)
    b = torch.empty(out_f).uniform_(-bound, bound)
    return w, b


def basenet2_init(num_features: int, num_classes: int, conv_feat: int = 1600):
    """State dict with the key names / shapes / RNG order of models.py:98-128
    (default torch init; draws from the global torch CPU generator)."""
    sd = {}
    for name, (o, i, k) in (("conv0", (64, 60, 1)), ("conv1", (64, 64, 3)), ("conv2", (64, 64, 3))):
        sd[name + ".weight"], sd[name + ".bias"] = _conv_init(o, i, k)
    for name, (o, i) in (("feat_spe", (1024, num_features)), ("feat_ss", (256, 1024)),
                         ("feat_ss2", (64, 1024)), ("feat_ss3", (64, 256)),
                         ("classifier", (num_classes, conv_feat + 1024))):
        sd[name + ".weight"], sd[name + ".bias"] = _lin_init(o, i)
    return sd


def normalize(x: torch.Tensor) -> torch.Tensor:
    """models.py:87-90 (no epsilon)."""
    return x.div(x.pow(2).sum(1, keepdim=True).pow(0.5))


def basenet2_forward(sd, x, y, dropout_mask=None, return_parts: bool = False, relu_masks=None):
    """models.py:130-152.  ``dropout_mask`` (already scaled by 1/(1-p), or None) replaces
    nn.Dropout so the test harness can inject it.  ``relu_masks`` (the 0/1 masks of the two
    trunk ReLUs, [n,64,20,20] and [n,64,10,10], or None) replaces ReLU's own sign test, so that a
    reduced-precision forward's masks can be imposed on this one."""
    relu = lambda z, i: F.relu(z) if relu_masks is None else z * relu_masks[i]
    x = F.conv2d(x, sd["conv0.weight"], sd["conv0.bias"])
    x = relu(F.conv2d(x, sd["conv1.weight"], sd["conv1.bias"], padding=1) + x, 0)
    x = F.avg_pool2d(x, 2, 2)
    x = relu(F.conv2d(x, sd["conv2.weight"], sd["conv2.bias"], padding=1) + x, 1)
    x = F.avg_pool2d(x, 2, 2)
    x = x.reshape(x.size(0), -1)
    y = F.relu(F.linear(y, sd["feat_spe.weight"], sd["feat_spe.bias"]))
    cat = torch.cat([x, y], 1)
    feat = normalize(y)
    if dropout_mask is not None:
        cat = cat * dropout_mask
    logits = F.linear(cat, sd["classifier.weight"], sd["classifier.bias"])
    if return_parts:
        return logits, feat, x, y
    return logits, feat


def test_whole(sd, cube_pca: np.ndarray, spectra: np.ndarray, w: int = 20, batch: int = 512,
               odd_mode: bool = False, rows=None, return_logits: bool = False,
               loop_extract: bool = False):
    """hyper_tools.py:416-437 on top of the patch path: every pixel (or the pixels of
    ``rows=(r0,r1)``) in raster order, argmax with first-index tie rule -> int64 labels."""
    R, C, _ = cube_pca.shape
    r0, r1 = (0, R) if rows is None else rows
    idx_all = np.arange(r0 * C, r1 * C)
    labels, logits_all = [], []
    XP_all = extract_patches_loop(cube_pca, w, odd_mode) if loop_extract else None
    with torch.no_grad():
        for s in range(0, idx_all.size, batch):
            idx = idx_all[s:s + batch]
            XP = XP_all[idx] if loop_extract else extract_patches_at(cube_pca, w, idx, odd_mode)
            lo, _ = basenet2_forward(sd, torch.from_numpy(XP),
                                     torch.from_numpy(spectra[idx].astype(np.float32)))
            labels.append(torch.max(lo, 1)[1].numpy())
            if return_logits:
                logits_all.append(lo.numpy())
    lab = np.concatenate(labels)
    return (lab, np.concatenate(logits_all)) if return_logits else lab


# --------------------------------------------------------------------------
# a14: metrics (hyper_tools.py:208-223)
# --------------------------------------------------------------------------


def confusion_matrix(predict: np.ndarray, label: np.ndarray, num_classes: int) -> np.ndarray:
    """int64 [C, C], rows = true label, cols = prediction (labels outside [0,C) ignored)."""
    cm = np.zeros((num_classes, num_classes), dtype=np.int64)
    ok = (label >= 0) & (label < num_classes) & (predict >= 0) & (predict < num_classes)
    np.add.at(cm, (label[ok].astype(np.int64), predict[ok].astype(np.int64)), 1)
    return cm


def cal_accuracy(predict: np.ndarray, label: np.ndarray):
    """hyper_tools.py:208-223 verbatim semantics (float64 ratios of integer counts)."""
    n = label.shape[0]
    OA = np.sum(predict == label) * 1.0 / n
    nc = int(max(label)) + 1
    correct = np.zeros(nc)
    real = np.zeros(nc)
    pred = np.zeros(nc)
    pa = np.zeros(nc)
    for i in range(nc):
        correct[i] = np.sum(label[np.where(predict == i)] == i)
        real[i] = np.sum(label == i)
        pred[i] = np.sum(predict == i)
        pa[i] = correct[i] / real[i]
    kappa = (n * np.sum(correct) - np.sum(real * pred)) * 1.0 / (n * n - np.sum(real * pred))
    return OA, kappa, pa


def accuracy_from_confusion(cm: np.ndarray, n: int | None = None):
    """OA/kappa/PA from an integer confusion matrix; equals cal_accuracy when every
    prediction lies in [0, C) (diag / row sums / col sums, SURVEY a14)."""
    cm = cm.astype(np.float64)
    n = cm.sum() if n is None else float(n)
    correct = np.diag(cm)
    real = cm.sum(1)
    pred = cm.sum(0)
    OA = correct.sum() * 1.0 / n
    kappa = (n * correct.sum() - np.sum(real * pred)) * 1.0 / (n * n - np.sum(real * pred))
    return OA, kappa, correct / real


# --------------------------------------------------------------------------
# a15: ContrastiveLoss / NT-Xent (models.py:14-39)
# --------------------------------------------------------------------------


def nt_xent(emb_i: torch.Tensor, emb_j: torch.Tensor, temperature: float = 0.5) -> torch.Tensor:
    bs = emb_i.shape[0]
    z = torch.cat([F.normalize(emb_i, dim=1), F.normalize(emb_j, dim=1)], 0)
    S = z @ z.t()                                   # cosine: rows already unit norm
    pos = torch.cat([torch.diag(S, bs), torch.diag(S, -bs)], 0)
    neg_mask = 1.0 - torch.eye(2 * bs, dtype=S.dtype)
    denom = (neg_mask * torch.exp(S / temperature)).sum(1)
    return torch.sum(-torch.log(torch.exp(pos / temperature) / denom)) / (2 * bs)


# --------------------------------------------------------------------------
# a8-a11: the loss terms of train.py:191-265 as functions
# --------------------------------------------------------------------------


def bank_smooth(probs, feats, queue_feats, queue_probs, alpha, T):
    """train.py:213-215."""
    A = torch.exp(feats @ queue_feats.t() / T)
    A = A / A.sum(1, keepdim=True)
    return alpha * probs + (1 - alpha) * (A @ queue_probs)


def soft_ce(logits, probs, mask):
    """train.py:239,241: mean_i( -sum_c log_softmax(z)_ic p_ic * mask_i )."""
    return (-(F.log_softmax(logits, dim=1) * probs).sum(1) * mask).mean()


def graph_targets(probs1, probs):
    """train.py:249-256 -> (Q, Q_n)."""
    Q0 = probs1 @ probs.t()
    Q0.fill_diagonal_(1)
    Q = Q0 * (Q0 >= 0.8).float()
    Q = Q / Q.sum(1, keepdim=True)
    Qn = (1 - Q0) * (Q0 <= 0.3).float()
    Qn = Qn / (Qn.sum(1, keepdim=True) + 1e-8)
    return Q, Qn


def graph_contrast(f_row, f_col, Q, Qn, T):
    """train.py:246-247,260-262 (also :257-258,263-265 with operands swapped by the caller)."""
    sim = torch.exp(f_row @ f_col.t() / T)
    sp = sim / sim.sum(1, keepdim=True)
    return (-(torch.log(sp) * Q).sum(1)).mean() + ((torch.log(sp + 1) * Qn).sum(1)).mean()


def compute_unsupervised_loss(predict, target, percent, pred_teacher):
    """loss_helper.py:242-261 (mutates ``target`` in place like the reference)."""
    batch_size, _ = predict.shape
    with torch.no_grad():
        prob = torch.softmax(pred_teacher, dim=1)
        entropy = -torch.sum(prob * torch.log(prob + 1e-10), dim=1)
        thresh = np.percentile(entropy[target != 255].detach().cpu().numpy().flatten(), percent)
        thresh_mask = entropy.ge(thresh).bool() * (target != 255).bool()
        target[thresh_mask] = 255
        weight = batch_size / torch.sum(target != 255)
    return weight * F.cross_entropy(predict, target, ignore_index=255)


# --------------------------------------------------------------------------
# a7-a12: one mutual-learning step (train.py:146-272), restated as a function
# --------------------------------------------------------------------------


@dataclass
class StepArgs:
    noise: float = 0.5
    alpha: float = 0.95
    temperature: float = 0.3
    thr: float = 1.0
    queue_batch: float = 17
    num_epochs: int = 20
    lr: float = 5e-4
    labeled_batch_size: int = 128


@dataclass
class TrainState:
    """Everything train.py keeps across steps (train.py:118-145)."""
    sd: dict            # Base   (requires_grad leaves)
    sd1: dict           # Base1
    opt: torch.optim.Optimizer
    opt1: torch.optim.Optimizer
    queue_feats: torch.Tensor
    queue_probs: torch.Tensor
    queue_feats1: torch.Tensor
    queue_probs1: torch.Tensor
    queue_ptr: int = 0
    queue_ptr1: int = 0
    extras: dict = field(default_factory=dict)


def make_state(sd, sd1, num_classes, args: StepArgs) -> TrainState:
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    sd1 = {k: v.clone().requires_grad_(True) for k, v in sd1.items()}
    qs = 5 * args.labeled_batch_size * 2                       # train.py:138
    return TrainState(
        sd, sd1,
        torch.optim.Adam(list(sd.values()), lr=args.lr),       # train.py:131
        torch.optim.Adam(list(sd1.values()), lr=args.lr),
        torch.zeros(qs, 1024), torch.zeros(qs, num_classes),
        torch.zeros(qs, 1024), torch.zeros(qs, num_classes))


def ref_step(st: TrainState, XP_l, X_l, Y_l, XP_u, X_u, noise, epoch, batch_index,
             args: StepArgs, drop_masks=(None, None), relu_masks=(None, None)):
    """train.py:150-278.  ``noise`` is a dict of the eight standard-normal tensors the
    reference draws (keys: xp_l1,x_l1,xp_l2,x_l2,xp_u1,x_u1,xp_u2,x_u2; in draw order
    train.py:157,158,163,164,170,171,181,182).  ``relu_masks`` imposes the trunk ReLU masks
    per net (see basenet2_forward).  Returns the five loss_hist columns plus the tensors the
    parity tests compare."""
    T = args.temperature
    st.opt1.zero_grad()
    st.opt.zero_grad()
    bs = XP_l.size(0)
    XP_b_all = torch.cat([XP_l + noise["xp_l1"] * args.noise, XP_u + noise["xp_u1"] * args.noise], 0)
    X_b_all = torch.cat([X_l + noise["x_l1"] * args.noise, X_u + noise["x_u1"] * args.noise], 0)
    XP_e_all = torch.cat([XP_l + noise["xp_l2"] * args.noise, XP_u + noise["xp_u2"] * args.noise], 0)
    X_e_all = torch.cat([X_l + noise["x_l2"] * args.noise, X_u + noise["x_u2"] * args.noise], 0)
    out_b, feat_b = basenet2_forward(st.sd, XP_b_all, X_b_all, drop_masks[0], relu_masks=relu_masks[0])
    out_e, feat_e = basenet2_forward(st.sd1, XP_e_all, X_e_all, drop_masks[1], relu_masks=relu_masks[1])
    labeled_output, x_feature = out_b[:bs], feat_b[:bs]
    un_b_output, xs_feature = out_b[bs:], feat_b[bs:]
    labeled_output1, x_feature1 = out_e[:bs], feat_e[:bs]
    un_e_output, xw_feature = out_e[bs:], feat_e[bs:]

    cls = F.cross_entropy(labeled_output, Y_l)                  # :191
    cls1 = F.cross_entropy(labeled_output1, Y_l)                # :192
    pred1 = torch.max(labeled_output1, 1)[1]                    # :194
    decay_adv = epoch / args.num_epochs                         # :147
    adap_thr = np.exp(-0.5 * (decay_adv ** 2))                  # :148
    with torch.no_grad():                                       # :195-237
        btu, bt = XP_u.size(0), XP_l.size(0)
        n = bt + btu
        C = out_b.size(1)
        feats_u_w = xw_feature.detach()
        probs = torch.softmax(un_e_output.detach(), dim=1)
        probs_orig = probs.clone()
        feats_u_s = xs_feature.detach()
        probs1 = torch.softmax(un_b_output.detach(), dim=1)
        probs_orig1 = probs1.clone()
        if epoch > 0 or batch_index > args.queue_batch:          # :212
            probs = bank_smooth(probs, feats_u_w, st.queue_feats, st.queue_probs, args.alpha, T)
            probs1 = bank_smooth(probs1, feats_u_s, st.queue_feats1, st.queue_probs1, args.alpha, T)
        scores = probs.max(1)[0]
        adap_mask = args.thr * adap_thr
        mask = scores.ge(adap_mask).float()
        onehot = torch.zeros(bt, C).scatter(1, Y_l.view(-1, 1), 1)
        feats_w = torch.cat([feats_u_w, x_feature.detach()], 0)
        probs_w = torch.cat([probs_orig, onehot], 0)
        masks = probs1.max(1)[0].ge(adap_mask).float()
        feats_s = torch.cat([feats_u_s, x_feature1.detach()], 0)
        probs_s = torch.cat([probs_orig1, onehot], 0)
        qs = st.queue_feats.size(0)
        st.queue_feats[st.queue_ptr:st.queue_ptr + n] = feats_w      # :232
        st.queue_probs[st.queue_ptr:st.queue_ptr + n] = probs_w
        st.queue_ptr = (st.queue_ptr + 256) % qs                     # :234 (literal 256)
        st.queue_feats1[st.queue_ptr1:st.queue_ptr1 + n] = feats_s
        st.queue_probs1[st.queue_ptr1:st.queue_ptr1 + n] = probs_s
        st.queue_ptr1 = (st.queue_ptr + 256) % qs                    # :237 (uses queue_ptr: reference quirk)
    con = soft_ce(un_b_output, probs, mask)                     # :239,241
    con1 = soft_ce(un_e_output, probs1, masks)                  # :240,242
    Q, Qn = graph_targets(probs1, probs)                        # :249-256
    lc = graph_contrast(xs_feature, xw_feature.detach(), Q, Qn, T)       # :246,260-262
    lc1 = graph_contrast(xs_feature.detach(), xw_feature, Q, Qn, T)      # :257,263-265
    total = cls + 0.5 * lc + 4 * con                            # :266
    total.backward()
    grads = {k: (v.grad.clone() if v.grad is not None else None) for k, v in st.sd.items()}
    st.opt.step()
    total1 = cls1 + 0.5 * lc1 + 4 * con1                        # :270
    total1.backward()
    grads1 = {k: (v.grad.clone() if v.grad is not None else None) for k, v in st.sd1.items()}
    st.opt1.step()
    acc = torch.mean((pred1 == Y_l).float()).item()             # :278
    hist = np.array([lc.item(), total.item(), cls.item(), con.item(), acc])
    return {"hist": hist, "total1": total1.item(), "cls1": cls1.item(), "con1": con1.item(),
            "lc1": lc1.item(), "logits": out_b.detach(), "logits1": out_e.detach(),
            "feat": feat_b.detach(), "feat1": feat_e.detach(), "probs": probs, "probs1": probs1,
            "mask": mask, "masks": masks, "grads": grads, "grads1": grads1}
