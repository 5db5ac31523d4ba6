"""Thin torch-tensor wrappers over the C ABI (include/cmlpl.h).

torch supplies device memory and the current stream; all arithmetic happens in
libcmlpl_sm100.so.  No wrapper has a non-CUDA code path.
"""
from __future__ import annotations

import torch

from . import _lib

_f32 = torch.float32

# label of a no-data pixel in scene_infer_raw(valid=...) (CMLPL_NODATA_LABEL: never a class, at most 32 classes)
NODATA_LABEL = 255


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _chk(t: torch.Tensor, dtype=_f32, name="tensor"):
    if not t.is_cuda:
        raise _lib.CmlplError(f"{name} must be a CUDA tensor (cmlpl_b200 has no CPU path)")
    if t.dtype != dtype:
        raise _lib.CmlplError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _lib.CmlplError(f"{name} must be contiguous")
    return t


def _p(t):
    return None if t is None else t.data_ptr()


# ------------------------------------------------------------------ patches
def patch_gather(cube: torch.Tensor, w: int, idx: torch.Tensor | None = None, first: int = 0,
                 n: int | None = None, odd_mode: bool = False, scene_rows: int | None = None,
                 slab_row0: int = 0, noise: torch.Tensor | None = None, noise_scale: float = 0.0,
                 out: torch.Tensor | None = None) -> torch.Tensor:
    """hyper_tools.py:226-243 / :300-317 for the pixels ``idx`` (or first..first+n)."""
    _chk(cube, name="cube")
    slab_rows, cols, feat = cube.shape
    scene_rows = slab_rows if scene_rows is None else scene_rows
    if idx is not None:
        _chk(idx, torch.int64, "idx")
        n = idx.numel()
    elif n is None:
        n = scene_rows * cols - first
    if out is None:
        out = torch.empty((n, feat, w, w), dtype=_f32, device=cube.device)
    else:
        _chk(out, name="out")
    if noise is not None:
        _chk(noise, name="noise")
    if n == 0:
        return out
    _lib.call("cmlpl_patch_gather_f32", cube.data_ptr(), scene_rows, cols, feat, slab_row0, slab_rows,
              w, int(odd_mode), _p(idx), first, n, _p(noise), float(noise_scale), out.data_ptr(), _stream())
    return out


# ------------------------------------------------------------------ fp32 blocks
def sgemm(A, B, transA=False, transB=False, bias=None, act=0, out=None, alpha=1.0, beta=0.0):
    """out = act(alpha * op(A) @ op(B) + bias + beta*out); A, B 2-D (any strides)."""
    M, K = (A.shape[1], A.shape[0]) if transA else A.shape
    K2, N = (B.shape[1], B.shape[0]) if transB else B.shape
    assert K == K2, (A.shape, B.shape, transA, transB)
    a_rs, a_cs = (A.stride(1), A.stride(0)) if transA else (A.stride(0), A.stride(1))
    b_rs, b_cs = (B.stride(1), B.stride(0)) if transB else (B.stride(0), B.stride(1))
    if out is None:
        out = torch.empty((M, N), dtype=_f32, device=A.device)
    for t in (A, B, out):
        if not t.is_cuda or t.dtype != _f32:
            raise _lib.CmlplError("sgemm operands must be CUDA float32 tensors")
    _lib.call("cmlpl_sgemm_f32", M, N, K, float(alpha), A.data_ptr(), a_rs, a_cs, B.data_ptr(), b_rs, b_cs,
              _p(bias), float(beta), out.data_ptr(), out.stride(0), out.stride(1), act, _stream())
    return out


def conv2d(x, wgt, bias=None, res=None, relu=False):
    _chk(x, name="x"); _chk(wgt, name="wgt")
    b, ci, h, w = x.shape
    co, ci2, k, _ = wgt.shape
    assert ci == ci2
    y = torch.empty((b, co, h, w), dtype=_f32, device=x.device)
    _lib.call("cmlpl_conv2d_f32", x.data_ptr(), wgt.data_ptr(), _p(bias), _p(res), y.data_ptr(),
              b, ci, co, h, w, k, int(relu), 0, _stream())
    return y


def conv2d_dgrad(dy, wgt, res=None):
    """dL/dx of y = conv(x, wgt, pad=k//2); ``res`` is added (residual branch gradient)."""
    _chk(dy, name="dy"); _chk(wgt, name="wgt")
    b, co, h, w = dy.shape
    co2, ci, k, _ = wgt.shape
    assert co == co2
    dx = torch.empty((b, ci, h, w), dtype=_f32, device=dy.device)
    _lib.call("cmlpl_conv2d_f32", dy.data_ptr(), wgt.data_ptr(), None, _p(res), dx.data_ptr(),
              b, ci, co, h, w, k, 0, 1, _stream())
    return dx


def conv2d_wgrad(x, dy, k):
    _chk(x, name="x"); _chk(dy, name="dy")
    b, ci, h, w = x.shape
    co = dy.shape[1]
    dw = torch.empty((co, ci, k, k), dtype=_f32, device=x.device)
    db = torch.empty((co,), dtype=_f32, device=x.device)
    _lib.call("cmlpl_conv2d_wgrad_f32", x.data_ptr(), dy.data_ptr(), dw.data_ptr(), db.data_ptr(),
              b, ci, co, h, w, k, _stream())
    return dw, db


def avgpool2(x):
    _chk(x, name="x")
    b, c, h, w = x.shape
    y = torch.empty((b, c, h // 2, w // 2), dtype=_f32, device=x.device)
    _lib.call("cmlpl_avgpool2_f32", x.data_ptr(), y.data_ptr(), b * c, h, w, _stream())
    return y


def avgpool2_bwd(dy, h, w):
    _chk(dy, name="dy")
    b, c = dy.shape[:2]
    dx = torch.empty((b, c, h, w), dtype=_f32, device=dy.device)
    _lib.call("cmlpl_avgpool2_bwd_f32", dy.data_ptr(), dx.data_ptr(), b * c, h, w, _stream())
    return dx


def relu_bwd(y, dy):
    _chk(y, name="y"); _chk(dy, name="dy")
    dx = torch.empty_like(dy)
    _lib.call("cmlpl_relu_bwd_f32", y.data_ptr(), dy.data_ptr(), dx.data_ptr(), y.numel(), _stream())
    return dx


def colsum(x):
    _chk(x, name="x")
    m, n = x.shape
    out = torch.empty((n,), dtype=_f32, device=x.device)
    _lib.call("cmlpl_colsum_f32", x.data_ptr(), out.data_ptr(), m, n, _stream())
    return out


def l2norm(x, eps=0.0):
    """x / max(||x||, eps) per row -> (y, unclamped norm).  eps = 0: models.py:87-90 Normalize (a zero row gives NaN);
    eps = 1e-12: F.normalize."""
    _chk(x, name="x")
    rows, cols = x.shape
    y = torch.empty_like(x)
    norm = torch.empty((rows,), dtype=_f32, device=x.device)
    _lib.call("cmlpl_l2norm_f32", x.data_ptr(), y.data_ptr(), norm.data_ptr(), rows, cols, float(eps), _stream())
    return y, norm


def l2norm_bwd(y, norm, dy, eps=0.0):
    """Backward of l2norm(x, eps) given its outputs."""
    _chk(y, name="y"); _chk(dy, name="dy")
    dx = torch.empty_like(dy)
    _lib.call("cmlpl_l2norm_bwd_f32", y.data_ptr(), norm.data_ptr(), dy.data_ptr(), dx.data_ptr(),
              y.shape[0], y.shape[1], float(eps), _stream())
    return dx


# ------------------------------------------------------------------ scene inference
def pack_basenet2(sd: dict, num_features: int, num_classes: int, w: int = 20) -> torch.Tensor:
    """Repack reference-keyed weights (models.py:102-127) for the scene kernels."""
    keys = ("conv0.weight", "conv0.bias", "conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias",
            "feat_spe.weight", "feat_spe.bias", "classifier.weight", "classifier.bias")
    ts = [_chk(sd[k].detach().contiguous(), name=k) for k in keys]
    lib = _lib.load()
    nbytes = lib.cmlpl_packed_bytes(num_features, num_classes, w)
    packed = torch.empty((nbytes,), dtype=torch.uint8, device=ts[0].device)
    _lib.call("cmlpl_pack_basenet2", *[t.data_ptr() for t in ts], num_features, num_classes, w,
              packed.data_ptr(), _stream())
    packed._cmlpl_keepalive = ts
    return packed


def scene_workspace(band_rows: int, cols: int, num_features: int, num_classes: int, w: int, device) -> torch.Tensor:
    nbytes = _lib.load().cmlpl_scene_workspace_bytes(band_rows, cols, num_features, num_classes, w)
    return torch.empty((nbytes,), dtype=torch.uint8, device=device)


def scene_infer(cube, spectra, packed, num_classes: int, w: int = 20, band_row0: int = 0,
                band_rows: int | None = None, scene_rows: int | None = None, slab_row0: int = 0,
                want_logits: bool = False, workspace: torch.Tensor | None = None,
                labels: torch.Tensor | None = None):
    """hyper_tools.py:416-437 for scene rows [band_row0, band_row0+band_rows).

    cube f32 [slab_rows, cols, 60] (rows slab_row0.. of the scene), spectra f32 [band_rows*cols, B].
    Returns uint8 labels [band_rows*cols] (and f32 logits when asked)."""
    _chk(cube, name="cube"); _chk(spectra, name="spectra")
    slab_rows, cols, f = cube.shape
    if f != 60:
        raise _lib.CmlplError("BaseNet2.conv0 is hard-wired to 60 PCA channels (models.py:102)")
    scene_rows = slab_rows if scene_rows is None else scene_rows
    band_rows = scene_rows - band_row0 if band_rows is None else band_rows
    n = band_rows * cols
    B = spectra.shape[1]
    if spectra.shape[0] != n:
        raise _lib.CmlplError(f"spectra has {spectra.shape[0]} rows, band has {n} pixels")
    if workspace is None:
        workspace = scene_workspace(band_rows, cols, B, num_classes, w, cube.device)
    if labels is None:
        labels = torch.empty((n,), dtype=torch.uint8, device=cube.device)
    logits = torch.empty((n, num_classes), dtype=_f32, device=cube.device) if want_logits else None
    _lib.call("cmlpl_scene_infer", cube.data_ptr(), scene_rows, cols, slab_row0, slab_rows, spectra.data_ptr(),
              B, num_classes, w, band_row0, band_rows, packed.data_ptr(), workspace.data_ptr(),
              workspace.numel(), labels.data_ptr(), _p(logits), _stream())
    return (labels, logits) if want_logits else labels


def scene_infer_raw(raw, folded, packed, num_classes: int, cols: int, w: int = 20, band_row0: int = 0,
                    band_rows: int | None = None, scene_rows: int | None = None, slab_row0: int = 0,
                    want_logits: bool = False, workspace: torch.Tensor | None = None,
                    labels: torch.Tensor | None = None, interleave: str = "bip", valid: torch.Tensor | None = None):
    """hyper_tools.py:285-292 + :416-437 from the RAW cube: raw uint16 / f32 / int16 holding scene rows slab_row0..
    in the layout ``interleave`` -- "bip" [slab_rows*cols, B] or [slab_rows, cols, B], "bil" [slab_rows, B, cols],
    "bsq" [B, slab_rows, cols] -- and ``folded`` = Preproc.folded_conv0(...) (conv0 folded with PCA + z-scores; band
    mean / 1/std).  Neither the PCA cube nor the z-scored spectra are materialised.  Results do not depend on the
    interleave.

    ``valid`` (u8 [slab_rows, cols], 1 = valid; preprocess.valid_mask or any mask of that layout): a no-data pixel
    stands in as its band-mean spectrum wherever it is read -- in its neighbours' windows and as its own spectral input
    -- and is labelled NODATA_LABEL; its logits, when asked for, are those of the imputed pixel."""
    from . import preprocess
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("raw must be a contiguous CUDA tensor (cmlpl_b200 has no CPU path)")
    code = preprocess._dtype_code(raw)
    slab_rows, _, B = preprocess.raw_geometry(raw.shape, interleave, cols=cols)
    code |= preprocess.INTERLEAVE[interleave]
    scene_rows = slab_rows if scene_rows is None else scene_rows
    band_rows = scene_rows - band_row0 if band_rows is None else band_rows
    n = band_rows * cols
    for k in ("wf", "bf", "mu", "inv_sigma"):
        _chk(folded[k], name=k)
    if folded["wf"].shape != (B, 64):
        raise _lib.CmlplError(f"folded conv0 weight must be [{B}, 64]")
    if workspace is None:
        workspace = scene_workspace(band_rows, cols, B, num_classes, w, raw.device)
    if labels is None:
        labels = torch.empty((n,), dtype=torch.uint8, device=raw.device)
    logits = torch.empty((n, num_classes), dtype=_f32, device=raw.device) if want_logits else None
    pre = (folded["wf"].data_ptr(), folded["bf"].data_ptr(), folded["mu"].data_ptr(), folded["inv_sigma"].data_ptr())
    post = (packed.data_ptr(), workspace.data_ptr(), workspace.numel(), labels.data_ptr(), _p(logits), _stream())
    geom = (code, scene_rows, cols, slab_row0, slab_rows, B, num_classes, w, band_row0, band_rows)
    if valid is None:
        _lib.call("cmlpl_scene_infer_raw", raw.data_ptr(), *geom, *pre, *post)
    else:
        _chk(valid, torch.uint8, "valid")
        if valid.numel() != slab_rows * cols:
            raise _lib.CmlplError(f"valid has {valid.numel()} pixels, the slab {slab_rows} x {cols}")
        _lib.call("cmlpl_scene_infer_raw_masked", raw.data_ptr(), *geom, *pre, valid.data_ptr(), *post)
    return (labels, logits) if want_logits else labels


def argmax_u8(logits):
    _chk(logits, name="logits")
    n, c = logits.shape
    out = torch.empty((n,), dtype=torch.uint8, device=logits.device)
    _lib.call("cmlpl_argmax_u8", logits.data_ptr(), n, c, out.data_ptr(), _stream())
    return out


def confusion(pred_u8, label_i64, num_classes: int, cm: torch.Tensor | None = None):
    _chk(pred_u8, torch.uint8, "pred"); _chk(label_i64, torch.int64, "label")
    if cm is None:
        cm = torch.zeros((num_classes, num_classes), dtype=torch.int64, device=pred_u8.device)
    _lib.call("cmlpl_confusion_i64", pred_u8.data_ptr(), label_i64.data_ptr(), pred_u8.numel(), num_classes,
              cm.data_ptr(), _stream())
    return cm


# ------------------------------------------------------------------ losses / optimizer
def ce_fwd_bwd(logits, labels=None, probs=None, mask=None, scale=1.0, want_grad=True):
    """train.py:191 (labels) / :239-242 (probs, mask) -> (loss scalar tensor, dlogits or None)."""
    _chk(logits, name="logits")
    rows, C = logits.shape
    loss = torch.zeros((), dtype=_f32, device=logits.device)
    dz = torch.empty_like(logits) if want_grad else None
    if labels is not None:
        _chk(labels, torch.int64, "labels")
    if probs is not None:
        _chk(probs, name="probs")
    if mask is not None:
        _chk(mask, name="mask")
    _lib.call("cmlpl_ce_fwd_bwd_f32", logits.data_ptr(), _p(labels), _p(probs), _p(mask), rows, C, float(scale),
              loss.data_ptr(), _p(dz), _stream())
    return loss, dz


def softmax_js(logits, targets, scale=1.0, want_grad=True):
    """trian_CCT.py:76-84 -> (scale*L, scale*dL/dlogits)."""
    _chk(logits, name="logits"); _chk(targets, name="targets")
    if logits.shape != targets.shape or logits.dim() != 2:
        raise _lib.CmlplError("softmax_js: logits and targets must be [rows, C] of the same shape")
    rows, C = logits.shape
    loss = torch.zeros((), dtype=_f32, device=logits.device)
    dz = torch.empty_like(logits) if want_grad else None
    _lib.call("cmlpl_softmax_js_f32", logits.data_ptr(), targets.data_ptr(), rows, C, float(scale), loss.data_ptr(),
              _p(dz), _stream())
    return loss, dz


def bank_smooth(logits, feats, queue_feats, queue_probs, alpha, T, smooth, thr):
    """train.py:203-222 -> (probs_orig, probs, mask)."""
    _chk(logits, name="logits")
    rows, C = logits.shape
    probs_orig = torch.empty_like(logits)
    probs = torch.empty_like(logits)
    mask = torch.empty((rows,), dtype=_f32, device=logits.device)
    work = None
    queue, dim = 0, 0
    if smooth:
        _chk(feats, name="feats"); _chk(queue_feats, name="queue_feats"); _chk(queue_probs, name="queue_probs")
        queue, dim = queue_feats.shape
        work = torch.empty((rows, queue), dtype=_f32, device=logits.device)
    _lib.call("cmlpl_bank_smooth_f32", logits.data_ptr(), _p(feats), _p(queue_feats), _p(queue_probs), rows, C, dim,
              queue, float(alpha), float(T), int(bool(smooth)), float(thr), _p(work), probs_orig.data_ptr(),
              probs.data_ptr(), mask.data_ptr(), _stream())
    return probs_orig, probs, mask


def graph_contrast(f_row, f_col, p1, p, T, grad_side, scale=1.0, want_grad=True):
    """train.py:246-265 -> (scale*L, scale*dL/d(f_row|f_col))."""
    for t, n in ((f_row, "f_row"), (f_col, "f_col"), (p1, "p1"), (p, "p")):
        _chk(t, name=n)
    n, dim = f_row.shape
    C = p.shape[1]
    work = torch.empty((3 * n * n,), dtype=_f32, device=f_row.device)
    loss = torch.zeros((), dtype=_f32, device=f_row.device)
    df = torch.empty_like(f_row) if want_grad else None
    _lib.call("cmlpl_graph_contrast_f32", f_row.data_ptr(), f_col.data_ptr(), p1.data_ptr(), p.data_ptr(), n, dim, C,
              float(T), int(grad_side), float(scale), work.data_ptr(), loss.data_ptr(), _p(df), _stream())
    return loss, df


def ntxent(z, bs, T, want_grad=True):
    """models.py:22-39 on unit-norm rows z [2bs, dim] -> (L, dL/dz)."""
    _chk(z, name="z")
    n, dim = z.shape
    assert n == 2 * bs
    work = torch.empty((2 * n * n,), dtype=_f32, device=z.device)
    loss = torch.zeros((), dtype=_f32, device=z.device)
    dz = torch.empty_like(z) if want_grad else None
    _lib.call("cmlpl_ntxent_f32", z.data_ptr(), bs, dim, float(T), work.data_ptr(), loss.data_ptr(), _p(dz), _stream())
    return loss, dz


def adam_multi(params, grads, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, step):
    """One fused Adam update over a list of tensors (grads entries may be None = skipped)."""
    import ctypes
    n = len(params)
    PP = ctypes.c_void_p * n
    LL = ctypes.c_int64 * n
    for t in list(params) + list(exp_avg) + list(exp_avg_sq) + [g for g in grads if g is not None]:
        _chk(t, name="adam tensor")
    _lib.call("cmlpl_adam_multi_f32", n, PP(*[t.data_ptr() for t in params]),
              PP(*[(g.data_ptr() if g is not None else None) for g in grads]),
              PP(*[t.data_ptr() for t in exp_avg]), PP(*[t.data_ptr() for t in exp_avg_sq]),
              LL(*[t.numel() for t in params]), float(lr), float(beta1), float(beta2), float(eps), int(step), _stream())


def softmax_entropy(logits, eps=1e-10):
    """loss_helper.py:247-248 -> f32 [rows]."""
    _chk(logits, name="logits")
    rows, C = logits.shape
    ent = torch.empty((rows,), dtype=_f32, device=logits.device)
    _lib.call("cmlpl_softmax_entropy_f32", logits.data_ptr(), rows, C, float(eps), ent.data_ptr(), _stream())
    return ent
