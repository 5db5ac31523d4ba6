"""Scene preprocessing on the GPU (SURVEY 8-f1): the reference's ``featureNormalize`` + ``PCANorm``
(tools/hyper_tools.py:8-32, used at :289-292) as fit (float64 moments on device, B x B SVD on the
host) and apply (raw cube -> z-scored spectra + z-scored PCA cube in one pass).  Both inputs of the
scene path are affine functions of the raw cube, so ``apply`` lets the end-to-end entry point ship only
the raw uint16 cube over PCIe."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib


@dataclass
class Preproc:
    mu: np.ndarray          # f64 [B]   band means                         (featureNormalize / PCANorm mean)
    sigma: np.ndarray       # f64 [B]   band population std                (np.std, hyper_tools.py:14)
    U: np.ndarray           # f64 [B, n_PC] leading left-singular vectors of np.cov   (hyper_tools.py:29-31)
    pca_mu: np.ndarray      # f64 [n_PC] mean of the projected data (~0)
    pca_sigma: np.ndarray   # f64 [n_PC] population std of the projected data
    _dev: dict = None

    def device_params(self, device):
        if self._dev is None or self._dev["device"] != device:
            t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device)
            self._dev = {"device": device, "mu": t(self.mu), "inv_sigma": t(1.0 / self.sigma),
                         "Us": t(self.U / self.pca_sigma[None, :]), "shift": t(self.pca_mu / self.pca_sigma)}
        return self._dev

    def folded_conv0(self, conv0_w, conv0_b, device):
        """PCA projection, both z-scores and conv0 (models.py:102,132) are per-pixel affine maps of the raw
        spectrum, so they fold into F0 = wf^T (x - mu) + bf (SURVEY 8-f1).  Returns device f32 tensors
        wf [B, 64], bf [64] (+ mu, inv_sigma [B]) for cmlpl_scene_infer_raw; folded in float64 on the host."""
        W0 = conv0_w.detach().double().cpu().numpy().reshape(conv0_w.shape[0], -1)        # [64, n_PC]
        b0 = conv0_b.detach().double().cpu().numpy()
        Us = self.U / self.pca_sigma[None, :]                                              # [B, n_PC]
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device)
        d = self.device_params(device)
        return {"wf": t(Us @ W0.T), "bf": t(b0 - W0 @ (self.pca_mu / self.pca_sigma)), "mu": d["mu"],
                "inv_sigma": d["inv_sigma"]}


def _dtype_code(x: torch.Tensor) -> int:
    """The raw sample type code of include/cmlpl.h (CMLPL_RAW_U16 / F32 / I16)."""
    if x.dtype == torch.uint16:
        return 0
    if x.dtype == torch.float32:
        return 1
    if x.dtype == torch.int16:
        return 2
    raise _lib.CmlplError(f"raw scene must be uint16, float32 or int16, got {x.dtype}")


# interleave codes of include/cmlpl.h (CMLPL_RAW_BIP / BIL / BSQ), or'ed into the sample type code
INTERLEAVE = {"bip": 0x00, "bil": 0x10, "bsq": 0x20}


def raw_geometry(shape, interleave: str = "bip", cols: int | None = None, bands: int | None = None):
    """(rows, cols, bands) of a raw cube of this shape, checked against ``cols`` / ``bands`` when given:
    BIP [rows*cols, B] or [rows, cols, B]; BIL [rows, B, cols]; BSQ [B, rows, cols].  A 2-D BIP cube without
    ``cols`` is one row per pixel (rows = N, cols = 1).  Raises CmlplError on a mismatch."""
    if interleave not in INTERLEAVE:
        raise _lib.CmlplError(f"interleave must be one of {sorted(INTERLEAVE)}, got {interleave!r}")
    shape = tuple(int(d) for d in shape)
    if interleave == "bip" and len(shape) == 2:
        n, B = shape
        c = 1 if cols is None else cols
        if c <= 0 or n % c:
            raise _lib.CmlplError(f"raw BIP [rows*cols, B] = {list(shape)}: rows are not a multiple of cols = {cols}")
        r = n // c
    elif len(shape) == 3:
        r, c, B = {"bip": (0, 1, 2), "bil": (0, 2, 1), "bsq": (1, 2, 0)}[interleave]
        r, c, B = shape[r], shape[c], shape[B]
        if cols is not None and c != cols:
            raise _lib.CmlplError(f"raw {interleave.upper()} {list(shape)} has {c} columns, expected {cols}")
    else:
        want = {"bip": "[rows*cols, B] or [rows, cols, B]", "bil": "[rows, B, cols]", "bsq": "[B, rows, cols]"}
        raise _lib.CmlplError(f"raw {interleave.upper()} must be {want[interleave]}, got {list(shape)}")
    if bands is not None and B != bands:
        raise _lib.CmlplError(f"raw {interleave.upper()} {list(shape)} has {B} bands, expected {bands}")
    if r <= 0 or c <= 0 or B <= 0:
        raise _lib.CmlplError(f"raw {interleave.upper()} {list(shape)} is empty")
    if max(c, B) >= 2 ** 31 or (interleave != "bip" and r >= 2 ** 31):    # the C int arguments (BIP rows are int64)
        raise _lib.CmlplError(f"raw {interleave.upper()} {list(shape)}: a dimension exceeds the library's int range")
    return r, c, B


def _fill_value(raw: torch.Tensor, fill):
    """The fill value of ``valid_mask`` as the library takes it: None is NaN (non-finite samples only) for float32 and an
    error for integer cubes."""
    if fill is None:
        if raw.dtype != torch.float32:
            raise _lib.CmlplError(f"valid_mask: a {raw.dtype} cube needs its fill value (fill=None means NaN / Inf only, "
                                  "for float32)")
        return float("nan")
    return float(fill)


def valid_mask(raw: torch.Tensor, fill=None, interleave: str = "bip", cols: int | None = None):
    """No-data pixels of a raw CUDA cube in the layout ``interleave`` (see ``raw_geometry``; a 2-D BIP cube takes ``cols``).
    A sample is missing when it equals ``fill`` in the sample type, and a float32 sample also when it is not finite (fill
    None: only then); a pixel with any band missing is no-data.  One read of the cube on the device.
    -> (valid u8 CUDA [rows, cols] with 1 = valid, n_valid, band_missing int64 [B] = pixels in which each band is missing)."""
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("valid_mask needs a contiguous CUDA tensor")
    rows, c, B = raw_geometry(raw.shape, interleave, cols=cols)
    valid = torch.empty((rows, c), dtype=torch.uint8, device=raw.device)
    counts = torch.empty(B + 1, dtype=torch.int64, device=raw.device)          # [n_valid, band_missing[B]]
    mask_into(raw, fill, interleave, rows, c, B, valid, counts)
    counts = counts.cpu().numpy()
    return valid, int(counts[0]), counts[1:]


def mask_into(raw: torch.Tensor, fill, interleave: str, rows: int, cols: int, B: int, valid: torch.Tensor,
              counts: torch.Tensor):
    """valid_mask without a host synchronisation, into caller buffers: valid u8 [rows * cols] and counts int64 [B + 1]
    (n_valid, then band_missing), on the current stream.  ``raw`` holds the rows x cols pixels in ``interleave``."""
    _lib.call("cmlpl_valid_mask_u8", raw.data_ptr(), _dtype_code(raw) | INTERLEAVE[interleave], rows, cols, B,
              _fill_value(raw, fill), valid.data_ptr(), counts.data_ptr(), counts.data_ptr() + 8,
              torch.cuda.current_stream().cuda_stream)


def _check_valid(valid: torch.Tensor, n: int, what: str):
    if not valid.is_cuda or valid.dtype != torch.uint8 or not valid.is_contiguous() or valid.numel() != n:
        raise _lib.CmlplError(f"{what}: valid must be a contiguous uint8 CUDA mask of {n} pixels, got {valid.dtype} "
                              f"{list(valid.shape)}")


def fit(raw: torch.Tensor, n_PC: int = 60, interleave: str = "bip", valid: torch.Tensor | None = None,
        fill=None) -> Preproc:
    """raw: CUDA tensor (uint16, float32 or int16) in the layout ``interleave`` (see ``raw_geometry``).  Moments in
    float64 on device, SVD on the host.  ``valid`` (u8 [rows, cols], ``valid_mask``) or ``fill`` (its mask is built
    here): the moments of the valid pixels only.  Fewer than 2 valid pixels raise an error that names the bands missing
    in every pixel (known when ``fill`` is given)."""
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("fit needs a contiguous CUDA tensor")
    rows, cols, B = raw_geometry(raw.shape, interleave)
    n = rows * cols
    mean = torch.empty(B, dtype=torch.float64, device=raw.device)
    gram = torch.empty(B, B, dtype=torch.float64, device=raw.device)
    stream = torch.cuda.current_stream().cuda_stream
    band_missing = None
    if fill is not None:
        if valid is not None:
            raise _lib.CmlplError("fit: pass valid= or fill=, not both")
        valid, _, band_missing = valid_mask(raw, fill, interleave)
    if valid is not None:
        _check_valid(valid, n, "fit")
        count = torch.empty(1, dtype=torch.int64, device=raw.device)
        _lib.call("cmlpl_preprocess_fit_masked_f64", raw.data_ptr(), _dtype_code(raw) | INTERLEAVE[interleave], rows, cols,
                  B, valid.data_ptr(), mean.data_ptr(), gram.data_ptr(), count.data_ptr(), stream)
        n = int(count.item())
        if n < 2:
            every = [] if band_missing is None else [int(b) for b in np.flatnonzero(band_missing == rows * cols)]
            raise _lib.CmlplError(f"fit: {n} valid pixels of {rows * cols}; the moments need at least 2"
                                  + (f"; bands missing in every pixel: {every}" if every else ""))
    elif interleave == "bip":                                     # one pixel per row: the int64 pixel count
        _lib.call("cmlpl_preprocess_fit_f64", raw.data_ptr(), _dtype_code(raw), n, B, mean.data_ptr(), gram.data_ptr(),
                  stream)
    else:
        _lib.call("cmlpl_preprocess_fit_cube_f64", raw.data_ptr(), _dtype_code(raw) | INTERLEAVE[interleave], rows, cols,
                  B, mean.data_ptr(), gram.data_ptr(), stream)
    g = gram.cpu().numpy()
    g = np.triu(g) + np.triu(g, 1).T                              # the kernel fills upper tiles only
    mu = mean.cpu().numpy()
    U = np.linalg.svd(g / (n - 1))[0][:, :n_PC]                   # np.cov + np.linalg.svd (hyper_tools.py:29-30)
    pca_var = np.einsum("bk,bc,ck->k", U, g, U) / n               # population variance of the projection
    return Preproc(mu=mu, sigma=np.sqrt(np.diag(g) / n), U=U, pca_mu=np.zeros(n_PC), pca_sigma=np.sqrt(pca_var))


def apply(raw: torch.Tensor, pp: Preproc, want_spectra: bool = True, cube: torch.Tensor | None = None,
          spectra: torch.Tensor | None = None, valid: torch.Tensor | None = None):
    """raw CUDA [N, B] (BIP) -> (cube f32 [N, n_PC], spectra f32 [N, B] or None).  ``valid`` (u8 [N] or [rows, cols]):
    a no-data pixel is written as its band means, i.e. spectra row 0 and cube row -shift."""
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("apply needs a contiguous CUDA tensor")
    n, B = raw.shape
    d = pp.device_params(raw.device)
    npc = d["Us"].shape[1]
    if cube is None:
        cube = torch.empty((n, npc), dtype=torch.float32, device=raw.device)
    if want_spectra and spectra is None:
        spectra = torch.empty((n, B), dtype=torch.float32, device=raw.device)
    args = (raw.data_ptr(), _dtype_code(raw), n, B, npc, d["mu"].data_ptr(), d["inv_sigma"].data_ptr(), d["Us"].data_ptr(),
            d["shift"].data_ptr())
    outs = (cube.data_ptr(), spectra.data_ptr() if want_spectra else None, torch.cuda.current_stream().cuda_stream)
    if valid is None:
        _lib.call("cmlpl_preprocess_apply", *args, *outs)
    else:
        _check_valid(valid, n, "apply")
        _lib.call("cmlpl_preprocess_apply_masked", *args, valid.data_ptr(), *outs)
    return cube, (spectra if want_spectra else None)
