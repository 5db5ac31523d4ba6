"""Scene preprocessing on the GPU (SURVEY 8-f1): the reference's ``featureNormalize`` + ``PCANorm``
(tools/hyper_tools.py:8-32, used at :289-292) as fit (float64 moments on device, B x B SVD on the
host) and apply (raw cube -> z-scored spectra + z-scored PCA cube in one pass).  Both inputs of the
scene path are affine functions of the raw cube, so ``apply`` lets the end-to-end entry point ship only
the raw uint16 cube over PCIe.

Band selection: ``bands`` (strictly increasing raw band indices) makes the mask, the fit and the apply read only those
bands of the cube -- e.g. the "corrected" bands of an AVIRIS product without its water-absorption bands, or a Hyperion
L1R cube without its uncalibrated, zero-filled bands (``dead_bands`` finds those).  A ``Preproc`` fitted with a list
records it, and ``folded_conv0`` hands it to ``ops.scene_infer_raw``, so the fit and the scene call read the same bands."""
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
    bands: np.ndarray | None = None   # i32 [nsel] raw bands the fit read (features = these bands), or None: all of them
    raw_bands: int | None = None      # band count of the raw cube the fit read

    def device_params(self, device):
        if self._dev is None or self._dev["device"] != device:
            t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device)
            self._dev = {"device": device, "mu": t(self.mu), "inv_sigma": t(1.0 / self.sigma),
                         "Us": t(self.U / self.pca_sigma[None, :]), "shift": t(self.pca_mu / self.pca_sigma)}
        return self._dev

    def folded_conv0(self, conv0_w, conv0_b, device):
        """PCA projection, both z-scores and conv0 (models.py:102,132) are per-pixel affine maps of the raw
        spectrum, so they fold into F0 = wf^T (x - mu) + bf (SURVEY 8-f1).  Returns device f32 tensors
        wf [B, 64], bf [64] (+ mu, inv_sigma [B]) for cmlpl_scene_infer_raw; folded in float64 on the host.  B is the
        number of features: the listed bands of a fit with ``bands``, which come along as "bands" (host i32, or None) and
        "raw_bands" (the raw cube's band count)."""
        W0 = conv0_w.detach().double().cpu().numpy().reshape(conv0_w.shape[0], -1)        # [64, n_PC]
        b0 = conv0_b.detach().double().cpu().numpy()
        Us = self.U / self.pca_sigma[None, :]                                              # [B, n_PC]
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device)
        d = self.device_params(device)
        return {"wf": t(Us @ W0.T), "bf": t(b0 - W0 @ (self.pca_mu / self.pca_sigma)), "mu": d["mu"],
                "inv_sigma": d["inv_sigma"], "bands": self.bands, "raw_bands": self.raw_bands}


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


def band_list(bands) -> np.ndarray:
    """``bands`` as the library takes it: a contiguous host int32 array (the library checks that it is non-empty, strictly
    increasing and inside the cube's bands)."""
    a = np.asarray(bands.cpu() if isinstance(bands, torch.Tensor) else bands)
    if a.ndim != 1 or not (a.size == 0 or np.issubdtype(a.dtype, np.integer)):
        raise _lib.CmlplError(f"bands must be a 1-D list of band indices, got {a.dtype} {list(a.shape)}")
    if a.size and (a.min() < np.iinfo(np.int32).min or a.max() > np.iinfo(np.int32).max):
        raise _lib.CmlplError("bands: an entry exceeds the int32 range")
    return np.ascontiguousarray(a, dtype=np.int32)


def _fill_value(raw: torch.Tensor, fill):
    """The fill value of ``valid_mask`` as the library takes it: None is NaN (non-finite samples only) for float32 and an
    error for integer cubes."""
    if fill is None:
        if raw.dtype != torch.float32:
            raise _lib.CmlplError(f"valid_mask: a {raw.dtype} cube needs its fill value (fill=None means NaN / Inf only, "
                                  "for float32)")
        return float("nan")
    return float(fill)


def valid_mask(raw: torch.Tensor, fill=None, interleave: str = "bip", cols: int | None = None, bands=None):
    """No-data pixels of a raw CUDA cube in the layout ``interleave`` (see ``raw_geometry``; a 2-D BIP cube takes ``cols``).
    A sample is missing when it equals ``fill`` in the sample type, and a float32 sample also when it is not finite (fill
    None: only then); a pixel with any band missing is no-data.  One read of the cube on the device.  ``bands``: only
    these raw bands decide, and band_missing has one entry per listed band.
    -> (valid u8 CUDA [rows, cols] with 1 = valid, n_valid, band_missing int64 [B] = pixels in which each band is missing)."""
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("valid_mask needs a contiguous CUDA tensor")
    rows, c, B = raw_geometry(raw.shape, interleave, cols=cols)
    nf = B if bands is None else band_list(bands).size
    valid = torch.empty((rows, c), dtype=torch.uint8, device=raw.device)
    counts = torch.empty(nf + 1, dtype=torch.int64, device=raw.device)          # [n_valid, band_missing[nf]]
    mask_into(raw, fill, interleave, rows, c, B, valid, counts, bands)
    counts = counts.cpu().numpy()
    return valid, int(counts[0]), counts[1:]


def mask_into(raw: torch.Tensor, fill, interleave: str, rows: int, cols: int, B: int, valid: torch.Tensor,
              counts: torch.Tensor, bands=None):
    """valid_mask without a host synchronisation, into caller buffers: valid u8 [rows * cols] and counts int64 [nf + 1]
    (n_valid, then band_missing), on the current stream.  ``raw`` holds the rows x cols pixels of B bands in
    ``interleave``; ``bands`` (nf of them, else nf = B) decide."""
    head = (raw.data_ptr(), _dtype_code(raw) | INTERLEAVE[interleave], rows, cols, B)
    tail = (_fill_value(raw, fill), valid.data_ptr(), counts.data_ptr(), counts.data_ptr() + 8,
            torch.cuda.current_stream().cuda_stream)
    if bands is None:
        _lib.call("cmlpl_valid_mask_u8", *head, *tail)
    else:
        sel = band_list(bands)
        _lib.call("cmlpl_valid_mask_sel_u8", *head, sel.ctypes.data, sel.size, *tail)


def _check_valid(valid: torch.Tensor, n: int, what: str):
    if not valid.is_cuda or valid.dtype != torch.uint8 or not valid.is_contiguous() or valid.numel() != n:
        raise _lib.CmlplError(f"{what}: valid must be a contiguous uint8 CUDA mask of {n} pixels, got {valid.dtype} "
                              f"{list(valid.shape)}")


def _zero_variance(mu: np.ndarray, var: np.ndarray) -> np.ndarray:
    """Bands whose values are all equal: a population std at the rounding level of the float64 mean."""
    return np.sqrt(np.maximum(var, 0.0)) <= 1e-9 * np.maximum(np.abs(mu), 1.0)


def _moments_sel(raw, interleave, rows, cols, B, sel, valid):
    """Device moments of the listed bands (cmlpl_preprocess_fit_sel_f64) -> (mean [nsel], full gram [nsel, nsel], pixel
    count)."""
    nsel = sel.size
    mean = torch.empty(nsel, dtype=torch.float64, device=raw.device)
    gram = torch.empty(nsel, nsel, dtype=torch.float64, device=raw.device)
    count = torch.empty(1, dtype=torch.int64, device=raw.device)
    _lib.call("cmlpl_preprocess_fit_sel_f64", raw.data_ptr(), _dtype_code(raw) | INTERLEAVE[interleave], rows, cols, B,
              sel.ctypes.data, nsel, None if valid is None else valid.data_ptr(), mean.data_ptr(), gram.data_ptr(),
              None if valid is None else count.data_ptr(), torch.cuda.current_stream().cuda_stream)
    n = rows * cols if valid is None else int(count.item())
    g = gram.cpu().numpy()
    return mean.cpu().numpy(), np.triu(g) + np.triu(g, 1).T, n


def fit(raw: torch.Tensor, n_PC: int = 60, interleave: str = "bip", valid: torch.Tensor | None = None,
        fill=None, bands=None) -> Preproc:
    """raw: CUDA tensor (uint16, float32 or int16) in the layout ``interleave`` (see ``raw_geometry``).  Moments in
    float64 on device, SVD on the host.  ``valid`` (u8 [rows, cols], ``valid_mask``) or ``fill`` (its mask is built
    here): the moments of the valid pixels only.  Fewer than 2 valid pixels raise an error that names the bands missing
    in every pixel (known when ``fill`` is given).  ``bands``: the fit reads only these raw bands (the mask built from
    ``fill`` too), refuses a listed band with zero variance, and the Preproc records the list."""
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("fit needs a contiguous CUDA tensor")
    rows, cols, B = raw_geometry(raw.shape, interleave)
    if bands is not None:
        return _fit_sel(raw, n_PC, interleave, valid, fill, band_list(bands), rows, cols, B)
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
    return _from_moments(mu, g, n, n_PC, raw_bands=B)


def _from_moments(mu, g, n, n_PC, raw_bands, bands=None) -> Preproc:
    U = np.linalg.svd(g / (n - 1))[0][:, :n_PC]                   # np.cov + np.linalg.svd (hyper_tools.py:29-30)
    pca_var = np.einsum("bk,bc,ck->k", U, g, U) / n               # population variance of the projection
    return Preproc(mu=mu, sigma=np.sqrt(np.diag(g) / n), U=U, pca_mu=np.zeros(n_PC), pca_sigma=np.sqrt(pca_var),
                   bands=bands, raw_bands=raw_bands)


def _fit_sel(raw, n_PC, interleave, valid, fill, sel, rows, cols, B) -> Preproc:
    band_missing = None
    if fill is not None:
        if valid is not None:
            raise _lib.CmlplError("fit: pass valid= or fill=, not both")
        valid, _, band_missing = valid_mask(raw, fill, interleave, bands=sel)
    if valid is not None:
        _check_valid(valid, rows * cols, "fit")
    mu, g, n = _moments_sel(raw, interleave, rows, cols, B, sel, valid)
    if n < 2:
        every = [] if band_missing is None else [int(sel[k]) for k in np.flatnonzero(band_missing == rows * cols)]
        raise _lib.CmlplError(f"fit: {n} valid pixels of {rows * cols}; the moments need at least 2"
                              + (f"; bands missing in every pixel: {every}" if every else ""))
    flat = np.flatnonzero(_zero_variance(mu, np.diag(g) / n))
    if flat.size:
        raise _lib.CmlplError(f"fit: listed bands with zero variance (their z-score divides by 0): "
                              f"{[int(sel[k]) for k in flat]}; leave them out of bands= (preprocess.dead_bands)")
    return _from_moments(mu, g, n, n_PC, raw_bands=B, bands=sel)


def dead_bands(raw: torch.Tensor, fill=None, interleave: str = "bip") -> np.ndarray:
    """Raw bands no model can use: missing in every pixel (equal to ``fill``, or not finite in a float32 cube) or constant
    over the pixels that have data in all other bands (zero variance, e.g. uncalibrated zero-filled bands without a
    fill value).  -> sorted int array of raw band indices, the ones to leave out of ``fit(bands=...)``."""
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("dead_bands needs a contiguous CUDA tensor")
    rows, cols, B = raw_geometry(raw.shape, interleave)
    masked = fill is not None or raw.dtype == torch.float32
    dead = np.zeros(B, dtype=bool)
    if masked:
        dead |= valid_mask(raw, fill, interleave)[2] == rows * cols
    keep = band_list(np.flatnonzero(~dead))
    if keep.size:
        valid = valid_mask(raw, fill, interleave, bands=keep)[0] if masked else None
        mu, g, n = _moments_sel(raw, interleave, rows, cols, B, keep, valid)
        if n >= 2:
            dead[keep[_zero_variance(mu, np.diag(g) / n)]] = True
    return np.flatnonzero(dead)


def apply(raw: torch.Tensor, pp: Preproc, want_spectra: bool = True, cube: torch.Tensor | None = None,
          spectra: torch.Tensor | None = None, valid: torch.Tensor | None = None, bands=None):
    """raw CUDA [N, B] (BIP) -> (cube f32 [N, n_PC], spectra f32 [N, B] or None).  ``valid`` (u8 [N] or [rows, cols]):
    a no-data pixel is written as its band means, i.e. spectra row 0 and cube row -shift.  A ``pp`` fitted with a band
    list reads only those raw bands of ``raw`` (spectra [N, nsel]); ``bands``, when given, must be that list."""
    if not raw.is_cuda or not raw.is_contiguous():
        raise _lib.CmlplError("apply needs a contiguous CUDA tensor")
    n, B = raw.shape
    sel = pp.bands
    if bands is not None and (sel is None or not np.array_equal(band_list(bands), sel)):
        raise _lib.CmlplError("apply: bands= differs from the band list the Preproc was fitted on")
    if sel is not None and B != pp.raw_bands:
        raise _lib.CmlplError(f"apply: raw has {B} bands, the Preproc's band list is over {pp.raw_bands}")
    nf = B if sel is None else sel.size
    d = pp.device_params(raw.device)
    npc = d["Us"].shape[1]
    if cube is None:
        cube = torch.empty((n, npc), dtype=torch.float32, device=raw.device)
    if want_spectra and spectra is None:
        spectra = torch.empty((n, nf), dtype=torch.float32, device=raw.device)
    pre = (d["mu"].data_ptr(), d["inv_sigma"].data_ptr(), d["Us"].data_ptr(), d["shift"].data_ptr())
    args = (raw.data_ptr(), _dtype_code(raw), n, B, npc, *pre)
    outs = (cube.data_ptr(), spectra.data_ptr() if want_spectra else None, torch.cuda.current_stream().cuda_stream)
    if sel is not None:
        if valid is not None:
            _check_valid(valid, n, "apply")
        _lib.call("cmlpl_preprocess_apply_sel", raw.data_ptr(), _dtype_code(raw), n, B, sel.ctypes.data, sel.size, npc, *pre,
                  None if valid is None else valid.data_ptr(), *outs)
    elif valid is None:
        _lib.call("cmlpl_preprocess_apply", *args, *outs)
    else:
        _check_valid(valid, n, "apply")
        _lib.call("cmlpl_preprocess_apply_masked", *args, valid.data_ptr(), *outs)
    return cube, (spectra if want_spectra else None)
