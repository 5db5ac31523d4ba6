"""Prep / eval utilities of the reference's tools/hyper_tools.py on the B200 kernels.

Kept names and return conventions: MirrowCut, ExtractPatches, ExtractPatches_for_base,
featureNormalize, PCANorm, SampleGen, test_whole, CalAccuracy.  Patch extraction, scene
inference and the confusion matrix run in libcmlpl_sm100.so; PCA / z-scoring stay float64
numpy exactly like the reference (one-off preprocessing before the hot path, SURVEY 8f1).
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib, ops

# dataID -> (name, classes, bands).  5-7 are the WHU-Hi UAV scenes (LongKou 550 x 400, HanChuan 1217 x 303, HongHu
# 940 x 475), wider than 256 bands
DATASETS = {1: ("PaviaU", 9, 103), 2: ("Salinas", 16, 204), 3: ("Houston", 15, 144), 4: ("Indian_pines", 16, 200),
            5: ("WHU_Hi_LongKou", 9, 270), 6: ("WHU_Hi_HanChuan", 16, 274), 7: ("WHU_Hi_HongHu", 22, 270)}
# .mat file and variable names of the scene and of its ground truth (the WHU-Hi ones follow the public distribution)
_MAT = {1: ("PaviaU.mat", "paviaU", "PaviaU_gt.mat", "paviaU_gt"),
        2: ("salinas.mat", "HSI_original", "salinas_gt.mat", "Data_gt"),
        3: ("Houston.mat", "Houston", "Houston_gt.mat", "Houston_gt"),
        4: ("indian_pines_corrected.mat", "indian_pines_corrected", "indian_pines_gt.mat", "indian_pines_gt"),
        5: ("WHU_Hi_LongKou.mat", "WHU_Hi_LongKou", "WHU_Hi_LongKou_gt.mat", "WHU_Hi_LongKou_gt"),
        6: ("WHU_Hi_HanChuan.mat", "WHU_Hi_HanChuan", "WHU_Hi_HanChuan_gt.mat", "WHU_Hi_HanChuan_gt"),
        7: ("WHU_Hi_HongHu.mat", "WHU_Hi_HongHu", "WHU_Hi_HongHu_gt.mat", "WHU_Hi_HongHu_gt")}


def _device():
    _lib.require_device()
    return torch.device("cuda", torch.cuda.current_device())


# ------------------------------------------------------------------ preprocessing (host, float64)
def featureNormalize(X, type):
    """hyper_tools.py:8-22."""
    if type == 1:
        centred = X - np.mean(X, 0)
        return centred / np.std(centred, 0)
    if type == 2:
        lo, hi = np.min(X, 0), np.max(X, 0)
        return (X - lo) / (hi - lo)
    raise ValueError(f"featureNormalize: unknown type {type}")


def PCANorm(X, num_PC):
    """hyper_tools.py:25-32: project the centred data on the leading left-singular vectors of its covariance."""
    centred = X - np.mean(X, 0)
    basis = np.linalg.svd(np.cov(centred.T))[0][:, :num_PC]
    return centred @ basis


# ------------------------------------------------------------------ patches (device)
def _to_cube(X) -> torch.Tensor:
    if isinstance(X, torch.Tensor):
        return X.to(device=_device(), dtype=torch.float32).contiguous()
    # the reference assigns float64 windows into a float32 array (hyper_tools.py:233,240): the
    # cast commutes with the gather, so cast the cube once
    return torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)).to(_device())


def MirrowCut(X, hw):
    """hyper_tools.py:35-55 (== symmetric padding by hw).  Returned as float64 numpy like the reference.
    Implemented as a w=1 gather of the padded coordinate grid through the device index map of
    cmlpl_patch_gather_f32.  float64 input keeps its bits: the cube is handed to the (pure copy) kernel as
    2F float32 words per pixel and the result is viewed back as float64."""
    as_f64 = isinstance(X, np.ndarray) and X.dtype == np.float64
    if as_f64:
        Xc = np.ascontiguousarray(X)
        cube = torch.from_numpy(Xc).view(torch.float32).to(_device())          # [R, C, 2F] bit view
    else:
        cube = _to_cube(X)
    R, C, F = cube.shape
    if hw > R or hw > C:
        raise ValueError("MirrowCut: hw larger than the image")
    rr = torch.arange(-hw, R + hw, device=cube.device)
    cc = torch.arange(-hw, C + hw, device=cube.device)
    mr = torch.where(rr < 0, -rr - 1, torch.where(rr >= R, 2 * R - 1 - rr, rr))
    mc = torch.where(cc < 0, -cc - 1, torch.where(cc >= C, 2 * C - 1 - cc, cc))
    idx = (mr[:, None] * C + mc[None, :]).reshape(-1).contiguous()
    out = ops.patch_gather(cube, 1, idx=idx, odd_mode=True)          # [n, F, 1, 1]
    out = out.view(R + 2 * hw, C + 2 * hw, F)
    if as_f64:
        return out.cpu().contiguous().view(torch.float64).numpy()
    return out.cpu().numpy().astype(np.float64)


def ExtractPatches(X, w, idx=None, as_numpy=True):
    """hyper_tools.py:226-243: every pixel's w x w window (even w) -> f32 [K, F, w, w].
    ``idx`` (raster indices) restricts the gather; ``as_numpy=False`` keeps the CUDA tensor."""
    if w % 2:
        raise ValueError("ExtractPatches: could not broadcast an odd window (the reference raises too); "
                         "use ExtractPatches_for_base for odd w")
    return _extract(X, w, idx, False, as_numpy)


def ExtractPatches_for_base(X, w, idx=None, as_numpy=True):
    """hyper_tools.py:300-317: odd-w centred variant."""
    if w % 2 == 0:
        raise ValueError("ExtractPatches_for_base: w must be odd")
    return _extract(X, w, idx, True, as_numpy)


def _extract(X, w, idx, odd, as_numpy):
    cube = _to_cube(X)
    if idx is not None:
        idx = torch.as_tensor(np.asarray(idx), dtype=torch.int64).to(cube.device).contiguous()
    out = ops.patch_gather(cube, w, idx=idx, odd_mode=odd)
    return out.cpu().numpy() if as_numpy else out


def _loadmat(path):
    """scipy.io.loadmat, falling back to hdf5storage / h5py for MATLAB v7.3 (HDF5) files: the reference reads
    indian_pines_corrected.mat with hdf5storage.loadmat (hyper_tools.py:271-276) because it ships in that format."""
    import scipy.io as sio
    try:
        return sio.loadmat(path)
    except NotImplementedError:
        pass
    try:
        import hdf5storage
        return hdf5storage.loadmat(path)
    except ImportError:
        pass
    try:
        import h5py
    except ImportError as e:
        raise ImportError(f"{path} is a MATLAB v7.3 (HDF5) file: install hdf5storage or h5py to read it") from e
    with h5py.File(path, "r") as f:
        # HDF5 stores MATLAB arrays column-major: reverse the axes to get MATLAB's index order
        return {k: np.asarray(v).transpose() for k, v in f.items() if not k.startswith("#")}


def SampleGen(dataID=1, w=16, n_PC=3, root="./dataset/", as_numpy=True):
    """hyper_tools.py:246-297: load the .mat scene, PCA + z-score -> (XP, X, Y)."""
    fx, kx, fy, ky = _MAT[dataID]
    X = _loadmat(root + fx)[kx]
    Y = _loadmat(root + fy)[ky]
    row, col, n_feature = X.shape
    X = X.reshape(row * col, n_feature)
    X_PCA = featureNormalize(PCANorm(X, n_PC), 1).reshape(row, col, n_PC)
    X = featureNormalize(X, 1)
    XP = ExtractPatches(X_PCA, w, as_numpy=as_numpy)
    return XP, X, Y.reshape(row * col, )


# ------------------------------------------------------------------ inference + metrics
def test_whole(model, data_loader, print_per_batches=10):
    """hyper_tools.py:416-437: predicted label of every sample the loader yields, int64 numpy.

    When the loader wraps a cube-backed ``HSIDataSet('wholeset')`` the whole scene goes through
    the fused scene-inference kernels (patches never materialised); any other loader is consumed
    batch by batch through ``model(XP, X)`` on device like the reference."""
    model.eval()
    ds = getattr(data_loader, "dataset", None)
    if ds is not None and getattr(ds, "scene_ready", False) and ds.setindex == "wholeset":
        labels = scene_labels(model, ds.cube_device(), ds.spectra_device(), ds.w)
        return labels.cpu().numpy().astype(np.int64)
    outs = []
    num_batches = len(data_loader)
    dev = _device()
    with torch.no_grad():
        for batch_idx, data in enumerate(data_loader):
            XP, X = data[0], data[1]
            logits, _ = model(XP.to(dev, torch.float32), X.to(dev, torch.float32))
            outs.append(ops.argmax_u8(logits.contiguous()))
            if (batch_idx + 1) % print_per_batches == 0:
                print('---------------------Testing the whole set-[%d/%d]---------------------' % (
                    batch_idx + 1, num_batches))
    return torch.cat(outs).cpu().numpy().astype(np.int64)


def scene_labels(model, cube, spectra, w=20, band=None, scene_rows=None, slab_row0=0, want_logits=False):
    """Labels (uint8 CUDA tensor) of the scene rows ``band=(r0, r1)`` (default: all)."""
    R = cube.shape[0] if scene_rows is None else scene_rows
    r0, r1 = (0, R) if band is None else band
    packed = model.packed_weights(w)
    return ops.scene_infer(cube, spectra, packed, model.num_classes, w, band_row0=r0, band_rows=r1 - r0,
                           scene_rows=R, slab_row0=slab_row0, want_logits=want_logits)


class StreamedScene:
    """End-to-end scene inference from HOST buffers with the H2D copies overlapped with compute:
    the scene is cut into ``nsplit`` row bands; band k+1's cube rows (+halo) and spectra are copied on
    a side stream while band k runs through cmlpl_scene_infer on the current stream.  Device buffers,
    the workspace and the pinned label buffer are allocated once and reused across calls."""

    def __init__(self, scene_rows, cols, num_features, num_classes, w=20, nsplit=4, row0=0, rows=None, device=None):
        self.R, self.C, self.B, self.K, self.w = scene_rows, cols, num_features, num_classes, w
        self.r0 = row0
        self.r1 = scene_rows if rows is None else row0 + rows
        dev = _device() if device is None else device
        n = (self.r1 - self.r0) * cols
        lo = w // 2
        self.s0 = max(0, self.r0 - lo)
        self.s1 = min(scene_rows, self.r1 + (w - lo - 1))
        # mirrored halo rows at true scene edges always lie inside [s0, s1) because hw <= band rows here
        self.cube = torch.empty((self.s1 - self.s0, cols, 60), dtype=torch.float32, device=dev)
        self.spectra = torch.empty((n, num_features), dtype=torch.float32, device=dev)
        self.labels = torch.empty((n,), dtype=torch.uint8, device=dev)
        self.labels_host = torch.empty((n,), dtype=torch.uint8).pin_memory()
        per = -(-(self.r1 - self.r0) // nsplit)
        self.bands = [(a, min(a + per, self.r1)) for a in range(self.r0, self.r1, per)]
        self.ws = ops.scene_workspace(per, cols, num_features, num_classes, w, dev)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.events = [torch.cuda.Event() for _ in self.bands]
        self.done = torch.cuda.Event()
        self.d2h_done = torch.cuda.Event()

    def __call__(self, packed, cube_host, spectra_host, d2h=True):
        """cube_host f32 [s1-s0, C, 60] (pinned; slab rows s0..s1 of the scene), spectra_host f32
        [n, B] (pinned).  Returns the uint8 labels (pinned host tensor if d2h else the CUDA tensor)."""
        main = torch.cuda.current_stream()
        lo, C = self.w // 2, self.C
        self.copy_stream.wait_event(self.done)          # previous call's compute has consumed the buffers
        copied = self.s0
        with torch.cuda.stream(self.copy_stream):
            for (a, b), ev in zip(self.bands, self.events):
                upto = min(self.s1, b + (self.w - lo - 1))
                if upto > copied:
                    self.cube[copied - self.s0:upto - self.s0].copy_(cube_host[copied - self.s0:upto - self.s0], non_blocking=True)
                    copied = upto
                pa, pb = (a - self.r0) * C, (b - self.r0) * C
                self.spectra[pa:pb].copy_(spectra_host[pa:pb], non_blocking=True)
                ev.record(self.copy_stream)
        for (a, b), ev in zip(self.bands, self.events):
            main.wait_event(ev)
            pa, pb = (a - self.r0) * C, (b - self.r0) * C
            ops.scene_infer(self.cube, self.spectra[pa:pb], packed, self.K, self.w, band_row0=a, band_rows=b - a,
                            scene_rows=self.R, slab_row0=self.s0, workspace=self.ws, labels=self.labels[pa:pb])
        self.done.record(main)
        if not d2h:
            return self.labels
        self.labels_host.copy_(self.labels, non_blocking=True)
        self.d2h_done.record(main)
        return self.labels_host

    def wait(self):
        """Block the host until the labels of the last call have landed in ``labels_host`` (the D2H copy is
        asynchronous: read the returned pinned tensor only after this, or after synchronising the stream)."""
        self.d2h_done.synchronize()
        return self.labels_host


class StreamedRawScene:
    """Like StreamedScene, but from the RAW cube (uint16 / float32 / int16, pinned host memory) and a fitted
    ``cmlpl_b200.preprocess.Preproc``: each band's raw rows are copied on a side stream and fed
    to cmlpl_scene_infer_raw, whose first kernels apply the preprocessing folded into conv0 / the fp16
    conversion of the spectra (``folded=`` from Preproc.folded_conv0; nothing preprocessed touches HBM) --
    42.7 MB over PCIe for a PaviaU scene instead of 135 MB.  Without ``folded`` the rows go through
    cmlpl_preprocess_apply + cmlpl_scene_infer (materialised PCA cube / spectra; BIP only).  Two sets of device
    buffers alternate between calls, so the copies of the next scene overlap the compute of the current one
    when calls are issued back to back.

    ``interleave`` is the host cube's layout, kept on the device: "bip" [(s1-s0)*cols, B], "bil" [s1-s0, B, cols]
    (a row band is contiguous) or "bsq" [B, s1-s0, cols] (a row band is B plane segments, moved by one 2-D copy).
    ``h2d_bytes`` is the number of bytes the last call copied to the device.

    ``fill`` (a value of the sample type; NaN for float32 = non-finite samples only): the cube has no-data pixels.  The
    slab's validity mask is built on the device from the rows each copy brought (BSQ: from the whole slab once its last
    rows have landed, since a BSQ row band is not a cube of its own), so nothing more crosses PCIe; the calls run
    cmlpl_scene_infer_raw_masked and need ``folded=``.  No-data pixels get ops.NODATA_LABEL.

    A ``preproc`` fitted with ``bands`` (``num_features`` = the host cube's band count, its ``raw_bands``) makes every call
    read only those bands, and the model sees len(bands) features.  A BSQ cube copies only the listed planes, one 2-D copy
    per run of consecutive bands (``h2d_bytes`` shrinks to nsel / B of the whole); BIP and BIL copy whole rows and the
    kernels select the bands on the device."""

    def __init__(self, preproc, scene_rows, cols, num_features, num_classes, w=20, nsplit=2, row0=0, rows=None,
                 raw_dtype=torch.uint16, device=None, interleave="bip", fill=None):
        from .. import preprocess
        self._pp_mod, self.pp = preprocess, preproc
        self.R, self.C, self.B, self.K, self.w = scene_rows, cols, num_features, num_classes, w
        self.sel = None if preproc is None else preproc.bands
        if self.sel is not None and preproc.raw_bands != num_features:
            raise _lib.CmlplError(f"StreamedRawScene: the Preproc's band list selects from {preproc.raw_bands} bands, the "
                                  f"cube has num_features = {num_features}")
        self.nf = num_features if self.sel is None else self.sel.size          # the model's features
        self.r0 = row0
        self.r1 = scene_rows if rows is None else row0 + rows
        dev = _device() if device is None else device
        lo = w // 2
        self.s0 = max(0, self.r0 - lo)
        self.s1 = min(scene_rows, self.r1 + (w - lo - 1))
        ns = (self.s1 - self.s0) * cols
        n = (self.r1 - self.r0) * cols
        self._ns, self._dev = ns, dev
        sr = self.s1 - self.s0
        shape = {"bip": (ns, num_features), "bil": (sr, num_features, cols), "bsq": (num_features, sr, cols)}
        if interleave not in shape:
            raise _lib.CmlplError(f"interleave must be one of {sorted(shape)}, got {interleave!r}")
        self.interleave, self.h2d_bytes, self.fill = interleave, 0, fill
        self.host_shape = shape[interleave]
        # BSQ with a band list: the device slab holds the listed planes only, copied as runs (first raw band, first slab
        # plane, count) of consecutive bands; the kernels then read all of its planes
        sel = np.arange(num_features) if self.sel is None else self.sel
        self.runs = [(int(r[0]), int(np.searchsorted(sel, r[0])), len(r))
                     for r in np.split(sel, np.flatnonzero(np.diff(sel) != 1) + 1)]
        self.compact = interleave == "bsq" and self.sel is not None
        if self.compact:
            shape["bsq"] = (self.nf, sr, cols)
        if fill is not None:
            preprocess._fill_value(torch.empty(0, dtype=raw_dtype), fill)        # an integer cube needs a fill value
        self.sets = [dict(raw=torch.empty(shape[interleave], dtype=raw_dtype, device=dev), cube=None, spectra=None,
                          valid=torch.empty((sr, cols), dtype=torch.uint8, device=dev) if fill is not None else None,
                          counts=torch.empty(self.nf + 1, dtype=torch.int64, device=dev),
                          labels=torch.empty((n,), dtype=torch.uint8, device=dev),
                          labels_host=torch.empty((n,), dtype=torch.uint8).pin_memory(),
                          done=torch.cuda.Event()) for _ in range(2)]
        per = -(-(self.r1 - self.r0) // nsplit)
        self.bands = [(a, min(a + per, self.r1)) for a in range(self.r0, self.r1, per)]
        self.ws = ops.scene_workspace(per, cols, self.nf, num_classes, w, dev)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.events = [[torch.cuda.Event() for _ in self.bands] for _ in range(2)]
        self.calls = 0

    @property
    def labels_host(self):
        return self.sets[(self.calls - 1) & 1]["labels_host"]

    def __call__(self, packed, raw_host, d2h=True, folded=None):
        """raw_host pinned: raw rows s0..s1 of the scene in the layout of ``interleave`` ([(s1-s0)*cols, B] for BIP).
        Returns uint8 labels of the band (the pinned host tensor of this call's buffer set when d2h, else the CUDA
        tensor).  The D2H copy is asynchronous: call ``wait()`` (or synchronise the stream) before reading the pinned
        tensor."""
        il = self.interleave
        if folded is None and il != "bip":
            raise _lib.CmlplError(f"StreamedRawScene: a {il.upper()} cube needs folded= (preprocess.apply reads BIP)")
        if folded is None and self.fill is not None:
            raise _lib.CmlplError("StreamedRawScene: a cube with a fill value needs folded= (cmlpl_scene_infer_raw_masked)")
        want = self.sets[0]["raw"]
        if il != "bip" and (tuple(raw_host.shape) != self.host_shape or raw_host.dtype != want.dtype
                            or not raw_host.is_contiguous()):
            raise _lib.CmlplError(f"StreamedRawScene: raw_host must be contiguous {want.dtype} {list(self.host_shape)}, "
                                  f"got {raw_host.dtype} {list(raw_host.shape)}")
        if folded is not None:
            fb = folded.get("bands")
            if (fb is None) != (self.sel is None) or (fb is not None and not np.array_equal(fb, self.sel)):
                raise _lib.CmlplError("StreamedRawScene: folded= has another band list than the Preproc")
            if self.compact:                                  # the device planes are the listed bands
                folded = dict(folded, bands=None, raw_bands=self.nf)
        main = torch.cuda.current_stream()
        S, events = self.sets[self.calls & 1], self.events[self.calls & 1]
        self.calls += 1
        if folded is None and S["cube"] is None:
            S["cube"] = torch.empty((self.s1 - self.s0, self.C, 60), dtype=torch.float32, device=self._dev)
            S["spectra"] = torch.empty((self._ns, self.nf), dtype=torch.float32, device=self._dev)
        lo, C = self.w // 2, self.C
        self.copy_stream.wait_event(S["done"])               # the call two scenes ago has consumed this set
        copied, spans, raw = self.s0, [], S["raw"]
        esz, sr = raw.element_size(), self.s1 - self.s0
        self.h2d_bytes = 0
        with torch.cuda.stream(self.copy_stream):
            for (a, b), ev in zip(self.bands, events):
                upto = min(self.s1, b + (self.w - lo - 1))
                spans.append((copied, upto))
                if upto > copied:
                    ra, rb = copied - self.s0, upto - self.s0
                    if il == "bsq":                           # rows ra..rb of each (listed) plane, a 2-D copy per run
                        pitch, off, width = sr * C * esz, ra * C * esz, (rb - ra) * C * esz
                        for b0, k0, cnt in self.runs:
                            _lib.call("cmlpl_memcpy2d_async", raw.data_ptr() + k0 * pitch + off, pitch,
                                      raw_host.data_ptr() + b0 * pitch + off, pitch, width, cnt,
                                      self.copy_stream.cuda_stream)
                            self.h2d_bytes += width * cnt
                    else:                                     # BIP pixels of rows ra..rb, or BIL rows ra..rb: one block
                        src = raw_host[ra * C:rb * C] if il == "bip" else raw_host[ra:rb]
                        (raw[ra * C:rb * C] if il == "bip" else raw[ra:rb]).copy_(src, non_blocking=True)
                        self.h2d_bytes += src.nbytes
                    copied = upto
                ev.record(self.copy_stream)
        for i, ((a, b), ev, (c0, c1)) in enumerate(zip(self.bands, events, spans)):
            main.wait_event(ev)
            qa, qb = (a - self.r0) * C, (b - self.r0) * C
            if self.fill is not None:                         # the validity of the rows that just arrived
                ra, rb = c0 - self.s0, c1 - self.s0
                if il == "bsq" and i == 0:
                    main.wait_event(events[-1])
                    self._pp_mod.mask_into(raw, self.fill, il, sr, C, raw.shape[0], S["valid"], S["counts"],
                                           None if self.compact else self.sel)
                elif il != "bsq" and rb > ra:
                    rows = raw[ra * C:rb * C] if il == "bip" else raw[ra:rb]
                    self._pp_mod.mask_into(rows, self.fill, il, rb - ra, C, self.B, S["valid"][ra:rb], S["counts"],
                                           self.sel)
            if folded is not None:
                ops.scene_infer_raw(S["raw"], folded, packed, self.K, C, self.w, band_row0=a, band_rows=b - a,
                                    scene_rows=self.R, slab_row0=self.s0, workspace=self.ws, labels=S["labels"][qa:qb],
                                    interleave=il, valid=S["valid"])
                continue
            if c1 > c0:                                       # preprocess the rows that just arrived
                pa, pb = (c0 - self.s0) * C, (c1 - self.s0) * C
                self._pp_mod.apply(S["raw"][pa:pb], self.pp, cube=S["cube"].view(-1, 60)[pa:pb], spectra=S["spectra"][pa:pb])
            sa = (a - self.s0) * C
            ops.scene_infer(S["cube"], S["spectra"][sa:sa + (b - a) * C], packed, self.K, self.w, band_row0=a,
                            band_rows=b - a, scene_rows=self.R, slab_row0=self.s0, workspace=self.ws,
                            labels=S["labels"][qa:qb])
        if d2h:
            S["labels_host"].copy_(S["labels"], non_blocking=True)
        S["done"].record(main)                                # after the D2H copy: also the "labels landed" event
        return S["labels_host"] if d2h else S["labels"]

    def wait(self):
        """Block the host until the last call's labels have landed in its pinned buffer and return it (the D2H
        copy is asynchronous: read the tensor ``__call__`` returned only after this or a stream synchronise)."""
        S = self.sets[(self.calls - 1) & 1]
        S["done"].synchronize()
        return S["labels_host"]


def confusion_matrix(predict, label, num_classes):
    """int64 [C, C] counts cm[label, predict] computed on device."""
    dev = _device()
    p = torch.as_tensor(np.asarray(predict)).to(dev)
    if p.dtype != torch.uint8:
        if p.numel() and (int(p.min()) < 0 or int(p.max()) > 255):
            raise ValueError("predictions must lie in [0, 255]")
        p = p.to(torch.uint8)
    l = torch.as_tensor(np.asarray(label)).to(dev).to(torch.int64)
    return ops.confusion(p.contiguous(), l.contiguous(), num_classes).cpu().numpy()


def CalAccuracy(predict, label):
    """hyper_tools.py:208-223 -> (OA, Kappa, producerA[C]) with C = max(label)+1.

    Counts come from the device confusion matrix (sized to also hold predictions above
    max(label), which the reference counts in ``reali`` but in no per-class hit); the ratios are
    formed in float64 on the host in the reference's order of operations."""
    label = np.asarray(label)
    predict = np.asarray(predict)
    n = label.shape[0]
    C = int(label.max()) + 1
    full = max(C, int(predict.max()) + 1)
    cm = confusion_matrix(predict, label, full).astype(np.float64)
    correct_sum = np.diag(cm)[:C].copy()
    reali = cm.sum(1)[:C]
    predicti = cm.sum(0)[:C]
    OA = np.trace(cm) * 1.0 / n
    with np.errstate(divide="ignore", invalid="ignore"):
        producerA = correct_sum / reali
    Kappa = (n * np.sum(correct_sum) - np.sum(reali * predicti)) * 1.0 / (n * n - np.sum(reali * predicti))
    return OA, Kappa, producerA
