"""``HSIDataSet`` of the reference's hsi_loader.py, backed by the scene cube.

Same constructor, ``__len__`` and ``__getitem__`` tuples (hsi_loader.py:5-56,109-133) and the same
./dataset/<Name>/ file contract, except that the 19.9 GB ``XP.npy`` is optional: the dataset keeps
the PCA cube ``XPCA.npy`` f32 [R,C,n_PC] (49.8 MB for PaviaU) plus the index arrays and produces a
sample's patch on demand.  ``gather(indices)`` gives a whole batch on the GPU through the
patch-gather kernel; ``test_whole`` runs a 'wholeset' instance through the fused scene kernels.
"""
from __future__ import annotations

import os

import numpy as np
import torch
from torch.utils import data

ROOTS = {1: "./dataset/PaviaU/", 2: "./dataset/Salinas/", 3: "./dataset/Houston/", 4: "./dataset/Indian_pines/",
         5: "./dataset/WHU_Hi_LongKou/", 6: "./dataset/WHU_Hi_HanChuan/", 7: "./dataset/WHU_Hi_HongHu/"}


def _tile(arr, max_iters):
    """hsi_loader.py:29-34: whole repeats of the split followed by its head, max_iters rows in all."""
    whole = int(max_iters / len(arr))
    head = max_iters - whole * len(arr)
    return np.concatenate((np.tile(arr, whole), arr[:head]))


class HSIDataSet(data.Dataset):
    def __init__(self, dataID, setindex='label', max_iters=None, num_unlabel=1000, root=None, w=None):
        self.setindex = setindex
        try:
            dataID = int(dataID)            # train.py:357 declares --dataID as str
        except (TypeError, ValueError):
            pass
        self.root = root if root is not None else ROOTS[dataID]
        self.X = np.load(self.root + 'X.npy')                       # f64 [N, B]   (hsi_loader.py:21)
        self.Yall = np.load(self.root + 'Y.npy') - 1                # 0-based, background wraps (hsi_loader.py:22)
        self.scene_ready = os.path.exists(self.root + 'XPCA.npy')
        if self.scene_ready:
            self.cube = np.load(self.root + 'XPCA.npy')             # f32 [R, C, n_PC]
            meta = np.load(self.root + 'meta.npy') if os.path.exists(self.root + 'meta.npy') else None
            self.w = int(w if w is not None else (meta[0] if meta is not None else 20))
            self.XP = None
        else:
            self.XP = np.load(self.root + 'XP.npy', mmap_mode='r')   # reference layout f32 [N, F, w, w]
            self.w = self.XP.shape[-1]
        n_all = self.X.shape[0]
        if setindex == 'label':
            index = np.load(self.root + 'train_array.npy')
            if max_iters is not None:
                index = _tile(index, max_iters)
        elif setindex == 'unlabel':
            index = np.load(self.root + 'unlabel_array.npy')[0:num_unlabel]
            if max_iters is not None:
                index = _tile(index, max_iters)
        elif setindex == 'test':
            index = np.load(self.root + 'test_array.npy')
        elif setindex == 'wholeset':
            index = np.arange(n_all)
        else:
            raise ValueError(f"unknown setindex {setindex!r}")
        self.index = np.asarray(index, dtype=np.int64)
        self._dev = {}

    def __len__(self):
        return len(self.index)

    # ---- host-side single sample (DataLoader contract of the reference)
    def _patch_host(self, pix):
        if self.XP is not None:
            return np.asarray(self.XP[pix], dtype=np.float32)
        R, C, _ = self.cube.shape
        w, hw = self.w, self.w // 2
        r, c = divmod(int(pix), C)
        rr = np.arange(r - hw, r - hw + w)
        cc = np.arange(c - hw, c - hw + w)
        rr = np.where(rr < 0, -rr - 1, np.where(rr >= R, 2 * R - 1 - rr, rr))
        cc = np.where(cc < 0, -cc - 1, np.where(cc >= C, 2 * C - 1 - cc, cc))
        return np.ascontiguousarray(np.moveaxis(self.cube[rr[:, None], cc[None, :], :], 2, 0), dtype=np.float32)

    def __getitem__(self, index):
        pix = self.index[index]
        XP = self._patch_host(pix)
        X = self.X[pix].astype('float32')
        if self.setindex == 'wholeset':
            return XP.copy(), X.copy()
        return XP.copy(), X.copy(), self.Yall[pix].astype('int')

    # ---- device-side batch path (what cmlpl_b200.train uses)
    def cube_device(self):
        from . import _lib
        _lib.require_device()
        if not self.scene_ready:
            raise RuntimeError("this dataset directory has no XPCA.npy (run cmlpl_b200.sample_generation)")
        if 'cube' not in self._dev:
            self._dev['cube'] = torch.from_numpy(np.ascontiguousarray(self.cube, dtype=np.float32)).cuda()
        return self._dev['cube']

    def spectra_device(self):
        if 'X' not in self._dev:
            self._dev['X'] = torch.from_numpy(self.X[self.index].astype(np.float32)).cuda()
        return self._dev['X']

    def labels_device(self):
        if 'Y' not in self._dev:
            self._dev['Y'] = torch.from_numpy(self.Yall[self.index].astype(np.int64)).cuda()
        return self._dev['Y']

    def gather(self, positions: torch.Tensor, noise=None, noise_scale=0.0):
        """Batch for dataset positions (CUDA int64) -> (XP f32 [b,F,w,w], X f32 [b,B], Y i64 [b])."""
        from . import ops
        if 'pix' not in self._dev:
            self._dev['pix'] = torch.from_numpy(self.index).cuda()
        pix = self._dev['pix'][positions].contiguous()
        # odd w: ExtractPatches_for_base (hyper_tools.py:300-317), the window the odd-w scene path and model use
        XP = ops.patch_gather(self.cube_device(), self.w, idx=pix, noise=noise, noise_scale=noise_scale,
                              odd_mode=self.w % 2 == 1)
        return XP, self.spectra_device()[positions], self.labels_device()[positions]
