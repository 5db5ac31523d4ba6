"""Host side of w = 11 training (no GPU): the fused step's workspace, its window check, and the dataset's host items.

A w = 11 step runs in the w = 20 workspace at the same region offsets, so the w = 20 sizes and offsets must stay byte
for byte what they were before the w = 11 instantiations existed; the expected values below were recorded from that
build."""
import ctypes

import numpy as np
import pytest

from cmlpl_b200 import _lib
from oracle import cmlpl_oracle as O

# (bs, btu, bands, classes, queue) -> cmlpl_train_workspace_layout offsets[20] (the last one is the total size)
LAYOUT_W20 = {
    (128, 128, 103, 9, 1280): [0, 26214400, 52428800, 58982400, 60620800, 61030400, 66404352, 71778304, 71989248,
                               71991296, 72009728, 73058304, 78432256, 80529408, 106743808, 132958208, 133634048,
                               133699584, 133765120, 134953984],
    (128, 128, 224, 16, 1280): [0, 26214400, 52428800, 58982400, 60620800, 61030400, 66404352, 71778304, 72237056,
                                72239104, 72271872, 73320448, 78694400, 80791552, 107005952, 133220352, 133896192,
                                133961728, 134027264, 135223296],
    (5, 7, 7, 2, 1280): [0, 1228800, 2457600, 2764800, 2841600, 2860800, 3112704, 3364608, 3365376, 3365632, 3365888,
                         3423232, 3675136, 3773440, 5002240, 6231040, 6268160, 6268416, 6268672, 7448576],
    (100, 100, 103, 9, 1000): [0, 20480000, 40960000, 46080000, 47360000, 47680000, 51878400, 56076800, 56241664,
                               56243456, 56258048, 57077248, 61275648, 62914048, 83394048, 103874048, 104296448,
                               104336640, 104376832, 105563904],
    (64, 192, 103, 9, 1280): [0, 26214400, 52428800, 58982400, 60620800, 61030400, 66404352, 71778304, 71989248,
                              71991296, 72009728, 73582592, 78956544, 81053696, 107268096, 133482496, 134496256,
                              134643712, 134791168, 135984640],
}
WS_FIELDS = ("x16", "a0", "p1", "m1", "m2", "cat", "dmask", "ynoisy", "norm", "dlogits", "dfeat", "dcat", "dhp",
             "dz1", "da0", "S", "G", "dG", "probs_orig", "total")
# per-sample bytes of the w = 11 regions (include/cmlpl.h), and the cat row width
W11_STRIDES = {"x16": 8 * 121 * 16, "a0": 8 * 121 * 16, "dz1": 8 * 121 * 16, "da0": 8 * 121 * 16, "p1": 8 * 25 * 16,
               "m1": 121 * 8, "m2": 25 * 8, "cat": 1280 * 4, "dmask": 1280 * 4, "dcat": 1280 * 4}


@pytest.mark.parametrize("dims", list(LAYOUT_W20))
def test_train_workspace_w20_unchanged_and_bounds_w11(dims):
    lib = _lib.load()
    off = (ctypes.c_size_t * 20)()
    _lib.call("cmlpl_train_workspace_layout", *dims, off)
    assert list(off) == LAYOUT_W20[dims]
    assert lib.cmlpl_train_workspace_bytes(*dims) == LAYOUT_W20[dims][-1]
    # every w = 11 region, packed at its own per-sample stride, ends before the next region starts
    ns = 2 * (dims[0] + dims[1])
    at = dict(zip(WS_FIELDS, off))
    order = sorted(WS_FIELDS, key=lambda k: at[k])
    for k, stride in W11_STRIDES.items():
        nxt = order[order.index(k) + 1]
        assert at[k] + ns * stride <= at[nxt], k


def test_train_step_refuses_other_windows():
    """The window check comes before any device work: w = 13 fails with a message naming both supported windows."""
    from cmlpl_b200.fused_step import TrainIO
    io = TrainIO()
    io.bs, io.btu, io.bands, io.classes, io.w, io.queue = 4, 4, 8, 3, 13, 64
    with pytest.raises(_lib.CmlplError, match=r"w=13 unsupported \(20 .*11"):
        _lib.call("cmlpl_train_step", ctypes.byref(io), 15, None)


def _write_dataset(root, R, C, w, nf=60, B=7, seed=0):
    rng = np.random.default_rng(seed)
    np.save(root + "XPCA.npy", rng.standard_normal((R, C, nf)).astype(np.float32))
    np.save(root + "meta.npy", np.array([w, R, C], dtype=np.int64))
    np.save(root + "X.npy", rng.standard_normal((R * C, B)))
    np.save(root + "Y.npy", rng.integers(1, 4, R * C))
    idx = rng.permutation(R * C)
    np.save(root + "train_array.npy", idx[:40])
    np.save(root + "test_array.npy", idx[40:])
    np.save(root + "unlabel_array.npy", idx[40:])


@pytest.mark.parametrize("w", [11, 5, 20])
def test_hsi_dataset_host_items_match_the_oracle_windows(tmp_path, w):
    """HSIDataSet.__getitem__ (the DataLoader path, no device): odd w takes ExtractPatches_for_base's window, rows and
    columns r-(w-1)/2 .. r+(w-1)/2 mirrored at the scene edges -- the window the device gather uses with odd_mode --
    and even w ExtractPatches' window, as before.  Pixels on every edge and corner are included."""
    from cmlpl_b200.hsi_loader import HSIDataSet
    root = str(tmp_path) + "/"
    R, C = 13, 17
    _write_dataset(root, R, C, w)
    cube = np.load(root + "XPCA.npy")
    ds = HSIDataSet(1, "wholeset", root=root)
    assert ds.w == w
    pix = np.array([0, C - 1, (R - 1) * C, R * C - 1, 2 * C + 3, 6 * C + 8, C * 4, 5 * C + C - 2])
    want = O.extract_patches_at(cube, w, pix, odd_mode=w % 2 == 1)
    for i, p in enumerate(pix):
        XP, X = ds[int(p)]
        assert XP.shape == (60, w, w) and XP.dtype == np.float32
        assert np.array_equal(XP, want[i]), p
        assert np.array_equal(X, ds.X[p].astype(np.float32))
