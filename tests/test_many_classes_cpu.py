"""Host arithmetic of the 17-32-class scene path (no GPU): the packed-weight size and the scene workspace layout.

Up to 16 classes both must stay byte for byte what they were before the tensor-core path took 32-class widths; the
expected values below were recorded from that build.  17-32 classes take the dense path (class width NC = 32), and 33 or
more never do."""
import ctypes

import pytest

from cmlpl_b200 import _lib

# (B, C, w) -> cmlpl_packed_bytes
PACKED_16 = {
    (103, 9, 20): 1048832, (200, 16, 20): 1716224, (224, 16, 20): 1847296, (48, 1, 11): 560128,
    (103, 16, 11): 993280, (240, 16, 20): 1945600, (144, 15, 20): 1345280, (103, 5, 11): 936960,
}
# (path mode, (rows, cols, B, C, w)) -> offsets[12] of cmlpl_scene_workspace_layout
LAYOUT_16 = {
    (1, (610, 340, 103, 9, 20)): [0, 28903936, 75381248, 128498176, 128498176, 389771776, 651045376, 0, 0, 0, 723621376, 1],
    (1, (64, 257, 224, 16, 20)): [0, 2932224, 10329600, 14556672, 14556672, 41264640, 67972608, 0, 0, 0, 75391488, 1],
    (1, (37, 45, 200, 16, 11)): [0, 331008, 1076480, 1535232, 1535232, 4631808, 7728384, 0, 0, 0, 8588544, 1],
    (1, (10, 10, 240, 16, 20)): [0, 0, 0, 0, 0, 0, 0, 107776, 427776, 434176, 843776, 0],
    (1, (349, 1905, 144, 15, 20)): [0, 90628096, 282136576, 452366336, 452366336, 1268019200, 2083672064, 0, 0, 0,
                                   2310242304, 1],
    (1, (1, 13, 48, 3, 11)): [0, 32512, 44800, 77568, 77568, 409344, 741120, 0, 0, 0, 833280, 1],
    (0, (610, 340, 103, 9, 20)): [0, 28903936, 75381248, 0, 0, 0, 0, 128498176, 0, 0, 792178176, 0],
    (0, (64, 257, 224, 16, 20)): [0, 2932224, 10329600, 0, 0, 0, 0, 14556672, 0, 0, 67190272, 0],
    (0, (37, 45, 200, 16, 11)): [0, 331008, 1076480, 0, 0, 0, 0, 1535232, 0, 0, 2387712, 0],
    (0, (10, 10, 240, 16, 20)): [0, 0, 0, 0, 0, 0, 0, 107776, 427776, 434176, 843776, 0],
    (0, (349, 1905, 144, 15, 20)): [0, 90628096, 282136576, 0, 0, 0, 0, 452366336, 0, 0, 2579870464, 0],
    (0, (1, 13, 48, 3, 11)): [0, 32512, 44800, 0, 0, 0, 0, 77568, 0, 0, 84224, 0],
}
NAMES = ["f0pad", "x16", "h16", "g", "pm", "yq", "lmap", "p2", "spe", "hidden", "total", "dense"]


def _layout(mode, R, C, B, K, w):
    lib = _lib.load()
    off = (ctypes.c_size_t * 12)()
    _lib.call("cmlpl_set_scene_path_mode", mode)
    try:
        _lib.call("cmlpl_scene_workspace_layout", R, C, B, K, w, off)
        total = lib.cmlpl_scene_workspace_bytes(R, C, B, K, w)
    finally:
        _lib.call("cmlpl_set_scene_path_mode", 1)
    assert total == off[10]
    return dict(zip(NAMES, list(off)))


@pytest.mark.parametrize("shape", sorted(PACKED_16))
def test_packed_bytes_unchanged_up_to_16_classes(shape):
    assert _lib.load().cmlpl_packed_bytes(*shape) == PACKED_16[shape]


@pytest.mark.parametrize("key", sorted(LAYOUT_16))
def test_workspace_layout_unchanged_up_to_16_classes(key):
    mode, shape = key
    got = _layout(mode, *shape)
    assert [got[k] for k in NAMES] == LAYOUT_16[key]


@pytest.mark.parametrize("B,w", [(103, 20), (224, 20), (48, 11)])
def test_packed_bytes_grow_only_past_16_classes(B, w):
    lib = _lib.load()
    b16 = lib.cmlpl_packed_bytes(B, 16, w)
    assert lib.cmlpl_packed_bytes(B, 9, w) <= b16
    P = (w // 4) ** 2
    # wc16 and wcq take a class stride of 32: exactly one more copy of each, plus the wider f32 classifier columns
    grow = (P * 8 + 128) * 16 * 16 + 25 * 16 * 128
    for C in (17, 20, 32):
        got = lib.cmlpl_packed_bytes(B, C, w)
        assert got - b16 >= grow


@pytest.mark.parametrize("B,C,w", [(48, 20, 20), (103, 17, 20), (224, 32, 20), (103, 20, 11), (224, 32, 11)])
def test_dense_path_for_17_to_32_classes(B, C, w):
    R, cols = 61, 83
    n, mt = R * cols, (R * cols + 127) // 128
    qpos = 4 * ((R + w) // 2) * ((cols + w) // 2)
    d = _layout(1, R, cols, B, C, w)
    assert d["dense"] == 1
    assert d["h16"] - d["x16"] >= mt * ((B + 15) // 16) * 2 * 2048
    assert d["pm"] - d["h16"] >= 4 * mt * 128 * 32 * 4            # partial spectral logits [4][mtiles*128][32]
    assert d["total"] - d["lmap"] >= qpos * 5 * 32 * 4               # lmap [4][5][8 quads][PR2][PC2][4]
    # path mode 0 keeps the CUDA-core spectral head for the cube and the tensor-core one for the raw entry point
    z = _layout(0, R, cols, B, C, w)
    assert z["dense"] == 0 and z["lmap"] == 0
    assert z["h16"] > z["x16"] > 0 and z["p2"] > z["h16"]
    assert z["spe"] - z["p2"] >= n * (w // 4) ** 2 * 64 * 2 and z["hidden"] > z["spe"]


@pytest.mark.parametrize("B,C", [(103, 33), (103, 40), (240, 20)])
def test_no_dense_path_past_32_classes_or_224_bands(B, C):
    d = _layout(1, 40, 50, B, C, 20)
    assert d["dense"] == 0 and d["x16"] == 0 and d["h16"] == 0 and d["lmap"] == 0
    assert d["spe"] > d["p2"] > 0
