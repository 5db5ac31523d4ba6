"""Band selection without a GPU: every band-list rejection of the four *_sel entry points returns CMLPL_ERR_ARG with its
own message before any CUDA call, a valid list passes every check and fails only at its first CUDA call, the workspace of
196 of 242 bands is the dense 196-band one, ops.scene_infer_raw refuses a cube whose band count differs from the fit's,
and the new symbols are declared.

The entry points run in a child process in which no CUDA device is visible, with fake device pointers (as in
tests/test_wide_bands_cpu.py)."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CMLPL_ERR_ARG = -1
GiB = 1 << 30

# Runs one *_sel entry point per case from stdin and prints {case id: [return code, cmlpl_last_error()]}.
CHILD = r"""
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from cmlpl_b200 import _lib
lib = _lib.load()
GiB = 1 << 30
out = {}
for c in json.load(sys.stdin):
    B, sel = c["B"], c["bands"]
    arr = (ctypes.c_int * max(len(sel), 1))(*sel)
    lst = None if c.get("null") else arr
    e = c["entry"]
    if e == "scene":
        R, C = 30, 40
        rc = lib.cmlpl_scene_infer_raw_sel(1 * GiB, c.get("dtype", 0), R, C, 0, R, B, lst, len(sel), 16, c.get("w", 20), 0, R,
                                           3 * GiB, 4 * GiB, 5 * GiB, 6 * GiB, None, 7 * GiB, 8 * GiB, 1 << 40, 9 * GiB,
                                           None, None)
    elif e == "mask":
        rc = lib.cmlpl_valid_mask_sel_u8(1 * GiB, 0x10, 30, 40, B, lst, len(sel), 0.0, 2 * GiB, 3 * GiB, 4 * GiB, None)
    elif e == "fit":
        rc = lib.cmlpl_preprocess_fit_sel_f64(1 * GiB, 0x20, 30, 40, B, lst, len(sel), None, 2 * GiB, 3 * GiB, None, None)
    else:
        rc = lib.cmlpl_preprocess_apply_sel(1 * GiB, 0, 1200, B, lst, len(sel), 60, 2 * GiB, 3 * GiB, 4 * GiB, 5 * GiB, None,
                                            6 * GiB, 7 * GiB, None)
    out[c["id"]] = [rc, lib.cmlpl_last_error().decode()]
print(json.dumps(out))
"""

HYPERION_GOOD = [b for b in range(242) if not (b < 8 or 57 <= b < 77 or 224 <= b < 242)]     # 196 of 242
FN = {"scene": "scene_infer_raw_sel", "mask": "valid_mask_sel", "fit": "preprocess_fit_sel", "apply": "preprocess_apply_sel"}
BAD = {
    "unsorted": (242, [5, 3, 9], "band list not strictly increasing at entry 1 (3 after 5)"),
    "duplicate": (242, [5, 7, 7, 9], "band list not strictly increasing at entry 2 (7 after 7)"),
    "above": (242, [5, 242], "band list entry 1 = 242 outside [0, 242)"),
    "negative": (242, [-1, 4], "band list entry 0 = -1 outside [0, 242)"),
    "empty": (242, [], "empty band list"),
    "null": (242, [1, 2], "null band list"),
    "raw_bands": (8193, [1, 2], "raw band count 8193 outside 1..8192"),
}
CASES = [dict(id=f"{e}/{k}", entry=e, B=B, bands=b, null=k == "null") for e in FN for k, (B, b, _) in BAD.items()]
CASES += [dict(id="scene/513", entry="scene", B=600, bands=list(range(513)))]
CASES += [dict(id="apply/1025", entry="apply", B=2000, bands=list(range(1025)))]
CASES += [dict(id=f"scene/ok/{dt}/{w}", entry="scene", B=242, bands=HYPERION_GOOD, dtype=dt, w=w)
          for dt in (0x00, 0x12, 0x21) for w in (20, 11)]
CASES += [dict(id="scene/ok/wide", entry="scene", B=425, bands=sorted(set(range(0, 425, 2)) | set(range(1, 175, 2))))]
CASES += [dict(id=f"{e}/ok", entry=e, B=242, bands=HYPERION_GOOD) for e in ("mask", "fit", "apply")]


@pytest.fixture(scope="module")
def results():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-s", "-c", CHILD, ROOT], input=json.dumps(CASES), env=env, capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("entry", list(FN))
@pytest.mark.parametrize("case", list(BAD))
def test_bad_band_lists_are_refused_before_any_cuda_call(results, entry, case):
    rc, msg = results[f"{entry}/{case}"]
    assert rc == CMLPL_ERR_ARG and msg == f"{FN[entry]}: {BAD[case][2]}", msg


def test_scene_call_refuses_more_than_512_selected_bands(results):
    rc, msg = results["scene/513"]
    assert rc == CMLPL_ERR_ARG and msg == "scene_infer_raw_sel: band list of 513 bands, at most 512", msg


def test_apply_refuses_more_than_1024_selected_bands(results):
    rc, msg = results["apply/1025"]
    assert rc == CMLPL_ERR_ARG and msg == "preprocess_apply_sel: band list of 1025 bands, at most 1024", msg


@pytest.mark.parametrize("dtype", [0x00, 0x12, 0x21], ids=["bip-u16", "bil-i16", "bsq-f32"])
@pytest.mark.parametrize("w", [20, 11])
def test_hyperion_list_passes_every_check(results, dtype, w):
    """196 of 242 bands takes the dense path: its first CUDA call is the side stream, which cannot be created here."""
    rc, msg = results[f"scene/ok/{dtype}/{w}"]
    assert rc != 0 and msg == "scene_infer_raw_sel: cannot create the side stream", msg


def test_wide_list_passes_every_check(results):
    """300 of 425 bands takes the per-pixel path: its first CUDA call is the K-sliced conv0's shared-memory opt-in."""
    rc, msg = results["scene/ok/wide"]
    assert rc != 0 and not msg.startswith("scene_infer_raw_sel:") and "cudaFuncSetAttribute" in msg, msg


@pytest.mark.parametrize("entry", ["mask", "fit", "apply"])
def test_preprocessing_lists_pass_every_check(results, entry):
    rc, msg = results[f"{entry}/ok"]
    assert rc != 0 and not msg.startswith(FN[entry] + ":"), msg


def test_hyperion_workspace_is_the_dense_196_band_layout():
    """The workspace follows the selected count: 196 bands of a 242-band cube are sized and laid out as a 196-band call,
    the dense path (a 242-band call would be the per-pixel one)."""
    from cmlpl_b200 import _lib
    lib = _lib.load()
    for w in (20, 11):
        off = (ctypes.c_size_t * 12)()
        _lib.call("cmlpl_scene_workspace_layout", 610, 340, len(HYPERION_GOOD), 16, w, off)
        assert list(off)[11] == 1 and list(off)[10] == lib.cmlpl_scene_workspace_bytes(610, 340, 196, 16, w)
        _lib.call("cmlpl_scene_workspace_layout", 610, 340, 242, 16, w, off)
        assert list(off)[11] == 0


class _FakeCuda:
    """Stands in for a contiguous CUDA tensor (shape, dtype, pointer) so that a wrapper's checks run without a device."""
    is_cuda = True

    def __init__(self, shape, dtype=torch.float32):
        self.shape, self.dtype = tuple(shape), dtype

    def is_contiguous(self):
        return True

    def data_ptr(self):
        return GiB

    def numel(self):
        return int(np.prod(self.shape))


def test_scene_infer_raw_refuses_a_cube_of_another_band_count():
    """``folded`` carries the fit's list and the raw band count it selects from; a cube of another band count is refused
    before anything reaches the library."""
    from cmlpl_b200 import _lib, ops
    folded = {k: _FakeCuda(s) for k, s in (("wf", (196, 64)), ("bf", (64,)), ("mu", (196,)), ("inv_sigma", (196,)))}
    folded.update(bands=np.array(HYPERION_GOOD, dtype=np.int32), raw_bands=242)
    raw = _FakeCuda((30 * 40, 224), torch.uint16)
    with pytest.raises(_lib.CmlplError, match=r"raw has 224 bands, the band list of folded= selects from 242"):
        ops.scene_infer_raw(raw, folded, _FakeCuda((1,), torch.uint8), 16, 40, workspace=_FakeCuda((1,), torch.uint8),
                            labels=_FakeCuda((1200,), torch.uint8))


def test_band_list_helper():
    from cmlpl_b200 import _lib, preprocess
    assert preprocess.band_list([3, 5, 9]).dtype == np.int32
    assert preprocess.band_list(torch.tensor([1, 2])).tolist() == [1, 2]
    for bad in ([[1, 2]], [0.5, 1.5], [1 << 40]):
        with pytest.raises(_lib.CmlplError):
            preprocess.band_list(bad)


def test_sel_entry_points_are_declared():
    """The export test of test_oracle_cpu.py then checks them against the library."""
    from cmlpl_b200 import _lib
    for s in ("cmlpl_valid_mask_sel_u8", "cmlpl_preprocess_fit_sel_f64", "cmlpl_preprocess_apply_sel",
              "cmlpl_scene_infer_raw_sel"):
        assert s in _lib.SIGNATURES, s
    raw = _lib.SIGNATURES["cmlpl_scene_infer_raw"][1]
    P, I = ctypes.c_void_p, ctypes.c_int
    assert _lib.SIGNATURES["cmlpl_scene_infer_raw_sel"][1] == raw[:7] + [P, I] + raw[7:15] + [P] + raw[15:]
