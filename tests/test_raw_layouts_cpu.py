"""Raw cubes in BIL and BSQ and int16 samples, without a GPU: the raw codes (sample | interleave, include/cmlpl.h) of
`cmlpl_scene_infer_raw` and `cmlpl_preprocess_fit_cube_f64`, and the shape checks of the Python layer.

The entry points run in a child process in which no CUDA device is visible, with fake device pointers (as in
tests/test_scene_driver_cpu.py): a rejected code must return CMLPL_ERR_ARG with its own message before any CUDA call,
and every valid code must pass every check and fail only at its first CUDA call."""
import ctypes
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CMLPL_ERR_ARG = -1
GiB = 1 << 30
U16, F32, I16 = 0x00, 0x01, 0x02
BIP, BIL, BSQ = 0x00, 0x10, 0x20

# Runs the cases given on stdin and prints {case id: [return code, cmlpl_last_error()]}.
CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
from cmlpl_b200 import _lib
lib = _lib.load()
GiB = 1 << 30
out = {}
for c in json.load(sys.stdin):
    if c["entry"] == "scene_infer_raw":
        R, C = 30, 40
        rc = lib.cmlpl_scene_infer_raw(c["raw"], c["dtype"], R, C, 0, R, c["bands"], 22, c["w"], 0, R, 3 * GiB, 4 * GiB,
                                       5 * GiB, 6 * GiB, 7 * GiB, 8 * GiB, 1 << 40, 9 * GiB, None, None)
    elif c["entry"] == "fit_cube":
        rc = lib.cmlpl_preprocess_fit_cube_f64(c["raw"], c["dtype"], 30, 40, c["bands"], 2 * GiB, 3 * GiB, None)
    else:
        rc = lib.cmlpl_preprocess_fit_f64(c["raw"], c["dtype"], 1200, c["bands"], 2 * GiB, 3 * GiB, None)
    out[c["id"]] = [rc, lib.cmlpl_last_error().decode()]
print(json.dumps(out))
"""

CODES = [s | i for s in (U16, F32, I16) for i in (BIP, BIL, BSQ)]
VALID = [dict(id=f"raw/{code}/{w}/{B}", entry="scene_infer_raw", raw=GiB, dtype=code, w=w, bands=B)
         for code in CODES for w in (20, 11) for B in (103, 270, 512)]
VALID += [dict(id=f"fit_cube/{code}/{B}", entry="fit_cube", raw=GiB, dtype=code, w=20, bands=B)
          for code in CODES for B in (103, 270, 512)]
VALID += [dict(id=f"fit/{code}", entry="fit", raw=GiB, dtype=code, w=20, bands=103) for code in (U16, F32, I16)]

# id suffix -> (raw pointer, code, bands, message after "<entry point>: ")
REJECT = {
    "sample_3": (GiB, 3, 103, "unknown sample type 3 (0 = uint16, 1 = float32, 2 = int16)"),
    "interleave_0x30": (GiB, 0x30, 103, "unknown interleave 0x30 (0x00 = BIP, 0x10 = BIL, 0x20 = BSQ)"),
    "stray_bit_0x100": (GiB, 0x100 | BIL, 103, "dtype 0x110 has bits outside sample (0x0f) and interleave (0xf0)"),
    "negative_code": (GiB, -1, 103, "dtype 0xffffffff has bits outside sample (0x0f) and interleave (0xf0)"),
    "misaligned_f32": (GiB + 2, F32 | BSQ, 103, None),
    "misaligned_i16": (GiB + 1, I16 | BIL, 103, None),
}
CASES = VALID + [dict(id=f"{e}/{k}", entry=e, raw=r, dtype=d, w=20, bands=b)
                 for e in ("scene_infer_raw", "fit_cube") for k, (r, d, b, _) in REJECT.items()]
CASES += [dict(id="scene_infer_raw/513", entry="scene_infer_raw", raw=GiB, dtype=I16 | BSQ, w=20, bands=513),
          dict(id="fit/bil", entry="fit", raw=GiB, dtype=U16 | BIL, w=20, bands=103),
          dict(id="fit/bsq", entry="fit", raw=GiB, dtype=F32 | BSQ, w=20, bands=103),
          dict(id="fit/sample_3", entry="fit", raw=GiB, dtype=3, w=20, bands=103)]


@pytest.fixture(scope="module")
def results():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-s", "-c", CHILD, ROOT], input=json.dumps(CASES), env=env, capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("bands", [103, 270, 512])
@pytest.mark.parametrize("w", [20, 11])
@pytest.mark.parametrize("code", CODES, ids=[f"0x{c:02x}" for c in CODES])
def test_scene_infer_raw_accepts_every_sample_and_interleave(results, code, w, bands):
    """Up to 224 bands the first CUDA call is the side stream of the dense path; above, the K-sliced conv0 kernel's
    shared-memory opt-in.  Both fail without a device, after every check has passed."""
    rc, msg = results[f"raw/{code}/{w}/{bands}"]
    assert rc != 0, msg
    if bands <= 224:
        assert msg == "scene_infer_raw: cannot create the side stream", msg
    else:
        assert not msg.startswith("scene_infer_raw:") and "cudaFuncSetAttribute" in msg, msg


@pytest.mark.parametrize("bands", [103, 270, 512])
@pytest.mark.parametrize("code", CODES, ids=[f"0x{c:02x}" for c in CODES])
def test_fit_cube_accepts_every_sample_and_interleave(results, code, bands):
    rc, msg = results[f"fit_cube/{code}/{bands}"]
    assert rc != 0 and not msg.startswith("preprocess_fit_cube:") and "cudaMemsetAsync" in msg, msg


@pytest.mark.parametrize("code", [U16, F32, I16], ids=["u16", "f32", "i16"])
def test_fit_takes_bip_of_every_sample_type(results, code):
    rc, msg = results[f"fit/{code}"]
    assert rc != 0 and "cudaMemsetAsync" in msg, msg


@pytest.mark.parametrize("entry,name", [("scene_infer_raw", "scene_infer_raw"), ("fit_cube", "preprocess_fit_cube")])
@pytest.mark.parametrize("case", sorted(REJECT))
def test_bad_codes_are_refused_before_any_cuda_call(results, entry, name, case):
    rc, msg = results[f"{entry}/{case}"]
    want = REJECT[case][3]
    if want is None:
        esz = 4 if REJECT[case][1] & 0x0f == F32 else 2
        want = f"{'raw' if entry == 'scene_infer_raw' else 'x'} must be aligned to its {esz}-byte samples"
    assert rc == CMLPL_ERR_ARG and msg == f"{name}: {want}", msg


def test_513_bands_are_refused_in_every_code(results):
    rc, msg = results["scene_infer_raw/513"]
    assert rc == CMLPL_ERR_ARG and msg == "scene_infer_raw: needs <= 512 bands, got 513", msg


@pytest.mark.parametrize("case", ["bil", "bsq"])
def test_fit_of_n_by_b_refuses_band_major_codes(results, case):
    rc, msg = results[f"fit/{case}"]
    assert rc == CMLPL_ERR_ARG and msg.startswith("preprocess_fit: x is [n, B] band-interleaved-by-pixel"), msg


def test_fit_of_n_by_b_refuses_unknown_sample_type(results):
    rc, msg = results["fit/sample_3"]
    assert rc == CMLPL_ERR_ARG and msg == "preprocess_fit: unknown sample type 3 (0 = uint16, 1 = float32, 2 = int16)", msg


def test_workspace_takes_no_layout():
    """The workspace depends on the band's geometry only; the raw code is not one of its arguments."""
    from cmlpl_b200 import _lib
    assert _lib.SIGNATURES["cmlpl_scene_workspace_bytes"][1] == [ctypes.c_int] * 5
    assert _lib.SIGNATURES["cmlpl_scene_workspace_layout"][1] == [ctypes.c_int] * 5 + [ctypes.c_void_p]
    lib = _lib.load()
    lib.cmlpl_scene_workspace_bytes.restype = ctypes.c_size_t
    for B in (103, 270, 512):
        assert lib.cmlpl_scene_workspace_bytes(64, 475, B, 22, 20) > 0


# ------------------------------------------------------------------------------------------------- Python shapes
@pytest.mark.parametrize("interleave,shape,cols,want", [
    ("bip", (1200, 103), 40, (30, 40, 103)),
    ("bip", (1200, 103), None, (1200, 1, 103)),
    ("bip", (30, 40, 103), 40, (30, 40, 103)),
    ("bip", (30, 40, 103), None, (30, 40, 103)),
    ("bil", (30, 103, 40), 40, (30, 40, 103)),
    ("bil", (30, 103, 40), None, (30, 40, 103)),
    ("bsq", (103, 30, 40), 40, (30, 40, 103)),
    ("bsq", (103, 30, 40), None, (30, 40, 103)),
])
def test_raw_geometry_accepts_every_layout(interleave, shape, cols, want):
    from cmlpl_b200.preprocess import raw_geometry
    assert raw_geometry(shape, interleave, cols=cols) == want
    assert raw_geometry(shape, interleave, cols=cols, bands=103) == want


@pytest.mark.parametrize("interleave,shape,cols,bands", [
    ("bip", (1201, 103), 40, None),              # rows not a multiple of cols
    ("bip", (30, 41, 103), 40, None),            # wrong column count
    ("bip", (30, 40, 103), 40, 104),             # wrong band count
    ("bip", (1200,), None, None),                # wrong rank
    ("bil", (1200, 103), 40, None),              # 2-D is BIP only
    ("bil", (30, 40, 103), 40, 103),             # a BIP cube named BIL: 103 columns
    ("bil", (30, 103, 40), 40, 102),
    ("bsq", (30, 40, 103), 40, None),            # a BIP cube named BSQ
    ("bsq", (103, 30, 40), 41, None),
    ("bsq", (103, 30, 40, 1), 40, None),
    ("bsq", (103, 0, 40), 40, None),             # empty
    ("bis", (30, 40, 103), 40, None),            # unknown interleave
    ("bil", (2 ** 31, 103, 40), 40, None),       # rows beyond the C int of cmlpl_preprocess_fit_cube_f64
    ("bsq", (103, 30, 2 ** 31), None, None),     # columns beyond int
])
def test_raw_geometry_rejects_mismatched_shapes(interleave, shape, cols, bands):
    from cmlpl_b200._lib import CmlplError
    from cmlpl_b200.preprocess import raw_geometry
    with pytest.raises(CmlplError):
        raw_geometry(shape, interleave, cols=cols, bands=bands)


def test_raw_geometry_keeps_int64_bip_pixel_counts():
    """A 2-D BIP cube is fitted through cmlpl_preprocess_fit_f64, whose pixel count is int64."""
    from cmlpl_b200.preprocess import raw_geometry
    assert raw_geometry((2 ** 32 + 3, 4), "bip") == (2 ** 32 + 3, 1, 4)


def test_int16_is_a_raw_sample_type():
    import torch
    from cmlpl_b200._lib import CmlplError
    from cmlpl_b200.preprocess import INTERLEAVE, _dtype_code
    assert [_dtype_code(torch.empty(1, dtype=t)) for t in (torch.uint16, torch.float32, torch.int16)] == [0, 1, 2]
    assert INTERLEAVE == {"bip": BIP, "bil": BIL, "bsq": BSQ}
    with pytest.raises(CmlplError):
        _dtype_code(torch.empty(1, dtype=torch.int32))
