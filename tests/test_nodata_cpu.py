"""No-data pixels of raw sensor cubes, without a GPU: the float64 definitions the GPU tests compare against, and the
argument checks of the four entry points that take a fill value or a validity mask.

Definitions (include/cmlpl.h, "No-data pixels"):
  * a sample is missing when it equals the fill value in the sample type; a float32 sample that is not finite is always
    missing (fill NaN: only then);
  * a pixel with any band missing is no-data; the validity mask is u8 [rows, cols], 1 = valid;
  * a no-data pixel stands in as its band-mean spectrum x = mu everywhere it is read, and is labelled 255.
So the scene oracle is: overwrite the no-data pixels with mu in float64, run the oracle's test_whole, set their labels
to 255.

The entry points run in a child process in which no CUDA device is visible, with fake device pointers (as in
tests/test_scene_driver_cpu.py): a rejected call returns CMLPL_ERR_ARG with its own message before any CUDA call, and
the valid controls pass every check and fail only at their first CUDA call."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import cmlpl_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NODATA = 255


# ------------------------------------------------------------------------------------------------ oracle (float64)
def valid_mask(cube, fill=None):
    """cube [R, C, B] of the sample type -> (valid u8 [R, C], n_valid, band_missing int64 [B])."""
    cube = np.asarray(cube)
    if np.issubdtype(cube.dtype, np.floating):
        miss = ~np.isfinite(cube)
        if fill is not None and not np.isnan(fill):
            miss |= cube == cube.dtype.type(fill)
    else:
        if fill is None:
            raise ValueError("an integer cube needs a fill value")
        miss = cube == fill
    valid = ~miss.any(-1)
    return valid.astype(np.uint8), int(valid.sum()), miss.reshape(-1, cube.shape[-1]).sum(0).astype(np.int64)


def impute_nodata(cube, valid, mu):
    """float64 copy of cube [R, C, B] with every no-data pixel replaced by the band means mu [B]."""
    X = np.asarray(cube, dtype=np.float64).copy()
    X[np.asarray(valid) == 0] = mu
    return X


def nodata_pattern(R, C, kind, seed=0):
    """bool [R, C], True = no-data:
       "wedge"  the corner wedges outside a swath rotated by 20 degrees (~20-30 % of the pixels)
       "lines"  whole dropped scan lines (in the middle third of the rows)
       "pixels" isolated pixels (~1 %)
       "edge"   a block touching the top and left scene edges, so the mirror reflects it into the windows there"""
    rng = np.random.default_rng(seed)
    r, c = np.mgrid[0:R, 0:C]
    if kind == "wedge":
        t = np.deg2rad(20.0)
        u = (c - (C - 1) / 2) * np.cos(t) - (r - (R - 1) / 2) * np.sin(t)     # across-track coordinate
        return np.abs(u) > 0.36 * C
    if kind == "lines":
        m = np.zeros((R, C), bool)
        m[rng.choice(np.arange(R // 3, 2 * R // 3), max(2, R // 20), replace=False)] = True     # the middle third
        return m
    if kind == "pixels":
        return rng.random((R, C)) < 0.01
    if kind == "edge":
        m = np.zeros((R, C), bool)
        m[:max(2, R // 6), :max(3, C // 5)] = True
        return m
    raise ValueError(kind)


def with_nodata(cube, nodata, fill, seed=0):
    """cube with fill values at the no-data pixels: every band of most of them, a few bands of the others (one band
    missing makes the pixel no-data).  float32 cubes with fill None get NaN, +Inf or -Inf instead."""
    rng = np.random.default_rng(seed)
    out = cube.copy()
    rr, cc = np.nonzero(nodata)
    B = cube.shape[2]
    for i, (r, c) in enumerate(zip(rr, cc)):
        bands = slice(None) if i % 3 else rng.choice(B, 1 + i % 5, replace=False)
        if fill is None or (isinstance(fill, float) and np.isnan(fill)):
            out[r, c, bands] = (np.nan, np.inf, -np.inf)[i % 3]
        else:
            out[r, c, bands] = fill
    return out


def window_touches(nodata, w):
    """bool [R, C]: the pixel's w x w window, after mirroring at the scene edges, holds a no-data pixel."""
    R, C = nodata.shape
    lo = -(w // 2)
    rows = O.mirror_index(np.arange(R)[:, None] + lo + np.arange(w)[None], R)      # [R, w]
    cols = O.mirror_index(np.arange(C)[:, None] + lo + np.arange(w)[None], C)      # [C, w]
    t = nodata[rows].any(1)                                                          # [R, C]: any row of the window
    return t[:, cols].any(2)


def scene_oracle(sd, cube, valid, pp, w):
    """Labels and logits of the imputed scene: no-data pixels replaced by mu, test_whole, their labels set to 255."""
    Xp, Xs = O.apply_preprocess(impute_nodata(cube, valid, pp["mu"]), pp)
    lab, log = O.test_whole(sd, Xp.astype(np.float32), Xs.astype(np.float32), w, odd_mode=(w == 11), return_logits=True)
    lab = lab.astype(np.int64)
    lab[valid.reshape(-1) == 0] = NODATA
    return lab, log


def masked_params(cube, valid, n_PC=60):
    """preprocess_params over the valid pixels only."""
    B = cube.shape[2]
    return O.preprocess_params(cube.reshape(-1, B)[valid.reshape(-1) != 0][None], n_PC)


# ------------------------------------------------------------------------------------------------ the oracle itself
def test_mask_follows_the_rules_on_a_hand_built_cube():
    u16 = np.array([[[5, 5, 5], [0, 5, 5], [5, 5, 0]],
                    [[0, 0, 0], [7, 8, 9], [1, 2, 3]]], dtype=np.uint16)
    v, n, miss = valid_mask(u16, 0)
    assert v.tolist() == [[1, 0, 0], [0, 1, 1]] and n == 3 and miss.tolist() == [2, 1, 2]
    i16 = u16.astype(np.int16) - 1
    i16[0, 0, 1] = -32768
    v, n, miss = valid_mask(i16, -32768)
    assert v.tolist() == [[0, 1, 1], [1, 1, 1]] and n == 5 and miss.tolist() == [0, 1, 0]
    f = u16.astype(np.float32)
    f[1, 1, 2], f[1, 2, 0] = np.nan, -np.inf
    v, n, miss = valid_mask(f, None)                     # NaN / Inf only: the zeros are data
    assert v.tolist() == [[1, 1, 1], [1, 0, 0]] and n == 4 and miss.tolist() == [1, 0, 1]
    v, n, miss = valid_mask(f, 0.0)                      # zeros too
    assert v.tolist() == [[1, 0, 0], [0, 0, 0]] and n == 1 and miss.tolist() == [3, 1, 3]
    with pytest.raises(ValueError):
        valid_mask(u16, None)


def test_imputation_and_the_scene_oracle_on_a_small_scene():
    """Imputed pixels carry mu exactly, so their z-scored spectra are 0 and their PCA rows -pca_mu / pca_sigma; the
    scene oracle labels them 255 and leaves every pixel whose window holds no no-data pixel as on the clean scene."""
    R, C, B, K, w = 14, 15, 64, 4, 11
    cube, _ = O.sensor_scene(R, C, B, K, 4.0, seed=3, sample="u16", dc=100.0)
    nd = nodata_pattern(R, C, "edge")
    dirty = with_nodata(cube, nd, 0)
    valid, n, _ = valid_mask(dirty, 0)
    assert np.array_equal(valid == 0, nd) and n == R * C - nd.sum()
    pp = masked_params(dirty, valid)
    X = impute_nodata(dirty, valid, pp["mu"])
    assert np.array_equal(X[nd], np.broadcast_to(pp["mu"], (nd.sum(), B)))
    assert np.array_equal(X[~nd], cube[~nd].astype(np.float64))
    Xp, Xs = O.apply_preprocess(X, pp)
    assert np.abs(Xs.reshape(R, C, B)[nd]).max() == 0
    assert np.allclose(Xp[nd], -pp["pca_mu"] / pp["pca_sigma"], rtol=0, atol=1e-12)
    assert np.allclose(pp["pca_mu"], 0, atol=1e-9 * np.abs(pp["pca_mu"]).max() + 1e-9)
    sd = O.basenet2_init(B, K, conv_feat=64 * 2 * 2)
    lab, log = scene_oracle(sd, dirty, valid, pp, w)
    assert np.all(lab[nd.reshape(-1)] == NODATA)
    # the same scene with the no-data pixels set to mu by hand, through the unmodified oracle path
    Xp2, Xs2 = O.apply_preprocess(np.where(nd[..., None], pp["mu"], cube.astype(np.float64)), pp)
    lab2 = O.test_whole(sd, Xp2.astype(np.float32), Xs2.astype(np.float32), w, odd_mode=True)
    far = ~window_touches(nd, w).reshape(-1)
    assert far.sum() > 0 and np.array_equal(lab[far], lab2[far])


def test_patterns_cover_their_cases():
    R, C = 60, 70
    wedge = nodata_pattern(R, C, "wedge")
    assert 0.2 <= wedge.mean() <= 0.3 and wedge[0, -1] and wedge[-1, 0] and not wedge[R // 2, C // 2]
    lines = nodata_pattern(R, C, "lines")
    assert np.all(lines.all(1) | ~lines.any(1)) and lines.any()
    px = nodata_pattern(R, C, "pixels")
    assert 0 < px.mean() < 0.03
    edge = nodata_pattern(R, C, "edge")
    assert edge[0, 0] and not edge[-1, -1]
    # the block reaches the windows of pixels outside it, and through the mirror every copy of it is the block itself
    t = window_touches(edge, 20)
    assert t[0, 20] and t[15, 5] and not t[0, 30] and not t[-1, -1]
    f = with_nodata(np.ones((R, C, 8), np.float32), px, None)
    assert np.array_equal(valid_mask(f)[0] == 0, px)


def test_window_touches_matches_a_loop():
    rng = np.random.default_rng(1)
    nd = rng.random((13, 17)) < 0.05
    for w in (20, 11):
        got = window_touches(nd, w)
        lo = -(w // 2)
        for r in range(13):
            for c in range(17):
                rr = O.mirror_index(np.arange(r + lo, r + lo + w), 13)
                cc = O.mirror_index(np.arange(c + lo, c + lo + w), 17)
                assert got[r, c] == nd[np.ix_(rr, cc)].any()


# ------------------------------------------------------------------------------------------------ the C ABI
NEW = ("cmlpl_valid_mask_u8", "cmlpl_preprocess_fit_masked_f64", "cmlpl_preprocess_apply_masked",
       "cmlpl_scene_infer_raw_masked")


def test_new_symbols_are_declared_bound_and_exported():
    import ctypes
    from cmlpl_b200 import _lib
    header = open(os.path.join(ROOT, "include", "cmlpl.h")).read()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in NEW:
        assert re.search(r"\bint %s\(" % s, header), s
        assert s in _lib.SIGNATURES and hasattr(lib, s), s
    assert re.search(r"#define CMLPL_NODATA_LABEL 255\b", header)
    from cmlpl_b200 import ops
    assert ops.NODATA_LABEL == 255
    # the masked scene entry point takes the raw one's arguments plus the mask
    raw = _lib.SIGNATURES["cmlpl_scene_infer_raw"][1]
    assert _lib.SIGNATURES["cmlpl_scene_infer_raw_masked"][1] == raw[:15] + [ctypes.c_void_p] + raw[15:]
    app = _lib.SIGNATURES["cmlpl_preprocess_apply"][1]
    assert _lib.SIGNATURES["cmlpl_preprocess_apply_masked"][1] == app[:9] + [ctypes.c_void_p] + app[9:]


# Runs every case given on stdin and prints {case id: [return code, cmlpl_last_error()]}.
CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
from cmlpl_b200 import _lib
lib = _lib.load()
out = {}
for c in json.load(sys.stdin):
    a, e = c["args"], c["entry"]
    if e == "valid_mask":
        rc = lib.cmlpl_valid_mask_u8(a["raw"], a["dtype"], a["rows"], a["cols"], a["B"], float(a["fill"]), a["valid"],
                                     a["n_valid"], a["band_missing"], None)
    elif e == "fit_masked":
        rc = lib.cmlpl_preprocess_fit_masked_f64(a["raw"], a["dtype"], a["rows"], a["cols"], a["B"], a["valid"], a["mean"],
                                                 a["gram"], a["n_valid"], None)
    elif e == "apply_masked":
        rc = lib.cmlpl_preprocess_apply_masked(a["raw"], a["dtype"], a["rows"] * a["cols"], a["B"], 60, a["mu"],
                                               a["inv_sigma"], a["Us"], a["shift"], a["valid"], a["cube"], a["spectra"],
                                               None)
    else:
        rc = lib.cmlpl_scene_infer_raw_masked(a["raw"], a["dtype"], a["rows"], a["cols"], 0, a["rows"], a["B"], 9, a["w"],
                                              a["band_row0"], a["band_rows"], a["wf"], a["bf"], a["mu"], a["inv_sigma"],
                                              a["valid"], a["packed"], a["workspace"], 1 << 40, a["labels"], None, None)
    out[c["id"]] = [rc, lib.cmlpl_last_error().decode()]
print(json.dumps(out))
"""

GiB = 1 << 30
U16, F32, I16, BIL = 0x00, 0x01, 0x02, 0x10
VALID = dict(raw=GiB, dtype=U16, rows=30, cols=40, B=103, fill=0.0, valid=2 * GiB, n_valid=3 * GiB, band_missing=4 * GiB,
             mean=5 * GiB, gram=6 * GiB, mu=7 * GiB, inv_sigma=8 * GiB, Us=9 * GiB, shift=10 * GiB, cube=11 * GiB,
             spectra=12 * GiB, wf=13 * GiB, bf=14 * GiB, packed=15 * GiB, workspace=16 * GiB, labels=17 * GiB, w=20,
             band_row0=0, band_rows=30)
ENTRIES = ("valid_mask", "fit_masked", "apply_masked", "scene_infer_raw_masked")
NAMES = {"valid_mask": "valid_mask", "fit_masked": "preprocess_fit_masked", "apply_masked": "preprocess_apply_masked",
         "scene_infer_raw_masked": "scene_infer_raw_masked"}

# id -> (changed arguments, {entry: message after "<entry point name>: "})
CASES = {
    "null_valid": (dict(valid=None), {"valid_mask": "null pointer", "fit_masked": r"null valid mask or n_valid",
                                      "apply_masked": "null valid mask", "scene_infer_raw_masked": "null valid mask"}),
    "u16_fill_-9999": (dict(fill=-9999.0), {"valid_mask": "fill -9999 is not a uint16 value"}),
    "u16_fill_70000": (dict(fill=70000.0), {"valid_mask": "fill 70000 is not a uint16 value"}),
    "i16_fill_0.5": (dict(dtype=I16, fill=0.5), {"valid_mask": "fill 0.5 is not an int16 value"}),
    "i16_fill_40000": (dict(dtype=I16 | BIL, fill=40000.0), {"valid_mask": "fill 40000 is not an int16 value"}),
    "f32_fill_0.1": (dict(dtype=F32, fill=0.1), {"valid_mask": r"fill 0.10000000000000001 is not a float32 value"}),
    "u16_fill_nan": (dict(fill="nan"), {"valid_mask": "a NaN fill marks non-finite float32 samples; an integer cube needs "
                                                      "its fill value"}),
    "i16_fill_nan": (dict(dtype=I16, fill="nan"), {"valid_mask": "a NaN fill marks non-finite float32 samples; an integer "
                                                                 "cube needs its fill value"}),
    "no_rows": (dict(rows=0), {"valid_mask": r"bad dims \(rows=0 cols=40 bands=103; at most 8192 bands\)",
                               "fit_masked": r"bad dims \(rows=0 cols=40 bands=103\)"}),
    "no_bands": (dict(B=0), {"valid_mask": r"bad dims \(rows=30 cols=40 bands=0; at most 8192 bands\)",
                             "fit_masked": r"bad dims \(rows=30 cols=40 bands=0\)",
                             "apply_masked": r"bad args \(dtype: BIP uint16, float32 or int16\)",
                             "scene_infer_raw_masked": r"bad dims \(band_rows=30 cols=40 bands=0\)"}),
    "band_outside_the_scene": (dict(band_row0=25, band_rows=10), {"scene_infer_raw_masked": "band outside the scene"}),
    "w_16": (dict(w=16), {"scene_infer_raw_masked": r"w=16 unsupported \(20, or 11 for the odd-window variant\)"}),
    "bad_interleave": (dict(dtype=0x30), {e: r"unknown interleave 0x30 \(0x00 = BIP, 0x10 = BIL, 0x20 = BSQ\)"
                                          for e in ("valid_mask", "fit_masked", "scene_infer_raw_masked")}),
}
PARAMS = [(e, k) for k, (_, msgs) in CASES.items() for e in ENTRIES if e in msgs]
# controls: every sample type and a float32 NaN fill pass the mask's checks
CONTROLS = {"u16": dict(), "i16_-32768": dict(dtype=I16 | BIL, fill=-32768.0), "f32_nan": dict(dtype=F32, fill="nan"),
            "f32_-9999": dict(dtype=F32 | 0x20, fill=-9999.0), "u16_65535": dict(fill=65535.0)}


@pytest.fixture(scope="module")
def results():
    cases = [dict(id=f"{e}/{k}", entry=e, args={**VALID, **CASES[k][0]}) for e, k in PARAMS]
    cases += [dict(id=f"{e}/valid", entry=e, args=VALID) for e in ENTRIES]
    cases += [dict(id=f"valid_mask/valid/{k}", entry="valid_mask", args={**VALID, **a}) for k, a in CONTROLS.items()]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-s", "-c", CHILD, ROOT], input=json.dumps(cases), env=env, capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("entry,case", PARAMS)
def test_rejected_before_any_cuda_call(results, entry, case):
    rc, msg = results[f"{entry}/{case}"]
    assert rc == -1, msg
    assert re.fullmatch(f"{NAMES[entry]}: {CASES[case][1][entry]}", msg), msg


@pytest.mark.parametrize("entry", ENTRIES)
def test_valid_arguments_pass_every_check(results, entry):
    """The control: with no device visible, valid arguments fail at the first CUDA call (CMLPL_ERR_CUDA), not a check;
    the dense scene path's first CUDA call is the creation of the side stream, which has its own message."""
    rc, msg = results[f"{entry}/valid"]
    if entry == "scene_infer_raw_masked":
        assert rc != 0 and msg == "scene_infer_raw_masked: cannot create the side stream", msg
    else:
        assert rc == -2, msg


@pytest.mark.parametrize("case", list(CONTROLS))
def test_representable_fills_pass_the_mask_checks(results, case):
    rc, msg = results[f"valid_mask/valid/{case}"]
    assert rc == -2, msg


def test_python_layer_checks_without_a_device():
    import torch
    from cmlpl_b200 import _lib, preprocess
    with pytest.raises(_lib.CmlplError, match="needs its fill value"):
        preprocess._fill_value(torch.empty(0, dtype=torch.uint16), None)
    assert np.isnan(preprocess._fill_value(torch.empty(0, dtype=torch.float32), None))
    assert preprocess._fill_value(torch.empty(0, dtype=torch.int16), -32768) == -32768.0
    with pytest.raises(_lib.CmlplError, match="contiguous CUDA"):
        preprocess.valid_mask(torch.zeros(4, 3, dtype=torch.uint16), 0)
