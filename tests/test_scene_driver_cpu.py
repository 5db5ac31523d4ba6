"""Argument checks of the two scene entry points (no GPU).

A rejected `cmlpl_scene_infer` / `cmlpl_scene_infer_raw` call must return CMLPL_ERR_ARG, with a message that names the
entry point and the failed condition, before it makes any CUDA call: a call that enqueued work first and rejected its
arguments afterwards would leave a kernel writing into the caller's workspace on a stream the caller never waits on.

The calls run in a child process in which no CUDA device is visible, with fake device pointers, so no call can reach a
device.  There the first CUDA call of the dense path, the creation of the side stream, fails with its own message,
which replaces the expected one; the control case shows that a call with valid arguments gets that far."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CMLPL_ERR_ARG = -1

# Runs every case given on stdin and prints {case id: [return code, cmlpl_last_error()]}.
CHILD = r"""
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from cmlpl_b200 import _lib
lib = _lib.load()
out = {}
for c in json.load(sys.stdin):
    a = c["args"]
    if c["entry"] == "scene_infer":
        rc = lib.cmlpl_scene_infer(a["cube"], a["scene_rows"], a["cols"], a["slab_row0"], a["slab_rows"], a["spectra"],
                                   a["B"], a["K"], a["w"], a["band_row0"], a["band_rows"], a["packed"], a["workspace"],
                                   a["ws_bytes"], a["labels"], None, None)
    else:
        rc = lib.cmlpl_scene_infer_raw(a["cube"], 0, a["scene_rows"], a["cols"], a["slab_row0"], a["slab_rows"], a["B"],
                                       a["K"], a["w"], a["band_row0"], a["band_rows"], a["wf"], a["bf"], a["mu"],
                                       a["inv_sigma"], a["packed"], a["workspace"], a["ws_bytes"], a["labels"], None, None)
    out[c["id"]] = [rc, lib.cmlpl_last_error().decode()]
print(json.dumps(out))
"""

R, C, B, K, W = 30, 40, 103, 9, 20          # a shape of the dense path (path mode 1, the default)
GiB = 1 << 30
VALID = dict(cube=1 * GiB, spectra=2 * GiB, wf=3 * GiB, bf=4 * GiB, mu=5 * GiB, inv_sigma=6 * GiB, packed=7 * GiB,
             workspace=8 * GiB, labels=9 * GiB, ws_bytes=1 << 40, scene_rows=R, cols=C, slab_row0=0, slab_rows=R,
             B=B, K=K, w=W, band_row0=0, band_rows=R)


# id -> (changed arguments, message after "<entry point>: ", entry points)
CASES = {
    "band_outside_the_scene": (dict(band_row0=25, band_rows=10), "band outside the scene", None),
    # rows 0..9 need scene row 0 (and its mirror images); the slab starts at row 1
    "slab_misses_the_halo_at_the_top_edge": (dict(band_rows=10, slab_row0=1, slab_rows=R - 1),
                                             r"slab rows \[1,30\) do not cover the band's halo \[0,18\]", None),
    # rows 20..29 need the last scene row; the slab ends one row short
    "slab_misses_the_halo_at_the_bottom_edge": (dict(band_row0=20, band_rows=10, slab_row0=10, slab_rows=R - 11),
                                                r"slab rows \[10,29\) do not cover the band's halo \[10,29\]", None),
    "window_larger_than_the_scene": (dict(scene_rows=8, slab_rows=8, band_rows=8), "window larger than the scene", None),
    "no_bands": (dict(B=0), r"bad dims \(band_rows=30 cols=40 bands=0\)", None),
    "33_classes": (dict(K=33), "needs 1..32 classes, got 33", None),
    "w_16": (dict(w=16), r"w=16 unsupported \(20, or 11 for the odd-window variant\)", None),
    "workspace_too_small": (dict(ws_bytes="required - 1"), r"workspace (\d+) < required (\d+)", None),
    "workspace_not_256_byte_aligned": (dict(workspace=8 * GiB + 128), "workspace must be 256-byte aligned", None),
    "cube_not_16_byte_aligned": (dict(cube=1 * GiB + 4), "cube must be 16-byte aligned", ("scene_infer",)),
}
ENTRIES = ("scene_infer", "scene_infer_raw")
PARAMS = [(e, k) for k, (_, _, only) in CASES.items() for e in ENTRIES if only is None or e in only]


@pytest.fixture(scope="module")
def results():
    from cmlpl_b200 import _lib
    required = _lib.load().cmlpl_scene_workspace_bytes(R, C, B, K, W)
    cases = [dict(id=f"{e}/{k}", entry=e, args={**VALID, **CASES[k][0]}) for e, k in PARAMS]
    for c in cases:
        if c["args"]["ws_bytes"] == "required - 1":
            c["args"]["ws_bytes"] = required - 1
    cases += [dict(id=f"{e}/valid", entry=e, args=VALID) for e in ENTRIES]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-s", "-c", CHILD, ROOT], input=json.dumps(cases), env=env, capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("entry,case", PARAMS)
def test_rejected_before_any_cuda_call(results, entry, case):
    rc, msg = results[f"{entry}/{case}"]
    assert rc == CMLPL_ERR_ARG, msg
    m = re.fullmatch(f"{entry}: {CASES[case][1]}", msg)
    assert m, msg
    if case == "workspace_too_small":
        assert int(m[1]) + 1 == int(m[2]) > 0


@pytest.mark.parametrize("entry", ENTRIES)
def test_valid_arguments_reach_the_side_stream(results, entry):
    """The control: with no device visible, valid arguments pass every check and fail at the first CUDA call."""
    rc, msg = results[f"{entry}/valid"]
    assert rc != 0 and msg == f"{entry}: cannot create the side stream", msg
