"""Spectra beyond 256 bands without a GPU: the 512-band bounds of the raw scene entry point and of the fused training
step, the WHU-Hi scenes of the CLIs, and a numpy port of the step's device Philox stream (used by the GPU tests of
tests/test_gpu_wide_bands.py), checked against the published Philox4x32-10 known-answer vectors.

The entry points run in a child process in which no CUDA device is visible, with fake device pointers (as in
tests/test_scene_driver_cpu.py): a rejected call must return CMLPL_ERR_ARG with its own message before any CUDA call,
and the 512-band controls must pass every check and fail only at their first CUDA call."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CMLPL_ERR_ARG = -1
GiB = 1 << 30

# Runs the raw scene entry point and the training step with the band counts given on stdin and prints
# {case id: [return code, cmlpl_last_error()]}.
CHILD = r"""
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from cmlpl_b200 import _lib
from cmlpl_b200.fused_step import TrainIO
lib = _lib.load()
GiB = 1 << 30
out = {}
for c in json.load(sys.stdin):
    B = c["bands"]
    if c["entry"] == "scene_infer_raw":
        R, C = 30, 40
        rc = lib.cmlpl_scene_infer_raw(1 * GiB, c["dtype"], R, C, 0, R, B, 22, c["w"], 0, R, 3 * GiB, 4 * GiB, 5 * GiB,
                                       6 * GiB, 7 * GiB, 8 * GiB, 1 << 40, 9 * GiB, None, None)
    else:
        io = TrainIO()
        io.bs, io.btu, io.bands, io.classes, io.w, io.queue = 128, 128, B, 22, c["w"], 1280
        io.cube, io.scene_rows, io.cols, io.pix = 1 * GiB, 940, 475, 2 * GiB
        io.spectra, io.labels, io.params = 3 * GiB, 4 * GiB, 5 * GiB
        io.logits, io.feat, io.probs, io.mask, io.hist = 6 * GiB, 7 * GiB, 8 * GiB, 9 * GiB, 10 * GiB
        io.work, io.work_bytes = 11 * GiB, 1 << 40
        for e in range(2):
            for i in range(10):
                base = (16 + 64 * e + 4 * i) * GiB
                io.net[e].p[i], io.net[e].g[i], io.net[e].m[i], io.net[e].v[i] = base, base + GiB, base + 2 * GiB, base + 3 * GiB
            io.net[e].queue_feats, io.net[e].queue_probs = (200 + 2 * e) * GiB, (201 + 2 * e) * GiB
        rc = lib.cmlpl_train_step(ctypes.byref(io), 15, None)
    out[c["id"]] = [rc, lib.cmlpl_last_error().decode()]
print(json.dumps(out))
"""

CASES = [dict(id=f"raw/{dt}/{w}/{B}", entry="scene_infer_raw", dtype=dt, w=w, bands=B)
         for dt in (0, 1) for w in (20, 11) for B in (513, 512, 270)]
CASES += [dict(id=f"step/{w}/{B}", entry="train_step", dtype=0, w=w, bands=B) for w in (20, 11) for B in (513, 512, 270)]


@pytest.fixture(scope="module")
def results():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-s", "-c", CHILD, ROOT], input=json.dumps(CASES), env=env, capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("dtype", [0, 1], ids=["u16", "f32"])
@pytest.mark.parametrize("w", [20, 11])
def test_raw_entry_point_refuses_513_bands(results, dtype, w):
    rc, msg = results[f"raw/{dtype}/{w}/513"]
    assert rc == CMLPL_ERR_ARG and msg == "scene_infer_raw: needs <= 512 bands, got 513", msg


@pytest.mark.parametrize("bands", [512, 270])
@pytest.mark.parametrize("dtype", [0, 1], ids=["u16", "f32"])
@pytest.mark.parametrize("w", [20, 11])
def test_raw_entry_point_accepts_up_to_512_bands(results, bands, dtype, w):
    """Above 224 bands the raw entry point takes the per-pixel path: no side stream, so the first CUDA call it makes is
    the K-sliced conv0 kernel's shared-memory opt-in, which fails without a device."""
    rc, msg = results[f"raw/{dtype}/{w}/{bands}"]
    assert rc != 0 and not msg.startswith("scene_infer_raw:") and "cudaFuncSetAttribute" in msg, msg


@pytest.mark.parametrize("w", [20, 11])
def test_train_step_refuses_513_bands(results, w):
    rc, msg = results[f"step/{w}/513"]
    assert rc == CMLPL_ERR_ARG and msg == "train_step: needs <= 512 bands, got 513", msg


@pytest.mark.parametrize("bands", [512, 270])
@pytest.mark.parametrize("w", [20, 11])
def test_train_step_accepts_up_to_512_bands(results, bands, w):
    rc, msg = results[f"step/{w}/{bands}"]
    assert rc != 0 and msg == "train_step: could not create the side stream", msg


def test_wide_scene_workspace_is_the_per_pixel_layout():
    """A 270-band scene call runs the per-pixel path on both entry points: conv0 map, pooled features, spectral logits
    and the hidden chunk, with no tensor-core spectral regions and no dense regions."""
    from cmlpl_b200 import _lib
    off = (ctypes.c_size_t * 12)()
    for w in (20, 11):
        _lib.call("cmlpl_scene_workspace_layout", 64, 475, 270, 22, w, off)
        f0pad, x16, h16, g, pm, yq, lmap, p2, spe, hidden, total, dense = list(off)
        assert dense == 0 and x16 == h16 == g == pm == yq == lmap == 0
        assert 0 == f0pad < p2 < spe < hidden < total


# ------------------------------------------------------------------------------------------------------- the CLIs
def test_whu_hi_scenes_in_the_dataset_tables():
    from cmlpl_b200 import synth
    from cmlpl_b200.hsi_loader import ROOTS
    from cmlpl_b200.sample_generation import SYNTHETIC
    from cmlpl_b200.tools.hyper_tools import DATASETS, _MAT
    want = {5: ("WHU_Hi_LongKou", 550, 400, 270, 9), 6: ("WHU_Hi_HanChuan", 1217, 303, 274, 16),
            7: ("WHU_Hi_HongHu", 940, 475, 270, 22)}
    for i, (name, R, C, B, K) in want.items():
        assert DATASETS[i] == (name, K, B)
        assert _MAT[i] == (name + ".mat", name, name + "_gt.mat", name + "_gt")
        assert ROOTS[i] == f"./dataset/{name}/"
        assert synth.SHAPES[SYNTHETIC[i]] == (R, C, B, K)
    # the scenes that were there keep their entries
    assert DATASETS[1] == ("PaviaU", 9, 103) and DATASETS[4] == ("Indian_pines", 16, 200)
    assert [synth.SHAPES[SYNTHETIC[i]] for i in (1, 2, 3, 4)] == [(610, 340, 103, 9), (512, 217, 204, 16),
                                                                  (349, 1905, 144, 15), (145, 145, 200, 16)]


def test_synthetic_honghu_scene(monkeypatch):
    """``--synthetic`` with dataID 7 builds a HongHu-shaped scene: 270 uint16 bands, labels 0..22."""
    from cmlpl_b200 import sample_generation as SG, synth
    monkeypatch.setitem(synth.SHAPES, "whu_honghu", (40, 36, 270, 22))
    cube, gt = SG.load_scene(7, synthetic=True)
    assert cube.shape == (40, 36, 270) and cube.dtype == np.uint16
    assert gt.shape == (40, 36) and int(gt.max()) == 22


# ----------------------------------------------------------------------------------- device Philox stream, in numpy
PHILOX_PATCH, PHILOX_SPEC, PHILOX_DROP, PHILOX_SPEC_HI = 1, 2, 3, 4


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11) on uint32 arrays: ctr [..., 4], key [..., 2] (train_common.cuh)."""
    c = [ctr[..., i].astype(np.uint64) for i in range(4)]
    k0, k1 = key[..., 0].astype(np.uint64), key[..., 1].astype(np.uint64)
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & m32, p1 >> np.uint64(32), p1 & m32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m32, (k1 + np.uint64(0xBB67AE85)) & m32
    return np.stack([x.astype(np.uint32) for x in c], -1)


def philox_normal4(seed, offset, stream, index):
    """Four N(0,1) draws per (stream, index), Box-Muller on (0,1] uniforms, in float64 (the kernel's __logf / __sincosf
    differ from it in the last bits only)."""
    index = np.asarray(index, dtype=np.uint64)
    stream = np.broadcast_to(np.asarray(stream, dtype=np.uint64), index.shape)
    ctr = np.stack([index, stream, np.full_like(index, offset & 0xFFFFFFFF), np.full_like(index, offset >> 32)], -1)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64), index.shape + (2,))
    r = philox4x32_10(ctr.astype(np.uint32), key).astype(np.float64)
    u0 = (np.floor(r[..., 0] / 256) + 1) / 16777216.0
    u1 = np.floor(r[..., 1] / 256) / 16777216.0
    u2 = (np.floor(r[..., 2] / 256) + 1) / 16777216.0
    u3 = np.floor(r[..., 3] / 256) / 16777216.0
    ra, rb = np.sqrt(-2 * np.log(u0)), np.sqrt(-2 * np.log(u2))
    t1, t3 = 2 * np.pi * u1, 2 * np.pi * u3
    return np.stack([ra * np.cos(t1), ra * np.sin(t1), rb * np.cos(t3), rb * np.sin(t3)], -1)


def spectral_noise(seed, offset, samples, bands):
    """The draws of the fused step's spectral noise: [samples, bands] (train_common.cuh: spec_noise_counter)."""
    s = np.arange(samples, dtype=np.uint64)[:, None]
    j4 = np.arange((bands + 3) // 4, dtype=np.uint64)[None, :]
    g = j4 >> np.uint64(6)
    stream = np.where(g == 0, np.uint64(PHILOX_SPEC), np.uint64(PHILOX_SPEC_HI) + g - np.uint64(1))
    index = (s * np.uint64(64) + (j4 & np.uint64(63))) & np.uint64(0xFFFFFFFF)
    z = philox_normal4(seed, offset, np.broadcast_to(stream, index.shape), index)
    return z.reshape(samples, -1)[:, :bands]


def test_philox_port_matches_the_known_answer_vectors():
    """Random123's kat_vectors for philox4x32_10."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        got = philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
        assert [int(x) for x in got] == list(want)


def test_spectral_noise_layout_is_disjoint_up_to_512_bands_and_unchanged_below_256():
    """Bands 0..255 draw (PHILOX_SPEC, s*64 + j4) as before; no (stream, counter) pair repeats over 512 samples x 512
    bands, so no two positions of one step share a draw."""
    S, B = 512, 512
    s = np.arange(S)[:, None]
    j4 = np.arange(B // 4)[None, :]
    g = j4 >> 6
    stream = np.where(g == 0, PHILOX_SPEC, PHILOX_SPEC_HI + g - 1)
    index = s * 64 + (j4 & 63)
    key = stream.astype(np.int64) << 32 | index
    assert np.unique(key).size == S * B // 4
    assert (stream[:, :64] == PHILOX_SPEC).all() and (index[:, :64] == s * 64 + j4[:, :64]).all()
    assert not np.isin(stream, [PHILOX_PATCH, PHILOX_DROP]).any()
    z = spectral_noise(1088, 3, 8, 425)
    assert z.shape == (8, 425) and np.unique(z).size == z.size
