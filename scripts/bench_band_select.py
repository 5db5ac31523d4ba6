"""Band selection: what reading a band list from the whole raw cube costs raw-cube scene inference (GPU only; CUDA
events), and whether the entry points without a list kept their speed.

Workloads (w = 20, device-resident raw cubes of seeded random values in 1..8000, random-init nets):
  * paviau_bip_u16 / paviau_bil_i16: a PaviaU-size 610 x 340 scene of 224 raw bands, 200 listed (24 left out: the
    water-absorption bands 104-108, 150-163 and 220, 1-based, and the first four), 9 classes: the dense path;
  * hyperion_bil_i16: a Hyperion-like 1000 x 256 L1R scene of 242 raw bands, 196 listed (8-57, 77-224 in 0-based
    indices as in the band list of tests/test_gpu_band_select.py), 12 classes: the dense path (242 bands would not be);
  * honghu_bil_u16: a HongHu-shaped 940 x 475 scene of 300 raw bands, 270 listed, 22 classes: K-sliced conv0 and the
    CUDA-core spectral head.
Each compares, alternated round by round: the call with the list on the whole cube ("selected"), the call without a list
on the pre-compacted cube ("compacted"), and index_select + the call without a list ("index_select_then_call"); their
labels must be equal.

With --parent LIB (the parent commit's libcmlpl_sm100.so), the entry points without a list are also timed against it in
the same process, alternated round by round: cmlpl_scene_infer_raw on PaviaU (103 bands, BIP uint16) and HongHu (270
bands, BIL uint16), cmlpl_valid_mask_u8 and cmlpl_preprocess_fit_cube_f64 on the HongHu cube; their labels must be equal.
The card's name and power limit are read in the same run.

    python scripts/bench_band_select.py --parent scripts/_parent/libcmlpl_parent.so --out profiles/band_select.json
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from bench_raw_layouts import layout  # noqa: E402
from bench_wide_bands import card, timed_rounds  # noqa: E402
from cmlpl_b200 import _lib, ops, preprocess  # noqa: E402
from cmlpl_b200.tools.models import BaseNet2  # noqa: E402

INDIAN_PINES = np.setdiff1d(np.arange(224), np.r_[0:4, 103:108, 149:163, 219])                 # 200 of 224
HYPERION = np.r_[8:57, 77:224]                                                                   # 196 of 242
WORKLOADS = {"paviau_bip_u16": (610, 340, 224, INDIAN_PINES, 9, "bip", np.uint16),
             "paviau_bil_i16": (610, 340, 224, INDIAN_PINES, 9, "bil", np.int16),
             "hyperion_bil_i16": (1000, 256, 242, HYPERION, 12, "bil", np.int16),
             "honghu_bil_u16": (940, 475, 300, np.r_[0:150, 180:300], 22, "bil", np.uint16)}
AXIS = {"bip": 1, "bil": 1, "bsq": 0}                   # band axis of the layout tensors (BIP: [pixels, B])


def setup(R, C, B, nf, K, il, dt, dev, seed):
    cube = np.random.default_rng(seed).integers(1, 8001, (R, C, B)).astype(dt)
    raw = torch.from_numpy(layout(cube, il)).to(dev)
    torch.manual_seed(seed)
    net = BaseNet2(nf, 0, K).to(dev).eval()
    return raw, net


def band_workloads(a, dev, res):
    for name, (R, C, B, bands, K, il, dt) in WORKLOADS.items():
        bands = bands.astype(np.int32)
        raw, net = setup(R, C, B, bands.size, K, il, dt, dev, B)
        sel = torch.from_numpy(bands.astype(np.int64)).to(dev)
        compact = raw.index_select(AXIS[il], sel).contiguous()
        pp = preprocess.fit(compact.view(R, C, -1) if il == "bip" else compact, 60, interleave=il)
        sd = net.state_dict()
        folded0 = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
        folded = dict(folded0, bands=bands, raw_bands=B)
        packed = net.packed_weights(20)
        ws = ops.scene_workspace(R, C, bands.size, K, 20, dev)
        labs = {k: torch.empty(R * C, dtype=torch.uint8, device=dev)
                for k in ("selected", "compacted", "index_select_then_call")}
        call = lambda x, f, k: ops.scene_infer_raw(x, f, packed, K, C, 20, workspace=ws, labels=labs[k], interleave=il)
        runs = {"selected": lambda: call(raw, folded, "selected"),
                "compacted": lambda: call(compact, folded0, "compacted"),
                "index_select_then_call": lambda: call(raw.index_select(AXIS[il], sel).contiguous(), folded0,
                                                       "index_select_then_call")}
        t = timed_rounds(runs, a.rounds, a.seconds)
        torch.cuda.synchronize()
        med = {k: v["median_ms"] for k, v in t.items()}
        res[name] = {"scene": f"{R} x {C}, {B} raw bands ({np.dtype(dt).name} {il.upper()}), {bands.size} listed, {K} "
                              "classes, w = 20",
                     "dense_path": bool(bands.size <= 224),
                     "results": t,
                     "selected_over_compacted": round(med["selected"] / med["compacted"], 4),
                     "index_select_then_call_over_compacted": round(med["index_select_then_call"] / med["compacted"], 4),
                     "labels_equal": bool(torch.equal(labs["selected"], labs["compacted"])
                                          and torch.equal(labs["selected"], labs["index_select_then_call"]))}
        print(name, med, res[name]["labels_equal"], flush=True)
        del runs, ws, compact
        torch.cuda.empty_cache()


def load(path):
    """A build of the library with the signatures of the symbols it has (the parent lacks the *_sel ones)."""
    lib = ctypes.CDLL(os.path.abspath(path))
    for name, (r, args) in _lib.SIGNATURES.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = r, args
    return lib


def ab_parent(a, dev, res):
    libs = {"parent": load(a.parent), "this": _lib.load()}
    stream = lambda: torch.cuda.current_stream().cuda_stream

    def ok(lib, rc):
        if rc != 0:
            raise RuntimeError(lib.cmlpl_last_error().decode())

    out = {}
    for name, (R, C, B, K, il) in {"paviau_bip_u16_103": (610, 340, 103, 9, "bip"),
                                   "honghu_bil_u16_270": (940, 475, 270, 22, "bil")}.items():
        raw, net = setup(R, C, B, B, K, il, np.uint16, dev, B)
        code = preprocess.INTERLEAVE[il]
        pp = preprocess.fit(raw.view(R, C, B) if il == "bip" else raw, 60, interleave=il)
        sd = net.state_dict()
        f = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
        packed = net.packed_weights(20)
        ws = ops.scene_workspace(R, C, B, K, 20, dev)
        labs = {k: torch.empty(R * C, dtype=torch.uint8, device=dev) for k in libs}
        valid = torch.empty(R * C, dtype=torch.uint8, device=dev)
        counts = torch.empty(B + 1, dtype=torch.int64, device=dev)
        mean = torch.empty(B, dtype=torch.float64, device=dev)
        gram = torch.empty(B, B, dtype=torch.float64, device=dev)
        rows, cols = (R * C, 1) if il == "bip" else (R, C)
        runs = {}
        for k, lib in libs.items():
            runs[f"scene_infer_raw/{k}"] = lambda lib=lib, k=k: ok(lib, lib.cmlpl_scene_infer_raw(
                raw.data_ptr(), code, R, C, 0, R, B, K, 20, 0, R, f["wf"].data_ptr(), f["bf"].data_ptr(), f["mu"].data_ptr(),
                f["inv_sigma"].data_ptr(), packed.data_ptr(), ws.data_ptr(), ws.numel(), labs[k].data_ptr(), None, stream()))
            if il == "bil":
                runs[f"valid_mask_u8/{k}"] = lambda lib=lib: ok(lib, lib.cmlpl_valid_mask_u8(
                    raw.data_ptr(), code, R, C, B, 0.0, valid.data_ptr(), counts.data_ptr(), counts.data_ptr() + 8,
                    stream()))
                runs[f"preprocess_fit_cube_f64/{k}"] = lambda lib=lib: ok(lib, lib.cmlpl_preprocess_fit_cube_f64(
                    raw.data_ptr(), code, rows, cols, B, mean.data_ptr(), gram.data_ptr(), stream()))
        t = timed_rounds(runs, a.rounds, a.seconds)
        torch.cuda.synchronize()
        med = {k: v["median_ms"] for k, v in t.items()}
        ratios = {e: round(med[f"{e}/this"] / med[f"{e}/parent"], 4) for e in {k.split("/")[0] for k in runs}}
        out[name] = {"scene": f"{R} x {C} x {B} uint16 {il.upper()}, {K} classes, w = 20", "results": t,
                     "this_over_parent": ratios, "labels_equal": bool(torch.equal(labs["this"], labs["parent"]))}
        print(name, med, ratios, out[name]["labels_equal"], flush=True)
        del runs, ws
        torch.cuda.empty_cache()
    res["entry_points_without_a_list_vs_parent"] = out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--parent", default=None, help="the parent commit's libcmlpl_sm100.so")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    res = {"card": card(), "method": f"CUDA events, one window of >= {a.seconds} s per timing, variants alternated over "
                                     f"{a.rounds} rounds after warm-up", "unit": "ms per whole-scene call"}
    band_workloads(a, dev, res)
    if a.parent:
        ab_parent(a, dev, res)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
