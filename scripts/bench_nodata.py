"""No-data pixels: what a validity mask costs raw-cube scene inference and the device fit (GPU only; CUDA events).

In one session, alternating the variants round by round, on a PaviaU-shaped uint16 BIP scene (610 x 340 x 103, 9
classes: the dense path) and a WHU-Hi-HongHu-shaped uint16 BIL one (940 x 475 x 270, 22 classes: K-sliced conv0 and
the CUDA-core spectral head), w = 20, device-resident:
  * cmlpl_scene_infer_raw (unmasked), cmlpl_scene_infer_raw_masked with an all-valid mask, and the masked call on the
    same scene with a 25 % corner wedge of the rotated swath set to the fill value 0;
  * cmlpl_valid_mask_u8 on its own, against the HBM bound of one read of the cube plus the mask write (7.7 TB/s);
  * the device moments of the fit, unmasked against masked.
Then, in a separate profiled pass (torch.profiler, CUDA activities), the device time of every kernel of one call of each
scene variant.  The scenes are seeded random values in 1..8000 (no natural zeros): they do not change the work.  The
card's name and power limit are read in the same run.

    python scripts/bench_nodata.py --out profiles/nodata.json
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from bench_raw_layouts import layout  # noqa: E402
from bench_wide_bands import card, kernel_times, timed_rounds  # noqa: E402
from cmlpl_b200 import _lib, ops, preprocess  # noqa: E402
from cmlpl_b200.tools.models import BaseNet2  # noqa: E402

SCENES = {"paviau": (610, 340, 103, 9, "bip"), "honghu": (940, 475, 270, 22, "bil")}
HBM_BYTES_PER_S = 7.7e12


def wedge(R, C, frac=0.25):
    """the corner wedges outside a swath rotated by 20 degrees, widened until they hold `frac` of the pixels"""
    r, c = np.mgrid[0:R, 0:C]
    t = np.deg2rad(20.0)
    u = np.abs((c - (C - 1) / 2) * np.cos(t) - (r - (R - 1) / 2) * np.sin(t))
    return u > np.quantile(u, 1 - frac)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    stream = lambda: torch.cuda.current_stream().cuda_stream
    res = {"card": card(), "method": f"CUDA events, one window of >= {a.seconds} s per timing, variants alternated over "
                                     f"{a.rounds} rounds after warm-up; kernel times from torch.profiler in a "
                                     "separate pass", "unit": "ms"}
    for name, (R, C, B, K, il) in SCENES.items():
        cube = np.random.default_rng(B).integers(1, 8001, (R, C, B)).astype(np.uint16)
        nd = wedge(R, C)
        dirty = cube.copy()
        dirty[nd] = 0
        raw = torch.from_numpy(layout(cube, il)).to(dev)
        raw_w = torch.from_numpy(layout(dirty, il)).to(dev)
        code = preprocess.INTERLEAVE[il]
        pp = preprocess.fit(raw, 60, interleave=il)
        torch.manual_seed(3)
        net = BaseNet2(B, 0, K).to(dev).eval()
        sd = net.state_dict()
        packed = net.packed_weights(20)
        folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
        ws = ops.scene_workspace(R, C, B, K, 20, dev)
        ones = torch.ones((R, C), dtype=torch.uint8, device=dev)
        valid_w, n_valid, _ = preprocess.valid_mask(raw_w, 0, il, cols=C if il == "bip" else None)
        assert n_valid == R * C - int(nd.sum())
        labs = {k: torch.empty(R * C, dtype=torch.uint8, device=dev) for k in ("unmasked", "masked_all_valid", "masked_wedge")}
        runs = {"unmasked": lambda: ops.scene_infer_raw(raw, folded, packed, K, C, 20, workspace=ws, labels=labs["unmasked"],
                                                         interleave=il),
                "masked_all_valid": lambda: ops.scene_infer_raw(raw, folded, packed, K, C, 20, workspace=ws,
                                                                 labels=labs["masked_all_valid"], interleave=il, valid=ones),
                "masked_wedge": lambda: ops.scene_infer_raw(raw_w, folded, packed, K, C, 20, workspace=ws,
                                                             labels=labs["masked_wedge"], interleave=il, valid=valid_w)}
        vbuf = torch.empty((R, C), dtype=torch.uint8, device=dev)
        counts = torch.empty(B + 1, dtype=torch.int64, device=dev)
        runs["valid_mask"] = lambda: preprocess.mask_into(raw_w, 0, il, R, C, B, vbuf, counts)
        mean = torch.empty(B, dtype=torch.float64, device=dev)
        gram = torch.empty(B, B, dtype=torch.float64, device=dev)
        cnt = torch.empty(1, dtype=torch.int64, device=dev)
        rows, cols = (R * C, 1) if il == "bip" else (R, C)
        runs["fit_unmasked"] = lambda: _lib.call("cmlpl_preprocess_fit_cube_f64", raw.data_ptr(), code, rows, cols, B,
                                                 mean.data_ptr(), gram.data_ptr(), stream())
        runs["fit_masked"] = lambda: _lib.call("cmlpl_preprocess_fit_masked_f64", raw_w.data_ptr(), code, rows, cols, B,
                                               valid_w.data_ptr(), mean.data_ptr(), gram.data_ptr(), cnt.data_ptr(), stream())
        t = timed_rounds(runs, a.rounds, a.seconds)
        torch.cuda.synchronize()
        med = {k: v["median_ms"] for k, v in t.items()}
        hbm_ms = (R * C * B * 2 + R * C) / HBM_BYTES_PER_S * 1e3
        out = {"scene": f"{R} x {C} x {B} uint16 {il.upper()}, {K} classes, w = 20, device-resident raw cube; wedge "
                        f"{100 * nd.mean():.1f} % of the pixels",
               "what": "ms per call: one whole-scene scene_infer_raw call (unmasked / masked), cmlpl_valid_mask_u8, the "
                       "device moments of the fit",
               "results": t,
               "masked_all_valid_over_unmasked": round(med["masked_all_valid"] / med["unmasked"], 4),
               "masked_wedge_over_unmasked": round(med["masked_wedge"] / med["unmasked"], 4),
               "valid_mask_hbm_bound_ms": round(hbm_ms, 4),
               "valid_mask_share_of_hbm_bound": round(hbm_ms / med["valid_mask"], 3),
               "fit_masked_over_unmasked": round(med["fit_masked"] / med["fit_unmasked"], 4),
               "all_valid_labels_equal_unmasked": bool(torch.equal(labs["masked_all_valid"], labs["unmasked"])),
               "wedge_labels_nodata": bool(torch.all(labs["masked_wedge"][torch.from_numpy(nd.reshape(-1)).to(dev)]
                                                     == ops.NODATA_LABEL))}
        out["kernels_ms_per_call"] = {k: kernel_times(runs[k]) for k in ("unmasked", "masked_all_valid", "masked_wedge")}
        res[name] = out
        print(name, med, {k: v for k, v in out.items() if k.endswith(("unmasked", "bound", "equal_unmasked", "nodata"))},
              flush=True)
        del runs, ws
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
