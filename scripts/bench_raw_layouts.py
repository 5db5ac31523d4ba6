"""Raw cubes in BIP, BIL and BSQ and in uint16 / int16 / float32: time raw-cube scene inference (GPU only; CUDA events).

In one session, alternating the variants round by round:
  * device-resident cmlpl_scene_infer_raw for BIP / BIL / BSQ x uint16 / int16 on a PaviaU-shaped scene (610 x 340 x
    103, 9 classes: the dense path) and a WHU-Hi-HongHu-shaped one (940 x 475 x 270, 22 classes: K-sliced conv0 and
    the CUDA-core spectral head), w = 20;
  * end to end, StreamedRawScene (pinned host cube -> labels on the host, nsplit = 2) on the PaviaU shape for every
    layout in uint16, int16 and float32, next to the host-to-device copy of the same cube alone.
Then, in a separate profiled pass (torch.profiler, CUDA activities), the device time of every kernel of one
device-resident call of each variant, which gives conv0 and the spectral branch's input conversion on their own.
The scenes are seeded random values: they do not change the work.  The card's name and power limit are read in the
same run.

    python scripts/bench_raw_layouts.py --out profiles/raw_layouts.json
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
from bench_wide_bands import card, kernel_times, timed_rounds  # noqa: E402
from cmlpl_b200 import _lib, ops, preprocess  # noqa: E402
from cmlpl_b200.tools.hyper_tools import StreamedRawScene  # noqa: E402
from cmlpl_b200.tools.models import BaseNet2  # noqa: E402

SCENES = {"paviau": (610, 340, 103, 9), "honghu": (940, 475, 270, 22)}
DTYPES = {"u16": (torch.uint16, np.uint16), "i16": (torch.int16, np.int16), "f32": (torch.float32, np.float32)}


def layout(cube, il):
    """[R, C, B] numpy -> contiguous numpy array in the layout."""
    return np.ascontiguousarray({"bip": cube.reshape(-1, cube.shape[2]), "bil": cube.transpose(0, 2, 1),
                                 "bsq": cube.transpose(2, 0, 1)}[il])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    res = {"card": card(), "method": f"CUDA events, one window of >= {a.seconds} s per timing, variants alternated over "
                                     f"{a.rounds} rounds after warm-up; kernel times from torch.profiler in a "
                                     "separate pass", "unit": "ms"}
    for name, (R, C, B, K) in SCENES.items():
        cube = np.random.default_rng(B).integers(0, 8000, (R, C, B)).astype(np.uint16)
        pp = preprocess.fit(torch.from_numpy(layout(cube, "bip")).to(dev), 60)
        torch.manual_seed(3)
        net = BaseNet2(B, 0, K).to(dev).eval()
        sd = net.state_dict()
        packed = net.packed_weights(20)
        folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
        ws = ops.scene_workspace(R, C, B, K, 20, dev)
        labels = {}
        calls = {}
        for dt in ("u16", "i16"):
            for il in ("bip", "bil", "bsq"):
                raw = torch.from_numpy(layout(cube.astype(DTYPES[dt][1]), il)).to(dev)
                lab = labels[dt, il] = torch.empty(R * C, dtype=torch.uint8, device=dev)
                calls[f"{il}_{dt}"] = (lambda raw=raw, il=il, lab=lab: ops.scene_infer_raw(
                    raw, folded, packed, K, C, 20, workspace=ws, labels=lab, interleave=il))
        out = {"scene": f"{R} x {C} x {B}, {K} classes, w = 20, device-resident raw cube",
               "what": "one whole-scene cmlpl_scene_infer_raw call, ms", "results": timed_rounds(calls, a.rounds, a.seconds)}
        torch.cuda.synchronize()
        ref = labels["u16", "bip"]
        out["labels_equal_to_bip_u16"] = {f"{il}_{dt}": bool(torch.equal(v, ref)) for (dt, il), v in labels.items()}
        out["kernels_ms_per_call"] = {k: kernel_times(fn) for k, fn in calls.items()}
        res[name] = out
        print(name, {k: v["median_ms"] for k, v in out["results"].items()}, flush=True)
        del calls, labels, ws
        torch.cuda.empty_cache()

    # ---- end to end from pinned host memory, PaviaU shape
    R, C, B, K = SCENES["paviau"]
    cube = np.random.default_rng(B).integers(0, 8000, (R, C, B)).astype(np.uint16)
    pp = preprocess.fit(torch.from_numpy(layout(cube, "bip")).to(dev), 60)
    torch.manual_seed(3)
    net = BaseNet2(B, 0, K).to(dev).eval()
    sd = net.state_dict()
    packed = net.packed_weights(20)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    runs, nbytes = {}, {}
    for dt, (tdt, ndt) in DTYPES.items():
        for il in ("bip", "bil", "bsq"):
            host = torch.from_numpy(layout(cube.astype(ndt), il)).pin_memory()
            st = StreamedRawScene(pp, R, C, B, K, 20, nsplit=2, raw_dtype=tdt, interleave=il)
            runs[f"e2e_{il}_{dt}"] = (lambda st=st, host=host: (st(packed, host, folded=folded), st.wait()))
            dst = torch.empty(host.shape, dtype=tdt, device=dev)
            if il == "bip":
                runs[f"h2d_only_{dt}"] = (lambda dst=dst, host=host: dst.copy_(host, non_blocking=True))
            runs[f"e2e_{il}_{dt}"]()
            nbytes[f"{il}_{dt}"] = st.h2d_bytes
    e2e = {"scene": f"{R} x {C} x {B}, {K} classes, w = 20, pinned host raw cube, StreamedRawScene nsplit = 2",
           "what": "one call including the host-to-device copy and the labels back on the host, ms; h2d_only_* is the "
                   "copy of the same cube alone", "h2d_bytes": nbytes, "results": timed_rounds(runs, a.rounds, a.seconds)}
    res["e2e_paviau"] = e2e
    print("e2e", {k: v["median_ms"] for k, v in e2e["results"].items()}, flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
