"""Scene inference beyond 16 classes: cmlpl_scene_infer and cmlpl_scene_infer_raw at 9, 16, 20 and 32 classes on a
PaviaU-shaped scene (610 x 340 x 103) and at 20 classes on a Houston-2018-shaped one (601 x 2384 x 48; the public scene
has 20 classes and 48 bands), w = 20 in path modes 1 (dense, exact compute sharing) and 0 (per-pixel kernels: for
17-32 classes the per-pixel patch CNN + CUDA-core heads on the cube path), and w = 11 at 20 classes.

Timing: CUDA events around back-to-back calls on preallocated workspaces, every shape warmed up first, each window at
least --window seconds.  Inputs are seeded random (values do not change the work).  At every timed size the script also
checks that mode 1 and mode 0 agree on every label whose mode-0 top-2 logit margin exceeds 2e-3 * max|logits|.
Prints one JSON line (with the card's nvidia-smi name and power limit); --out also writes it to a file.

    python scripts/bench_many_classes.py [--window 1.0] [--out profiles/many_classes.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cmlpl_b200 import _lib, ops, preprocess  # noqa: E402
from cmlpl_b200.tools.models import BaseNet2  # noqa: E402

BAR = 2e-3


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    row = out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else ""
    parts = [p.strip() for p in row.split(",")] if row else []
    return dict(zip(["name", "power_limit", "sm_max_clock"], parts)) if len(parts) == 3 else {"nvidia_smi": "unavailable"}


def time_calls(fn, window):
    """ms per call: warm-up, then back-to-back calls between two CUDA events until the window is at least `window` s"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter(); fn(); torch.cuda.synchronize()
    once = max(time.perf_counter() - t0, 1e-5)
    iters = max(5, int(np.ceil(window / once)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return ms / iters, iters, ms / 1e3


def agreement(lab1, lab0, log0):
    """labels of mode 1 vs mode 0 outside the near ties of mode 0's logits"""
    srt = torch.sort(log0, 1).values
    margin = srt[:, -1] - srt[:, -2]
    firm = margin > BAR * float(log0.abs().max())
    bad = int(((lab1 != lab0) & firm).sum())
    return {"firm_pixels": int(firm.sum()), "firm_disagreements": bad, "all_equal_frac": float((lab1 == lab0).float().mean())}


def run_case(name, R, C, B, K, w, window, dev):
    n = R * C
    gen = torch.Generator(device=dev); gen.manual_seed(R + C + B + K + w)
    cube = torch.randn((R, C, 60), device=dev, generator=gen)
    spectra = torch.randn((n, B), device=dev, generator=gen)
    raw = torch.randint(0, 8000, (n, B), device=dev, generator=gen, dtype=torch.int32).to(torch.float32)
    torch.manual_seed(K)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    packed = net.packed_weights(w)
    sd = {k: v.detach() for k, v in net.state_dict().items()}
    res = {"case": name, "R": R, "C": C, "B": B, "classes": K, "w": w, "pixels": n}
    # the raw entry point folds the 60-component PCA into conv0: it needs >= 60 bands (not the 48 of Houston 2018)
    entries = ("cube", "raw") if B >= 60 else ("cube",)
    if B >= 60:
        folded = preprocess.fit(raw, 60).folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    else:
        res["raw"] = "not run: the 60 PCA components need >= 60 bands"
    out = {}
    for mode in (1, 0):
        _lib.call("cmlpl_set_scene_path_mode", mode)
        try:
            ws = ops.scene_workspace(R, C, B, K, w, dev)
            lab = torch.empty(n, dtype=torch.uint8, device=dev)
            for entry in entries:
                if entry == "cube":
                    fn = lambda: ops.scene_infer(cube, spectra, packed, K, w, workspace=ws, labels=lab)
                    ref = lambda: ops.scene_infer(cube, spectra, packed, K, w, workspace=ws, want_logits=True)
                else:
                    fn = lambda: ops.scene_infer_raw(raw, folded, packed, K, C, w, workspace=ws, labels=lab)
                    ref = lambda: ops.scene_infer_raw(raw, folded, packed, K, C, w, workspace=ws, want_logits=True)
                ms, iters, secs = time_calls(fn, window)
                l, z = ref()
                out[(entry, mode)] = (l.clone(), z.clone())
                res[f"{entry}_mode{mode}_ms"] = round(ms, 4)
                res[f"{entry}_mode{mode}_Mpx_s"] = round(n / ms / 1e3, 2)
                res[f"{entry}_mode{mode}_window"] = {"iters": iters, "s": round(secs, 3)}
            del ws
        finally:
            _lib.call("cmlpl_set_scene_path_mode", 1)
    res["dense_path"] = dense_flag(R, C, B, K, w)
    for entry in entries:
        res[f"{entry}_mode1_over_mode0"] = round(res[f"{entry}_mode0_ms"] / res[f"{entry}_mode1_ms"], 2)
        l1, _ = out[(entry, 1)]
        l0, z0 = out[(entry, 0)]
        res[f"{entry}_agreement"] = agreement(l1, l0, z0)
    torch.cuda.empty_cache()
    return res


def dense_flag(R, C, B, K, w):
    off = (ctypes.c_size_t * 12)()
    _lib.call("cmlpl_scene_workspace_layout", R, C, B, K, w, off)
    return int(off[11])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window (>= 1 s)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    cases = [("PaviaU", 610, 340, 103, K, 20) for K in (9, 16, 20, 32)]
    cases += [("Houston-2018-shaped", 601, 2384, 48, 20, 20), ("PaviaU w11", 610, 340, 103, 20, 11)]
    results = [run_case(*c, max(args.window, 1.0), dev) for c in cases]
    for r in results:
        print(json.dumps(r), file=sys.stderr)
    ok = all(r[f"{e}_agreement"]["firm_disagreements"] == 0 for r in results for e in ("cube", "raw") if f"{e}_agreement" in r)
    line = {"script": "scripts/bench_many_classes.py", "gpu": gpu_info(), "torch": torch.__version__,
            "timing": "CUDA events, back-to-back calls on a preallocated workspace, warmed up, windows >= 1 s",
            "labels_agree_outside_near_ties": ok, "results": results}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
