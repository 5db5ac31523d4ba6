"""Spectra beyond 256 bands: time the fused training step and raw-cube scene inference (GPU only; CUDA events).

In one session, alternating the variants round by round:
  * the fused step (cmlpl_train_step, cube mode with device Philox noise / dropout) replayed from its CUDA graph at
    103 / 256 / 270 / 425 bands, at w = 20 and w = 11 (128 labelled + 128 unlabelled rows, 9 classes, on a PaviaU-sized
    random PCA cube);
  * cmlpl_scene_infer_raw (uint16 raw cube) against cmlpl_scene_infer (PCA cube + z-scored spectra, as preprocess.apply
    makes them) on a WHU-Hi-HongHu-shaped scene, 940 x 475 x 270 with 22 classes, w = 20.  Both take the per-pixel path
    with the CUDA-core spectral head at 270 bands.
Then, in a separate profiled pass (torch.profiler, CUDA activities), the device time of every kernel of one call of
each entry point, which gives the raw conv0 stage (conv0_tc_sliced_kernel) on its own.  The scene inputs are seeded
random values: they do not change the work.  Each timing is one window of >= --seconds of back-to-back calls after
warm-up.  The card's name and power limit are read in the same run.

    python scripts/bench_wide_bands.py --out profiles/wide_bands.json
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cmlpl_b200 import _lib, ops, preprocess  # noqa: E402
from cmlpl_b200.fused_step import FusedMutualStep  # noqa: E402
from cmlpl_b200.tools.models import BaseNet2  # noqa: E402

R, C, BS, K_STEP = 610, 340, 128, 9
SCENE = (940, 475, 270, 22)              # WHU-Hi-HongHu


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    row = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [p.strip() for p in row.split(",")] if row else []
    if len(parts) == 3:
        return dict(zip(["name", "power_limit", "sm_max_clock"], parts))
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": "unavailable"}


def window(fn, seconds):
    """Mean ms per call over one window of >= `seconds` (count sized from a short probe)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        fn()
    e1.record()
    torch.cuda.synchronize()
    n = max(5, math.ceil(seconds * 1000.0 / (e0.elapsed_time(e1) / 3)))
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def fused_runner(dev, cube, spectra, B, w):
    torch.manual_seed(0)
    nets = [BaseNet2(B, 0.8, K_STEP, w=w).to(dev) for _ in range(2)]
    fs = FusedMutualStep(nets[0], nets[1], bs=BS, btu=BS, use_graph=True, thr=0.5)
    g = torch.Generator(device=dev).manual_seed(B * 100 + w)
    pix = torch.randint(0, R * C, (2 * BS,), device=dev, generator=g)
    labels = torch.randint(0, K_STEP, (BS,), device=dev, generator=g)
    it = [0]

    def step():
        fs.step(labels, 1, it[0] % 5, cube=cube, pix=pix, spectra=spectra)
        it[0] += 1
    return step


def timed_rounds(runners, rounds, seconds):
    for fn in runners.values():                                # warm-up: graph capture, module loads
        for _ in range(5):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in runners}
    for _ in range(rounds):
        for k, fn in runners.items():
            times[k].append(window(fn, seconds))
    return {k: {"ms": [round(t, 4) for t, _ in v], "calls": [n for _, n in v],
                "median_ms": round(sorted(t for t, _ in v)[len(v) // 2], 4)} for k, v in times.items()}


def kernel_times(fn, reps=5):
    """Device ms per call of every kernel of `fn`, from torch.profiler (CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0)
        if t > 0 and e.count >= reps:
            out[e.key[:90]] = round(t / 1e3 / reps, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


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

    # ---- the fused step, graph replay
    g = torch.Generator(device=dev).manual_seed(1)
    cube = torch.randn(R, C, 60, device=dev, generator=g)
    spectra = {B: torch.randn(R * C, B, device=dev, generator=g) for B in (103, 256, 270, 425)}
    runners = {f"B{B}_w{w}": fused_runner(dev, cube, spectra[B], B, w) for w in (20, 11) for B in (103, 256, 270, 425)}
    res["train_step"] = {"rows": f"{BS} + {BS}", "classes": K_STEP, "scene": f"{R} x {C} x 60 random PCA cube",
                         "what": "cmlpl_train_step replayed from its CUDA graph, ms per step",
                         "results": timed_rounds(runners, a.rounds, a.seconds)}
    print("train_step", {k: v["median_ms"] for k, v in res["train_step"]["results"].items()}, flush=True)
    del runners, spectra, cube
    torch.cuda.empty_cache()

    # ---- scene inference, raw against cube entry point
    SR, SC, B, K = SCENE
    raw = torch.from_numpy(np.random.default_rng(2).integers(0, 8000, (SR * SC, B), dtype=np.uint16)).to(dev)
    pp = preprocess.fit(raw, 60)
    pca, spec = preprocess.apply(raw, pp)
    pca = pca.view(SR, SC, 60)
    torch.manual_seed(3)
    net = BaseNet2(B, 0, K).to(dev).eval()
    sd = net.state_dict()
    packed = net.packed_weights(20)
    folded = pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev)
    ws = ops.scene_workspace(SR, SC, B, K, 20, dev)
    labels_raw = torch.empty(SR * SC, dtype=torch.uint8, device=dev)
    labels_cube = torch.empty(SR * SC, dtype=torch.uint8, device=dev)
    calls = {"scene_infer_raw": lambda: ops.scene_infer_raw(raw, folded, packed, K, SC, 20, workspace=ws, labels=labels_raw),
             "scene_infer": lambda: ops.scene_infer(pca, spec, packed, K, 20, workspace=ws, labels=labels_cube)}
    scene = {"scene": f"{SR} x {SC} x {B} (WHU-Hi-HongHu shape), {K} classes, w = 20, uint16 raw cube",
             "what": "one whole-scene call, ms", "results": timed_rounds(calls, a.rounds, a.seconds)}
    torch.cuda.synchronize()
    scene["label_agreement_raw_vs_cube"] = round(float((labels_raw == labels_cube).float().mean()), 6)
    scene["kernels_ms_per_call"] = {k: kernel_times(fn) for k, fn in calls.items()}
    res["scene"] = scene
    print("scene", {k: v["median_ms"] for k, v in scene["results"].items()}, flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
