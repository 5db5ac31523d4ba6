"""Time the mutual-learning step at w = 11 next to w = 20 (GPU only; CUDA events).

In one session, alternating the variants round by round:
  * the fused step (cmlpl_train_step, cube mode with device Philox noise / dropout) replayed from its CUDA graph, at
    w = 11 and w = 20;
  * the fp32 mutual_step at w = 11 (batches gathered on device like train.main's --fp32_step path).
128 labelled + 128 unlabelled rows on a PaviaU-sized random cube (610 x 340 x 60), at B = 103 / 9 classes and
B = 224 / 16 classes.  Each timing is one window of >= 1 s of back-to-back steps after warm-up.
    python scripts/time_train_w11.py --out profiles/train_w11.json
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cmlpl_b200 import _lib, ops, train as T  # noqa: E402
from cmlpl_b200.fused_step import FusedMutualStep  # noqa: E402
from cmlpl_b200.tools.models import BaseNet2  # noqa: E402

R, C, BS = 610, 340, 128


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def fused_runner(dev, cube, spectra, B, K, w):
    torch.manual_seed(0)
    nets = [BaseNet2(B, 0.8, K, w=w).to(dev) for _ in range(2)]
    fs = FusedMutualStep(nets[0], nets[1], bs=BS, btu=BS, use_graph=True, thr=0.5)
    g = torch.Generator(device=dev).manual_seed(w)
    pix = torch.randint(0, R * C, (2 * BS,), device=dev, generator=g)
    labels = torch.randint(0, K, (BS,), device=dev, generator=g)
    it = [0]

    def step():
        fs.step(labels, 1, it[0] % 5, cube=cube, pix=pix, spectra=spectra)
        it[0] += 1
    return step


def fp32_runner(dev, cube, spectra, B, K, w):
    args = argparse.Namespace(temperature=0.3, thr=0.5, num_epochs=20, queue_batch=17, alpha=0.95, lr=5e-4,
                              labeled_batch_size=BS, dropout=0.8, noise=0.5)
    torch.manual_seed(0)
    st = T.make_state(B, K, args, dev, w=w)
    g = torch.Generator(device=dev).manual_seed(w + 1)
    Y = torch.randint(0, K, (BS,), device=dev, generator=g)
    it = [0]

    def batch(idx):
        z = torch.randn((idx.numel(), 60, w, w), device=dev)
        XP = ops.patch_gather(cube, w, idx=idx, noise=z, noise_scale=0.5, odd_mode=w % 2 == 1)
        return XP, spectra[idx] + torch.randn((idx.numel(), B), device=dev) * 0.5

    def step():
        idx = torch.randint(0, R * C, (2 * BS,), device=dev, generator=g)
        xb, sb = batch(idx)
        xe, se = batch(idx)
        T.mutual_step(st, xb, sb, xe, se, Y, 1, it[0] % 5, args)
        it[0] += 1
    return step


def window(step, seconds):
    """Mean ms per step over one window of >= `seconds` (count sized from a short probe)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        step()
    e1.record()
    torch.cuda.synchronize()
    n = max(10, math.ceil(seconds * 1000.0 / (e0.elapsed_time(e1) / 5)))
    e0.record()
    for _ in range(n):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1)
    cube = torch.randn(R, C, 60, device=dev, generator=g)
    res = {"card": card(), "rows": f"{BS} + {BS}", "scene": f"{R} x {C} x 60 random cube", "unit": "ms per step",
           "method": f"CUDA events, one window of >= {a.seconds} s per timing, variants alternated over {a.rounds} "
                     "rounds after warm-up", "results": {}}
    for B, K in ((103, 9), (224, 16)):
        spectra = torch.randn(R * C, B, device=dev, generator=g)
        runners = {"fused_w11_graph": fused_runner(dev, cube, spectra, B, K, 11),
                   "fused_w20_graph": fused_runner(dev, cube, spectra, B, K, 20),
                   "fp32_w11": fp32_runner(dev, cube, spectra, B, K, 11)}
        for step in runners.values():                          # warm-up: graph capture, module loads
            for _ in range(10):
                step()
        torch.cuda.synchronize()
        times = {k: [] for k in runners}
        for _ in range(a.rounds):
            for k, step in runners.items():
                times[k].append(window(step, a.seconds))
        key = f"B{B}_K{K}"
        res["results"][key] = {k: {"ms": [round(t, 4) for t, _ in v], "steps": [n for _, n in v],
                                   "median_ms": round(sorted(t for t, _ in v)[len(v) // 2], 4)} for k, v in times.items()}
        print(key, {k: v["median_ms"] for k, v in res["results"][key].items()}, flush=True)
        del runners
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
