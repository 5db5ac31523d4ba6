#!/usr/bin/env python
"""Headline benchmark: pixels/sec of full-scene inference on a synthetic scene of a BASELINE.json shape on N B200s of
one node, plus the train-step time (the second half of the BASELINE metric).

    python bench.py --gpus N --steps K --warmup W [--config c1|c2|c3|c4|c5]   # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...                   # the reference's own CPU path

Configs (BASELINE.json `configs`): c1 PaviaU-shaped 610x340x103 (default; the configuration the metric is quoted on),
c2 Indian-Pines-shaped 145x145x200 (train step + inference), c3 Salinas-shaped 512x217x204 (+ the contrastive-loss stress
at 1024 rows), c4 Houston-shaped 349x1905x144 (band-sharded), c5 8192x8192x224 with 11x11 patches (band-sharded).

One "step" = one pass of the hot path over the whole scene: conv0 map -> spectral branch -> scene-level tcgen05
conv1+pool / conv2 (exact compute sharing) -> pool + classifier partial maps -> sum head + argmax (+ label-map all-gather
and confusion all-reduce when N > 1).  `value` is device-resident throughput; `e2e` goes through the public call with
the RAW uint16 cube in pinned HOST memory (H2D + preprocessing folded into the first kernels + D2H of the label map
inside the timed region).
Multi-GPU: the scene is cut into N row bands (STRONG scaling: rank g infers ceil(R/N) rows + a read-only 19-row halo,
no data-path collective); the weak-scaling number (scene stacked N times) is reported beside it.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "c1": dict(name="PaviaU", key="paviau", R=610, C=340, B=103, K=9, w=20, baseline="configs[0]"),
    "c2": dict(name="Indian-Pines", key="indian_pines", R=145, C=145, B=200, K=16, w=20, baseline="configs[1]"),
    "c3": dict(name="Salinas", key="salinas", R=512, C=217, B=204, K=16, w=20, baseline="configs[2]"),
    "c4": dict(name="Houston-2013", key="houston", R=349, C=1905, B=144, K=15, w=20, baseline="configs[3]"),
    "c5": dict(name="AVIRIS-NG-scale", key=None, R=8192, C=8192, B=224, K=16, w=11, baseline="configs[4]"),
}


def flop_per_px(cfg):
    """SURVEY 8(d): the reference's per-patch arithmetic, 2 * MAC of tools/models.py:130-152."""
    w, B, K = cfg["w"], cfg["B"], cfg["K"]
    h1, h2 = w, w // 2
    p = (h2 // 2) ** 2
    conv0, conv1, conv2 = w * w * 60 * 64, h1 * h1 * 576 * 64, h2 * h2 * 576 * 64
    return {"conv0": 2 * conv0, "conv1": 2 * conv1, "conv2": 2 * conv2, "spectral": 2 * 1024 * B,
            "classifier": 2 * (64 * p + 1024) * K,
            "all": 2 * (conv0 + conv1 + conv2 + 1024 * B + (64 * p + 1024) * K)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        z = json.load(open(p))
        return {"hbm": z["hbm_gbs"], "tf_burst": z["bf16_tflops"], "tf_sustained": z["bf16_tflops_sustained"],
                "src": "measured"}
    return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


# ------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm = [float(r[1]) for r in rows if len(r) >= 8]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 8 for i in range(4) if r[4 + i].strip() == "Active"})
        busy = [s for s in sm if s > 0.5 * max(sm)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(rows[0][2]), "reasons": reasons,
                "samples": len(sm), "power_w_max": max(float(r[3]) for r in rows if len(r) >= 8)}


def workload_config(cfg, n_gpus):
    """Identical for both arms (the driver compares the two lines' `config`)."""
    R, C, B, K, w = cfg["R"], cfg["C"], cfg["B"], cfg["K"], cfg["w"]
    per = -(-R // n_gpus)
    return {"workload": f"{cfg['name']}-shaped synthetic scene {R}x{C}x{B}, {K} classes, w={w}, n_PC=60 "
                        f"(BASELINE.json {cfg['baseline']}); random-init BaseNet2 (seed 1088), synthetic cube seed 1088",
            "scene_rows": R, "scene_cols": C, "bands": B, "classes": K, "patch": w, "pixels_per_step": R * C,
            "parallelism": f"row bands x{n_gpus} (strong: the {R}-row scene is cut into bands of {per} rows + "
                           f"{w - 1} halo rows; scaling_weak holds the stacked-scene number)",
            "l2_policy": "the per-step working set (inputs + the intermediates of every stage, > 1 GB at PaviaU size) "
                         "exceeds the 126 MB L2; no explicit flush",
            "prewarm": "every timed loop is preceded by >= 1 s (first loop) / 0.2 s of untimed steps at full load and the W "
                       "warm-up steps, so clocks and the power state are steady"}


# ------------------------------------------------------------------ CPU arm
def _ref_dir():
    if os.environ.get("CMLPL_BENCH_NO_REF"):       # force the oracle-port fallback (tests)
        return None
    d = os.path.join(ROOT, "baseline", "_ref")
    need = ("hsi_loader.py", os.path.join("tools", "hyper_tools.py"), os.path.join("tools", "models.py"))
    return d if all(os.path.exists(os.path.join(d, f)) for f in need) else None


def cpu_port_pass(cube_pca, spectra, sd, rows, threads, w):
    """Oracle PORT of the reference's test_whole path on host cores for scene rows [rows[0], rows[1]): per-pixel window
    copy out of the mirror-padded cube (hyper_tools.py:231-243), batches of 512 through BaseNet2 in fp32
    (models.py:130-152), argmax (hyper_tools.py:426).  Returns (seconds, pixels)."""
    from oracle import cmlpl_oracle as O          # CPU baseline leg only

    torch.set_num_threads(threads)
    R, C, F = cube_pca.shape
    hw = w // 2
    Xm = O.mirrow_cut(cube_pca, hw)               # one-off for the scene: not timed (amortised over all pixels)
    r0, r1 = rows
    n = (r1 - r0) * C
    t0 = time.perf_counter()
    XP = np.zeros((n, w, w, F), dtype=np.float32)
    k = 0
    for r in range(r0, r1):
        for c in range(C):
            XP[k] = Xm[r:r + w, c:c + w, :]
            k += 1
    XP = np.moveaxis(XP, 3, 1).astype(np.float32)
    Xs = spectra[r0 * C:r1 * C]
    out = []
    with torch.no_grad():
        for s in range(0, n, 512):
            xp = torch.from_numpy(XP[s:s + 512].astype("float32").copy())
            xs = torch.from_numpy(Xs[s:s + 512].astype("float32").copy())
            lo, _ = O.basenet2_forward(sd, xp, xs)
            out.append(torch.max(lo, 1)[1].numpy())
    np.concatenate(out)
    return time.perf_counter() - t0, n


class StockReference:
    """The UNMODIFIED reference (files under baseline/_ref, copied there by __graft_entry__.build() in the build
    container): HSIDataSet('wholeset') + DataLoader(batch_size=512, num_workers=1) + tools.hyper_tools.test_whole on a
    row band of the scene whose XP.npy the reference's own ExtractPatches wrote.  CPU only (``.cuda()`` -> identity)."""

    def __init__(self, ref_dir, cfg, cube_pca, spectra, gt, rows):
        from oracle import ref_shims
        ref_shims.REFERENCE_ROOT = ref_dir
        ref_shims.install()
        import hsi_loader as RL
        from tools import hyper_tools as RH
        from tools import models as RM
        self.RL, self.RH = RL, RH
        R, C, B, K = cfg["R"], cfg["C"], cfg["B"], cfg["K"]
        r0, r1 = rows
        self.n = (r1 - r0) * C
        self.tmp = tempfile.mkdtemp(prefix="cmlpl_ref_")
        d = os.path.join(self.tmp, "dataset", "PaviaU")
        os.makedirs(d)
        hw = cfg["w"] // 2
        lo, hi = max(0, r0 - hw), min(R, r1 + hw)
        # the reference's own patch extraction on the band (+ halo rows), then the band's pixels
        XP = RH.ExtractPatches(cube_pca[lo:hi].astype(np.float64), cfg["w"])
        sel = np.arange((r0 - lo) * C, (r1 - lo) * C)
        np.save(os.path.join(d, "XP.npy"), np.ascontiguousarray(XP[sel]))
        np.save(os.path.join(d, "X.npy"), spectra[r0 * C:r1 * C].astype(np.float64))
        np.save(os.path.join(d, "Y.npy"), gt.reshape(-1)[r0 * C:r1 * C])
        for f in ("train_array", "test_array", "unlabel_array"):
            np.save(os.path.join(d, f + ".npy"), np.arange(8))
        torch.manual_seed(1088)
        self.model = RM.BaseNet2(num_features=B, dropout=0, num_classes=K)
        self.cwd = os.getcwd()

    def one_pass(self):
        from torch.utils import data
        os.chdir(self.tmp)
        try:
            t0 = time.perf_counter()
            ds = self.RL.HSIDataSet(1, setindex="wholeset")              # np.load of XP.npy included, like train.py:112
            loader = data.DataLoader(ds, batch_size=512, shuffle=False, num_workers=1)
            pred = self.RH.test_whole(self.model, loader, print_per_batches=10 ** 9)
            assert pred.shape[0] == self.n
            return time.perf_counter() - t0, self.n
        finally:
            os.chdir(self.cwd)


def run_reference_arm(args, cfg, scene):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cube_pca, spectra, gt = scene
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    R, C = cfg["R"], cfg["C"]
    rows_per_step = max(1, 10200 // C)             # ~10 k px per step: amortises the DataLoader worker start-up
    ref_dir = _ref_dir() if cfg["w"] == 20 else None
    times, npx = [], 0
    if ref_dir:
        kind = "reference"
        r0 = min(37, R - rows_per_step)
        stock = StockReference(ref_dir, cfg, cube_pca, spectra, gt, (r0, r0 + rows_per_step))
        for i in range(args.warmup + args.steps):
            dt, npx = stock.one_pass()
            if i >= args.warmup:
                times.append(dt)
        sample = (f"{rows_per_step} rows x {C} cols = {npx} px per step through the UNMODIFIED reference (baseline/_ref): "
                  "HSIDataSet('wholeset') np.load of XP.npy + DataLoader(bs 512, num_workers=1) + tools.hyper_tools.test_whole "
                  "on CPU; XP.npy written beforehand by the reference's ExtractPatches (not timed)")
    else:
        kind = "port"
        from oracle import cmlpl_oracle as O
        torch.manual_seed(1088)
        p = ((cfg["w"] // 2) // 2) ** 2
        sd = O.basenet2_init(cfg["B"], cfg["K"], conv_feat=64 * p)
        for i in range(args.warmup + args.steps):
            r0 = (37 + i * rows_per_step) % max(1, R - rows_per_step)
            dt, npx = cpu_port_pass(cube_pca, spectra, sd, (r0, r0 + rows_per_step), threads, cfg["w"])
            if i >= args.warmup:
                times.append(dt)
        sample = (f"{rows_per_step} rows x {C} cols = {npx} px per step through the oracle PORT of the ExtractPatches loop + "
                  "BaseNet2 fp32 (bs 512) + argmax (baseline/_ref not present)")
    ms = 1e3 * float(np.mean(times))
    val = npx / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "pixels/sec full-scene inference", "value": val, "unit": "pixels/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, args.gpus),
        "cpu_baseline": {"value": val, "unit": "pixels/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "pixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ helpers of the GPU arm
def make_timed(world, dev, dist):
    state = {"first": True}

    def timed(fn, steps, warmup):
        # clocks ramp from idle and the power state settles over the first second of load: hold the load before timing
        # (a COUNT agreed between the ranks, never a per-rank clock: the steps contain collectives)
        target = 1.0 if state["first"] else 0.2
        state["first"] = False
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        est = max((time.perf_counter() - t0) / 5, 1e-5)
        n_pre = torch.tensor([min(int(math.ceil(target / est)), 20000)], device=dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(n_pre, op=dist.ReduceOp.MAX)
        for _ in range(int(n_pre.item()) + warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    return timed


def dump_outputs(path, outputs, limit=64 << 20):
    """Write every output as <path>/<name>.npy in float32 (float64 stays float64).  An array larger than its equal share
    of half of `limit` bytes is replaced by a fixed, seeded sample of its elements, with their flat indices in
    <name>_index.npy, so the directory stays below `limit`."""
    os.makedirs(path, exist_ok=True)
    share = limit // (2 * max(1, len(outputs)))
    for name, a in outputs.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > share:
            idx = np.sort(np.random.default_rng(1088).choice(a.size, share // 16, replace=False))
            np.save(os.path.join(path, name + "_index.npy"), idx.astype(np.float64))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a)


def synthetic_scene(cfg):
    from cmlpl_b200 import synth
    return synth.preprocessed_scene(cfg["R"], cfg["C"], cfg["B"], cfg["K"], 60, 1088, return_raw=True)


def train_step_bench(cfg, dev, slab, spec_dev, truth, steps, outputs=None):
    """One mutual-learning step (train.py:149-278), 128 labelled + 128 unlabelled, dropout 0.8, noise 0.5:
    the fused tcgen05 step from a CUDA graph (inputs gathered from the cube inside the first kernel, Philox noise),
    the fp32 reference-precision path, and the oracle's ref_step on the host cores.  When `outputs` is a dict, the
    losses and both nets' parameters after the last timed fused step are stored in it."""
    from cmlpl_b200 import ops, train as T
    from cmlpl_b200.fused_step import FusedMutualStep
    from cmlpl_b200.tools.models import BaseNet2
    B, K = cfg["B"], cfg["K"]
    torch.manual_seed(1088)
    nets = [BaseNet2(B, 0.8, K).to(dev) for _ in range(2)]
    fs = FusedMutualStep(nets[0], nets[1], use_graph=True, thr=1.0)
    lab_idx = torch.nonzero(truth >= 0).flatten()
    li = lab_idx[torch.randint(0, lab_idx.numel(), (128,), device=dev)]
    ui = lab_idx[torch.randint(0, lab_idx.numel(), (128,), device=dev)]
    pix, labels = torch.cat([li, ui]).contiguous(), truth[li].contiguous()
    state = {"i": 0}

    def fused():
        fs.step(labels, 1, state["i"], cube=slab, pix=pix, spectra=spec_dev)
        state["i"] += 1

    for _ in range(5):
        fused()
    torch.cuda.synchronize()
    n = steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fused()
    e1.record()
    torch.cuda.synchronize()
    fused_ms = e0.elapsed_time(e1) / n
    if outputs is not None:
        outputs["train_losses"] = fs.hist.cpu().numpy()
        for e, net in enumerate(nets):
            outputs.update({f"train_net{e}.{k}": p.detach().cpu().numpy() for k, p in net.named_parameters()})
    # per phase (eager C calls on the same state; forward / losses / backward / Adam)
    io = fs._io(slab, None, spec_dev, None, None, None, None)
    st = torch.cuda.current_stream().cuda_stream
    phase_ms = {}
    for name, ph in (("forward", 1), ("losses", 2), ("backward", 4), ("adam", 8)):
        from cmlpl_b200 import _lib
        for _ in range(3):
            _lib.call("cmlpl_train_step", ctypes.byref(io), ph, ctypes.c_void_p(st))
        e0.record()
        for _ in range(50):
            _lib.call("cmlpl_train_step", ctypes.byref(io), ph, ctypes.c_void_p(st))
        e1.record()
        torch.cuda.synchronize()
        phase_ms[name] = e0.elapsed_time(e1) / 50
    # fp32 path (cmlpl_b200.train.mutual_step)
    targs = argparse.Namespace(temperature=0.3, thr=1.0, num_epochs=20, queue_batch=17, alpha=0.95, lr=5e-4,
                               labeled_batch_size=128, dropout=0.8, noise=0.5)
    tst = T.make_state(B, K, targs, dev)

    def fp32_step(i):
        def batch():
            z = torch.randn((256, 60, 20, 20), device=dev)
            xp = ops.patch_gather(slab, 20, idx=pix, noise=z, noise_scale=0.5)          # train.py:157,170 fused
            xs = spec_dev[pix] + torch.randn((256, B), device=dev) * 0.5                # train.py:158,171
            return xp, xs
        xb, sb = batch()
        xe, se = batch()
        T.mutual_step(tst, xb, sb, xe, se, labels, 1, i, targs)

    for i in range(3):
        fp32_step(i)
    torch.cuda.synchronize()
    e0.record()
    for i in range(10):
        fp32_step(3 + i)
    e1.record()
    torch.cuda.synchronize()
    fp32_ms = e0.elapsed_time(e1) / 10
    return fs, fused_ms, phase_ms, fp32_ms


def cpu_ref_step_ms(cfg, cube_pca, spectra, gt, threads):
    """The oracle's ref_step (pinned against the reference's train.main) on the host cores: one 128+128 step."""
    from oracle import cmlpl_oracle as O
    torch.set_num_threads(threads)
    B, K = cfg["B"], cfg["K"]
    g = torch.Generator().manual_seed(0)
    lab = np.nonzero(gt.reshape(-1) > 0)[0]
    li = lab[torch.randint(0, len(lab), (128,), generator=g).numpy()]
    ui = lab[torch.randint(0, len(lab), (128,), generator=g).numpy()]
    torch.manual_seed(1088)
    sa = O.StepArgs(num_epochs=20)
    st = O.make_state(O.basenet2_init(B, K), O.basenet2_init(B, K), K, sa)
    XP_l = torch.from_numpy(O.extract_patches_at(cube_pca, 20, li)); X_l = torch.from_numpy(spectra[li])
    XP_u = torch.from_numpy(O.extract_patches_at(cube_pca, 20, ui)); X_u = torch.from_numpy(spectra[ui])
    Y_l = torch.from_numpy(gt.reshape(-1)[li].astype(np.int64) - 1)
    ts = []
    for it in range(3):
        t0 = time.perf_counter()
        # the reference draws its noise on the CPU generator inside the step (train.py:157-182) and dropout in forward
        nz = {k: torch.randn(s) for k, s in (
            ("xp_l1", XP_l.shape), ("x_l1", X_l.shape), ("xp_l2", XP_l.shape), ("x_l2", X_l.shape),
            ("xp_u1", XP_u.shape), ("x_u1", X_u.shape), ("xp_u2", XP_u.shape), ("x_u2", X_u.shape))}
        masks = tuple(torch.nn.functional.dropout(torch.ones(256, 2624), 0.8, True) for _ in range(2))
        st.queue_ptr, st.queue_ptr1 = 0, 256
        O.ref_step(st, XP_l, X_l, Y_l, XP_u, X_u, nz, 1, it, sa, masks)
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


# ------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="cmlpl_b200", choices=["cmlpl_b200", "reference"])
    ap.add_argument("--config", default="c1", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    # defaults that finish within minutes: 300 steps of ~1 ms on the GPU arm (3 of ~0.2 s at c5), 5 steps of ~5 s on
    # the CPU arm
    if args.steps is None:
        args.steps = 5 if args.impl == "reference" else (3 if args.config == "c5" else 300)
    if args.warmup is None:
        args.warmup = 1 if args.impl == "reference" else 5
    if args.config == "c5":
        from scripts import bench_c5
        return bench_c5.main(args, cfg)
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    R, C, B, K, W = cfg["R"], cfg["C"], cfg["B"], cfg["K"], cfg["w"]

    t_data = time.time()
    scene4 = synthetic_scene(cfg)
    scene, raw_u16 = scene4[:3], scene4[3]
    t_data = time.time() - t_data
    if args.impl == "reference":
        return run_reference_arm(args, cfg, scene)

    import torch.distributed as dist
    from cmlpl_b200 import _lib, ops, parallel, preprocess
    from cmlpl_b200.tools.hyper_tools import StreamedRawScene
    from cmlpl_b200.tools.models import BaseNet2

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    _lib.require_device()
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local)
    cube_pca, spectra, gt = scene
    timed = make_timed(world, dev, dist)
    torch.manual_seed(1088)
    net = BaseNet2(num_features=B, dropout=0, num_classes=K).to(dev).eval()
    packed = net.packed_weights(W)
    truth_all = torch.from_numpy(gt.reshape(-1).astype(np.int64) - 1).to(dev)          # -1 = unlabelled (ignored)
    pp = preprocess.fit(torch.from_numpy(np.ascontiguousarray(raw_u16.reshape(-1, B))).to(dev), 60)
    folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)

    class Band:
        """Everything one rank needs for rows [r0, r1) of a scene with `scene_rows` rows (= R, or R*world stacked)."""

        def __init__(self, scene_rows):
            self.scene_rows = scene_rows
            self.r0, self.r1 = parallel.band_of(rank, world, scene_rows)
            self.s0, self.s1 = parallel.slab_of(self.r0, self.r1, scene_rows, W)
            rows = np.arange(self.s0, self.s1) % R
            self.n = (self.r1 - self.r0) * C
            self.slab = torch.from_numpy(np.ascontiguousarray(cube_pca[rows])).to(dev)
            band_rows = np.arange(self.r0, self.r1) % R
            self.spec = torch.from_numpy(np.ascontiguousarray(spectra.reshape(R, C, B)[band_rows].reshape(-1, B))).to(dev)
            self.truth = truth_all.view(R, C)[torch.from_numpy(band_rows).to(dev)].reshape(-1).contiguous()
            self.raw_host = torch.from_numpy(np.ascontiguousarray(raw_u16[rows].reshape(-1, B))).pin_memory()
            self.raw_dev = torch.empty_like(self.raw_host, device=dev)
            self.ws = ops.scene_workspace(self.r1 - self.r0, C, B, K, W, dev)
            self.gather = parallel.LabelGather(scene_rows, C, dev) if world > 1 else None
            self.exchange = parallel.SceneExchange(scene_rows, C, K, dev) if world > 1 else None
            self.labels = self.exchange.local_labels[: self.n] if world > 1 else torch.empty(self.n, dtype=torch.uint8, device=dev)
            self.map_host = torch.empty(scene_rows * C, dtype=torch.uint8).pin_memory() if world > 1 else None
            self.streamed = StreamedRawScene(pp, scene_rows, C, B, K, W, nsplit=1, row0=self.r0, rows=self.r1 - self.r0,
                                             device=dev)

        def step_device(self):
            ops.scene_infer(self.slab, self.spec, packed, K, W, band_row0=self.r0, band_rows=self.r1 - self.r0,
                            scene_rows=self.scene_rows, slab_row0=self.s0, workspace=self.ws, labels=self.labels)
            if world > 1:
                # label-map all-gather + confusion all-reduce as ONE collective (parallel.SceneExchange); the labels and
                # the counts are produced directly in its send buffer
                self.exchange.local_cm.zero_()
                ops.confusion(self.labels, self.truth, K, self.exchange.local_cm)
                self.result = self.exchange()

        def step_e2e(self):
            # the RAW uint16 band (+halo) in pinned host memory in, uint8 labels out (label map of the whole scene on
            # every rank when sharded); preprocessing folded into the first kernels
            if world > 1:
                lab = self.streamed(packed, self.raw_host, d2h=False, folded=folded)
                self.map_host.copy_(self.gather(lab), non_blocking=True)
            else:
                self.streamed(packed, self.raw_host, folded=folded)

        def step_h2d_only(self):
            self.raw_dev.copy_(self.raw_host, non_blocking=True)

    sampler = ClockSampler(local)
    sampler.start()
    band = Band(R)
    outputs = {} if args.dump_outputs and rank == 0 else None
    ms_dev = timed(band.step_device, args.steps, args.warmup)
    if outputs is not None:
        # the label map of the whole scene (and the confusion counts when sharded), as the last timed step left them
        if world > 1:
            outputs["labels"], outputs["confusion"] = (t.cpu().numpy() for t in band.result)
        else:
            outputs["labels"] = band.labels.cpu().numpy()
    ms_e2e = timed(band.step_e2e, args.steps, args.warmup)
    if outputs is not None:
        outputs["labels_e2e"] = (band.map_host if world > 1 else band.streamed.labels_host).numpy().copy()
    ms_h2d = timed(band.step_h2d_only, args.steps, args.warmup)
    # a fixed >= 1 s window next to the K-step number (VERDICT r1: a 20-step region is 20 ms)
    n_steady = max(args.steps, int(math.ceil(1000.0 / max(ms_dev, 1e-3))))
    ms_dev_steady = timed(band.step_device, n_steady, args.warmup)
    ms_e2e_steady = timed(band.step_e2e, max(args.steps, int(math.ceil(1000.0 / max(ms_e2e, 1e-3)))), args.warmup)
    weak = None
    if world > 1:
        wband = Band(R * world)
        weak = {"ms_per_step": timed(wband.step_device, args.steps, args.warmup),
                "e2e_ms_per_step": timed(wband.step_e2e, args.steps, args.warmup)}
        del wband

    # ---- per-kernel durations of the same step, CUDA events on the launching stream
    L = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    nbr, r0, s0, s1 = band.r1 - band.r0, band.r0, band.s0, band.s1
    off = (ctypes.c_size_t * 12)()          # f0pad, x16, h16, g, pmq, yq, lmap, p2, spe, hidden, total, tc
    _lib.call("cmlpl_scene_workspace_layout", nbr, C, B, K, W, off)
    assert off[10] == band.ws.numel() and off[11] == 1, "bench expects the tensor-core scene path"
    o_f0, o_x16, o_h16, o_g, o_pmq, o_yq, o_lmap = (band.ws.data_ptr() + off[i] for i in range(7))
    pk = packed.data_ptr()
    names = ["conv0_map", "spectral_logits", "conv1_pool", "conv2_scene", "pool2_cls", "head_sum"]
    NS = len(names)
    nrep = min(args.steps, 50)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(NS + 1)] for _ in range(nrep)]
    for it in range(args.warmup + nrep):
        e = ev[it - args.warmup] if it >= args.warmup else [None] * (NS + 1)
        if e[0]: e[0].record()
        _lib.call("cmlpl_conv0_map_f16", band.slab.data_ptr(), R, C, s0, s1 - s0, W, r0, nbr, pk, o_f0, st)
        if e[1]: e[1].record()
        _lib.call("cmlpl_spectral_logits_tc", band.spec.data_ptr(), band.n, B, K, W, pk, o_x16, o_h16, st)
        if e[2]: e[2].record()
        _lib.call("cmlpl_conv1_pool_planes_f16", o_f0, C, W, nbr, pk, o_pmq, st)
        if e[3]: e[3].record()
        _lib.call("cmlpl_conv2_scene_f16", o_pmq, C, W, nbr, pk, o_yq, st)
        if e[4]: e[4].record()
        _lib.call("cmlpl_pool2_cls_f16", o_yq, C, W, nbr, B, K, pk, o_lmap, st)
        if e[5]: e[5].record()
        _lib.call("cmlpl_head_sum_lmap", o_h16, o_lmap, C, nbr, B, K, W, pk, band.labels.data_ptr(), None, st)
        if e[6]: e[6].record()
    torch.cuda.synchronize()
    stage_ms = {names[i]: float(np.mean([e[i].elapsed_time(e[i + 1]) for e in ev])) for i in range(NS)}

    # ---- the HBM-bound kernel of the path: materialising patch gather (training batches / ExtractPatches)
    gather = None
    if world == 1 and band.n >= 16384 + 50000:
        ng = 16384
        gout = torch.empty((ng, 60, W, W), dtype=torch.float32, device=dev)
        gres = {}
        for gname, gidx in (("contiguous", torch.arange(50000, 50000 + ng, device=dev)),
                            ("random", torch.randperm(band.n, device=dev)[:ng].contiguous())):
            for _ in range(3):
                ops.patch_gather(band.slab, W, idx=gidx, out=gout)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            g0.record()
            for _ in range(20):
                ops.patch_gather(band.slab, W, idx=gidx, out=gout)
            g1.record()
            torch.cuda.synchronize()
            gres[gname] = g0.elapsed_time(g1) / 20
        gather = {"kernel": "patch_gather_reg_kernel (16384 raster-consecutive pixels = ExtractPatches over scene rows, "
                            "60x20x20 f32 each; output 1.57 GB > L2)",
                  "bound": "hbm", "ms": gres["contiguous"], "bytes_per_pixel": 96240, "ms_random_pixels": gres["random"]}
        del gout

    # ---- second half of the BASELINE metric: one mutual-learning train step (train.py:149-278), 128+128
    train = None
    if world == 1 and not args.no_train and args.config in ("c1", "c2", "c3"):
        fs, fused_ms, phase_ms, fp32_ms = train_step_bench(cfg, dev, band.slab, band.spec, band.truth, args.steps, outputs)
        train = {"fused_ms": fused_ms, "phase_ms": phase_ms, "fp32_ms": fp32_ms, "launches": fs.launches()}
    clocks = sampler.stop()

    # ---- config 3: the contrastive / bank losses at 1024 rows (SURVEY 8d "C3 loss stress")
    loss_stress = None
    if world == 1 and args.config == "c3":
        from scripts import bench_loss_stress
        loss_stress = bench_loss_stress.run(dev, K)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    fl = flop_per_px(cfg)
    px_step = R * C
    value = px_step / (ms_dev / 1e3)
    e2e_val = px_step / (ms_e2e / 1e3)
    # dominant kernel: conv2_scene (tensor-bound).  FLOPs it EXECUTES: 169 tap products (64x64 MACs) per plane position
    # over the 25 border classes; the reference's per-patch arithmetic for the same layer (SURVEY 8d) is reported next
    # to it and exceeds the hardware peak by the sharing factor.
    cnn_ms = stage_ms["conv2_scene"]
    qpos = 4 * ((nbr + W) // 2) * ((C + W) // 2)
    ppos = (nbr + W - 1) * (C + W - 1)
    exec_flop = {"conv0_map": ppos * 2 * 60 * 64, "spectral_logits": band.n * (2 * B * 1024 + 2 * 1024 * 16),
                 "conv1_pool": ppos * 9 * 2 * 64 * 64, "conv2_scene": qpos * 169 * 2 * 64 * 64,
                 "pool2_cls": qpos * 1024 * 64 * 2, "head_sum": band.n * 9 * 16}
    achieved = exec_flop["conv2_scene"] / (cnn_ms / 1e3) / 1e12
    traffic, stage_dram = None, None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp) and args.config == "c1" and world == 1:
        tj = json.load(open(tp))
        traffic = tj.get("conv2_scene_dram_bytes_per_launch")
        stage_dram = tj.get("stage_dram_bytes")
    launches_per_step = 7 + (1 if world > 1 else 0)
    line = {
        "metric": "pixels/sec full-scene inference", "value": value, "unit": "pixels/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None,
        "dtype": "f16 operands / f32 accumulate (tcgen05 kind::f16; same 11-bit significand as the TF32 the "
                 "reference's torch 1.8 GPU path used); fp32 elsewhere",
        "data": "synthetic", "config": workload_config(cfg, world),
        "clocks": clocks,
        "steady_state": {"ms_per_step": ms_dev_steady, "value": px_step / (ms_dev_steady / 1e3), "steps": n_steady,
                         "e2e_ms_per_step": ms_e2e_steady, "e2e_value": px_step / (ms_e2e_steady / 1e3),
                         "note": "same loops over a >= 1 s timed window"},
        "e2e": {"value": e2e_val, "unit": "pixels/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(band.raw_host.numel() * 2), "d2h_bytes_per_step": int(band.n if world == 1 else px_step),
                "h2d_only_ms": ms_h2d,
                "h2d_only_gbs": band.raw_host.numel() * 2 / (ms_h2d / 1e3) / 1e9,
                "input": "this rank's band (+halo) of the raw uint16 cube in pinned host memory (bytes are per rank); "
                         "preprocessing parameters fitted beforehand; z-score + PCA projection folded into conv0 and "
                         "into the fp16 conversion of the spectra (cmlpl_scene_infer_raw); h2d_only_* = the same copy "
                         "alone, all ranks at once (memcpy control)"},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": {"kernel": "conv2_scene_kernel (tcgen05 conv2 + residual + ReLU once per scene position in 25 patch-border "
                               "classes, parity planes, row-tap fusion into N=192/128 MMAs, TMA tile loads; the border halves "
                               "of the 2x2 pool are added in the epilogue, 9 half-pooled maps leave the kernel)", "bound": "tensor",
                     "achieved": achieved, "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["tf_burst"], "traffic": traffic,
                     "frac_burst": achieved / peaks["tf_burst"], "frac_sustained": achieved / peaks["tf_sustained"],
                     "peak_source": f"{peaks['src']} bf16 burst (per-stage CUDA events: the kernel is timed alone in a "
                                    "short loop at full clocks); frac_sustained uses the sustained figure",
                     "executed_flop_per_launch": exec_flop["conv2_scene"], "positions_per_launch": qpos,
                     "pixels_per_launch": band.n,
                     "algorithmic_flop_per_launch": band.n * fl["conv2"],
                     "algorithmic_frac": band.n * fl["conv2"] / (cnn_ms / 1e3) / 1e12 / peaks["tf_burst"],
                     "note": "exact compute sharing (SURVEY section 7 / 8-f3): conv1 and conv2 are evaluated once per scene "
                             "position in 9 / 25 patch-border classes instead of once per pixel patch. `achieved` counts the "
                             "FLOPs the kernel EXECUTES (169 tap products of 64x64 MACs per plane position); algorithmic_frac "
                             "is the same launch in the reference's per-patch arithmetic (SURVEY 8d) and exceeds 1 by the "
                             "sharing factor",
                     "kernel_ms": cnn_ms, "stage_ms": stage_ms,
                     "stage_note": "each stage launched and timed alone (CUDA events); in the step itself the spectral branch "
                                   "(fp16 conversion + spectral_logits) runs on a forked side stream beside conv0 / conv1_pool, "
                                   "so ms_per_step is below the sum of the stages",
                     "stage_executed_tflops": {k: exec_flop[k] / (stage_ms[k] / 1e3) / 1e12 for k in names},
                     "stage_dram_bytes": stage_dram,
                     "whole_step_executed_tflops": sum(exec_flop.values()) / (ms_dev / 1e3) / 1e12 * (1 if world == 1 else world),
                     "whole_step_executed_frac_burst": sum(exec_flop.values()) / (ms_dev / 1e3) / 1e12 / peaks["tf_burst"],
                     "whole_step_algorithmic_tflops": band.n * fl["all"] / (ms_dev / 1e3) / 1e12},
        "host_prep_s": t_data,
    }
    if weak is not None:
        line["scaling_weak"] = {"scene_rows": R * world, "pixels_per_step": px_step * world,
                                "ms_per_step": weak["ms_per_step"], "value": px_step * world / (weak["ms_per_step"] / 1e3),
                                "e2e_ms_per_step": weak["e2e_ms_per_step"],
                                "e2e_value": px_step * world / (weak["e2e_ms_per_step"] / 1e3)}
    if train is not None:
        flop_step = 2 * 256 * 3 * fl["all"]
        line["train_step_ms"] = train["fused_ms"]
        line["train_step_config"] = ("BaseNet2 x2 mutual-learning step (train.py:149-278), 128 labelled + 128 unlabelled, "
                                     "dropout 0.8, noise 0.5, smoothing branch on: cmlpl_train_step replayed from a CUDA graph "
                                     "(gather + Philox noise inside the first kernel; tcgen05 conv forward / dgrad / wgrad in "
                                     "fp16 operands, fp32 accumulate)")
        line["train_launches_per_step"] = train["launches"]
        line["train_step_fp32_ms"] = train["fp32_ms"]
        line["train_roofline"] = {"bound": "tensor", "achieved": flop_step / (train["fused_ms"] / 1e3) / 1e12,
                                  "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                                  "frac": flop_step / (train["fused_ms"] / 1e3) / 1e12 / peaks["tf_burst"],
                                  "algorithmic_flop_per_step": flop_step, "phase_ms": train["phase_ms"],
                                  "note": "SURVEY 8d accounting: 2 nets x 256 samples x 3 (fwd + dgrad + wgrad) x FLOP/px; "
                                          "62 GFLOP is ~40 us of tensor time, so the step is launch/latency-bound by "
                                          "construction (15 launches)"}
    if gather is not None:
        gather["achieved"] = 16384 * 96240 / (gather["ms"] / 1e3) / 1e9
        gather["peak"] = peaks["hbm"]
        gather["unit"] = "GB/s"
        gather["frac"] = gather["achieved"] / peaks["hbm"]
        gather["frac_random_pixels"] = 16384 * 96240 / (gather["ms_random_pixels"] / 1e3) / 1e9 / peaks["hbm"]
        line["aux_roofline"] = gather
    if loss_stress is not None:
        line["loss_stress"] = loss_stress
    if world == 1 and not args.no_cpu_baseline:
        from oracle import cmlpl_oracle as O      # cpu_baseline leg: the oracle port is the thing timed here
        torch.manual_seed(1088)
        sd = O.basenet2_init(B, K)
        threads = os.cpu_count() or 1
        tot_t, tot_n, rows = 0.0, 0, max(1, 2040 // C)
        rr = min(100, R // 2)
        while tot_t < 10.0 and rr + rows < R:
            dt, n = cpu_port_pass(cube_pca, spectra, sd, (rr, rr + rows), threads, W)
            tot_t += dt; tot_n += n; rr += rows
        line["cpu_baseline"] = {"value": tot_n / tot_t, "unit": "pixels/s", "cores": threads, "kind": "port",
                                "sample": f"{tot_n} px (rows of the same scene) in {tot_t:.1f} s: oracle port of the "
                                          "reference test_whole path (per-pixel patch loop + BaseNet2 fp32 bs 512 + argmax), "
                                          "torch threads = all host cores; `--impl reference` times the stock reference"}
        if train is not None:
            line["cpu_baseline"]["ref_step_ms"] = cpu_ref_step_ms(cfg, cube_pca, spectra, gt, threads)
            line["cpu_baseline"]["ref_step_note"] = ("oracle ref_step (restatement of train.py:150-272 pinned against the "
                                                     "reference's train.main), median of 3, noise + dropout draws included")
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
