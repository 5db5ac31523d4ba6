"""BASELINE configs[4]: AVIRIS-NG-scale synthetic scene 8192 x 8192 x 224, 11 x 11 patches, 16 classes, full-scene
inference band-sharded over the ranks (python bench.py --config c5 [--gpus N]).

The scene (30 GB raw, 76 GB preprocessed) is never materialised: every rank walks its row band in sub-bands of
SUB rows whose inputs are ONE synthetic sub-band generated on the device from the seed (z-scored N(0,1) PCA cube +
spectra; the values do not influence the work done) and, for the end-to-end number, one pinned host sub-band of raw
uint16 that is copied for every sub-band (H2D bytes are counted in full).  Every pixel of the 8192 x 8192 scene is
inferred in every step by the scene-level kernels with exact compute sharing (the w = 11 classes and pooled cells are a
subset of the w = 20 ones: DESIGN 4.5): conv0 map || spectral branch -> conv1+pool -> conv2 -> pool/classifier maps -> head.
"""
import ctypes
import json
import os

import numpy as np
import torch

SUB = 512


def reference_arm(args, cfg):
    from bench import cpu_port_pass, workload_config
    from oracle import cmlpl_oracle as O
    R, C, B, K, W = cfg["R"], cfg["C"], cfg["B"], cfg["K"], cfg["w"]
    threads = os.cpu_count() or 1
    rng = np.random.default_rng(1088)
    rows = 1
    cube = rng.standard_normal((rows + 10, C, 60)).astype(np.float32)
    spectra = rng.standard_normal(((rows + 10) * C, B)).astype(np.float32)
    torch.manual_seed(1088)
    sd = O.basenet2_init(B, K, conv_feat=256)
    ts, n = [], 0
    for i in range(args.warmup + args.steps):
        dt, n = cpu_port_pass(cube, spectra, sd, (5, 5 + rows), threads, W)
        if i >= args.warmup:
            ts.append(dt)
    ms = 1e3 * float(np.mean(ts))
    val = n / (ms / 1e3)
    print(json.dumps({"impl": "reference", "metric": "pixels/sec full-scene inference", "value": val, "unit": "pixels/s",
                      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                      "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": workload_config(cfg, args.gpus),
                      "cpu_baseline": {"value": val, "unit": "pixels/s", "cores": threads, "kind": "port",
                                       "sample": f"{n} px (one scene row) per step through the oracle port (11x11 windows, "
                                                 "1280-input classifier: the reference's BaseNet2 cannot run w=11)"},
                      "e2e": {"value": val, "unit": "pixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def main(args, cfg):
    import torch.distributed as dist
    from bench import ClockSampler, dump_outputs, flop_per_px, measured_peaks, workload_config
    R, C, B, K, W = cfg["R"], cfg["C"], cfg["B"], cfg["K"], cfg["w"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, cfg)
        return
    from cmlpl_b200 import _lib, ops, parallel, preprocess
    from cmlpl_b200.tools.models import BaseNet2
    args.warmup = min(args.warmup, 1)
    torch.cuda.set_device(local)
    _lib.require_device()
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=300))
    dev = torch.device("cuda", local)
    torch.manual_seed(1088)
    net = BaseNet2(B, 0, K, w=W).to(dev).eval()
    packed = net.packed_weights(W)
    r0, r1 = parallel.band_of(rank, world, R)
    g = torch.Generator(device=dev).manual_seed(1088 + rank)
    hw = W // 2
    slab = torch.randn((SUB + 2 * hw, C, 60), device=dev, generator=g)
    spec = torch.randn((SUB * C, B), device=dev, generator=g)
    raw_host = torch.randint(0, 8000, ((SUB + 2 * hw) * C, B), dtype=torch.int32).to(torch.uint16).pin_memory()
    raw2 = [torch.empty_like(raw_host, device=dev) for _ in range(2)]
    # preprocessing parameters of a PaviaU-like dynamic range (the values are irrelevant for the work done)
    U = np.linalg.qr(np.random.default_rng(0).standard_normal((B, 60)))[0]
    pp = preprocess.Preproc(mu=np.full(B, 4000.0), sigma=np.full(B, 2300.0), U=U, pca_mu=np.zeros(60),
                            pca_sigma=np.full(60, 2300.0))
    folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    ws = ops.scene_workspace(SUB, C, B, K, W, dev)
    labels = torch.empty((r1 - r0) * C, dtype=torch.uint8, device=dev)
    gather = parallel.LabelGather(R, C, dev) if world > 1 else None
    copy_stream = torch.cuda.Stream(device=dev)
    subs = [(a, min(a + SUB, r1)) for a in range(r0, r1, SUB)]
    slabs = [parallel.slab_of(a, b, R, W) for a, b in subs]

    def step_device():
        for (a, b), (s0, s1) in zip(subs, slabs):
            ops.scene_infer(slab[: s1 - s0], spec[: (b - a) * C], packed, K, W, band_row0=a, band_rows=b - a, scene_rows=R,
                            slab_row0=s0, workspace=ws, labels=labels[(a - r0) * C:(b - r0) * C])
        if world > 1:
            gather(labels)

    ev = [torch.cuda.Event() for _ in range(2)]

    def step_e2e():
        main_s = torch.cuda.current_stream()
        for i, ((a, b), (s0, s1)) in enumerate(zip(subs, slabs)):
            buf = raw2[i & 1]
            copy_stream.wait_event(ev[i & 1])                       # the kernels that read this buffer two sub-bands ago
            with torch.cuda.stream(copy_stream):
                buf[: (s1 - s0) * C].copy_(raw_host[: (s1 - s0) * C], non_blocking=True)
                done = torch.cuda.Event()
                done.record(copy_stream)
            main_s.wait_event(done)
            ops.scene_infer_raw(buf[: (s1 - s0) * C], folded, packed, K, C, W, band_row0=a, band_rows=b - a, scene_rows=R,
                                slab_row0=s0, workspace=ws, labels=labels[(a - r0) * C:(b - r0) * C])
            ev[i & 1].record(main_s)
        if world > 1:
            gather(labels)
        labels[:1024].cpu()                                        # the 67 MB label map itself stays on the device

    def timed(fn, steps, warmup):
        for _ in range(max(warmup, 1)):
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
        ms = e0.elapsed_time(e1)
        if world > 1:
            dist.barrier()
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    sampler = ClockSampler(local)
    sampler.start()
    outputs = {} if args.dump_outputs and rank == 0 else None
    ms_dev = timed(step_device, args.steps, args.warmup)
    if outputs is not None:
        outputs["labels"] = (gather.out[:R * C] if world > 1 else labels).cpu().numpy()
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    if outputs is not None:
        outputs["labels_e2e"] = (gather.out[:R * C] if world > 1 else labels).cpu().numpy()
    # the dominant kernel alone, one sub-band (its input planes are in the workspace from the last step)
    off = (ctypes.c_size_t * 12)()
    _lib.call("cmlpl_scene_workspace_layout", SUB, C, B, K, W, off)
    st = torch.cuda.current_stream().cuda_stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        _lib.call("cmlpl_conv2_scene_f16", ws.data_ptr() + off[4], C, W, SUB, packed.data_ptr(), ws.data_ptr() + off[5], st)
    e0.record()
    for _ in range(5):
        _lib.call("cmlpl_conv2_scene_f16", ws.data_ptr() + off[4], C, W, SUB, packed.data_ptr(), ws.data_ptr() + off[5], st)
    e1.record()
    torch.cuda.synchronize()
    cnn_ms = e0.elapsed_time(e1) / 5
    clocks = sampler.stop()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    fl = flop_per_px(cfg)
    px = R * C
    nsub = SUB * C
    qpos = 4 * ((SUB + W) // 2) * ((C + W) // 2)
    executed = qpos * 64 * 2 * 64 * 64               # the w = 11 instantiation: 8 x 8 = 64 tap products per plane position
    achieved = executed / (cnn_ms / 1e3) / 1e12
    line = {
        "metric": "pixels/sec full-scene inference", "value": px / (ms_dev / 1e3), "unit": "pixels/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f16 operands / f32 accumulate (tcgen05 kind::f16); fp32 elsewhere", "data": "synthetic",
        "config": workload_config(cfg, world), "clocks": clocks,
        "e2e": {"value": px / (ms_e2e / 1e3), "unit": "pixels/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(sum((s1 - s0) * C * B * 2 for s0, s1 in slabs)), "d2h_bytes_per_step": 1024,
                "input": "raw uint16 sub-bands (+halo) from pinned host memory (bytes per rank), double-buffered on a copy "
                         "stream, preprocessing folded into conv0 / the spectral fp16 conversion; the label map stays on "
                         "the device"},
        "gpu_launches": (7 * len(subs) + (1 if world > 1 else 0)) * args.steps,
        "roofline": {"kernel": "conv2_scene_kernel<W11> on one sub-band (tcgen05 conv2 once per scene position in the 9 border "
                               "classes of an 11x11 window: 64 tap products of 64x64 MACs per plane position)",
                     "bound": "tensor", "achieved": achieved, "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["tf_burst"], "frac_burst": achieved / peaks["tf_burst"],
                     "frac_sustained": achieved / peaks["tf_sustained"], "traffic": None,
                     "executed_flop_per_launch": executed,
                     "algorithmic_flop_per_launch": nsub * fl["conv2"], "kernel_ms": cnn_ms,
                     "note": "`achieved` counts the FLOPs the kernel executes (the shortened T groups run N=128 / N=64 MMAs at "
                             "the cost of N=128, so the array is less full than at w = 20); algorithmic = SURVEY 8d per-patch "
                             "arithmetic for w = 11 (conv2 on 5x5 positions per pixel)",
                     "whole_step_algorithmic_tflops": (r1 - r0) * C * fl["all"] / (ms_dev / 1e3) / 1e12},
        "sub_band_rows": SUB,
    }
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
