"""Two builds of libcmlpl_sm100.so side by side in ONE process: the conv1_pool stage and the whole scene call on the
PaviaU-shaped c1 scene (610 x 340 x 103, w = 20), plus the conv1_pool stage on a c5-shaped band (512 x 8192, w = 11),
timed in alternating windows of >= 1 s each so that both builds see the same clocks and neighbours; and the outputs of
the two builds on the same inputs (the pooled conv1 planes bit for bit, in fp16 ulps; the label maps).
usage: ab_conv1_pool.py BASE_LIB NEW_LIB [--rounds N] [--window-s S] [--json OUT]"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cmlpl_b200 import _lib, ops  # noqa: E402
from oracle import cmlpl_oracle as O  # noqa: E402


def load(path):
    lib = ctypes.CDLL(os.path.abspath(path))
    for name, (res, args) in _lib.SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def ok(lib, rc):
    if rc != 0:
        msg = lib.cmlpl_last_error()
        raise RuntimeError(msg.decode() if msg else str(rc))


def window(fn, seconds):
    """ms per call of fn over a window of >= `seconds` (CUDA events around the whole window)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    n = max(20, int(seconds / max(time.perf_counter() - t0, 1e-6)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def fp16_ulps(a, b):
    """largest |a - b| in fp16 ulps of b (2^-24 below the normal range)."""
    bf = b.float()
    _, e = torch.frexp(bf)
    e = torch.where(bf == 0, torch.full_like(e, -24), e - 11).clamp_min(-24)
    return float(((a.float() - bf).abs() / torch.ldexp(torch.ones_like(bf), e)).max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("base")
    ap.add_argument("new")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    libs = {"base": load(args.base), "new": load(args.new)}
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    # ---- c1: PaviaU-shaped scene, reference-initialised net
    R, C, B, K, w = 610, 340, 103, 9, 20
    rng = np.random.default_rng(1088)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
    torch.manual_seed(1088)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K).items()}
    packed = ops.pack_basenet2(sd, B, K, w)
    off = (ctypes.c_size_t * 12)()
    _lib.call("cmlpl_scene_workspace_layout", R, C, B, K, w, off)
    ws = {k: torch.zeros(off[10], dtype=torch.uint8, device=dev) for k in libs}
    labels = {k: torch.empty(R * C, dtype=torch.uint8, device=dev) for k in libs}
    PR, PC = R + w - 1, C + w - 1
    PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
    n_f0, n_planes = 8 * PR * PC * 8, 9 * 4 * 8 * PR2 * PC2 * 8       # f16 entries of the conv0 map / the pooled planes

    def scene(k):
        lib = libs[k]
        return lambda: ok(lib, lib.cmlpl_scene_infer(cube.data_ptr(), R, C, 0, R, spectra.data_ptr(), B, K, w, 0, R,
                                                     packed.data_ptr(), ws[k].data_ptr(), ws[k].numel(),
                                                     labels[k].data_ptr(), None, st))

    def conv1(k, f0, pmq, cols, win, rows, pk):
        lib = libs[k]
        return lambda: ok(lib, lib.cmlpl_conv1_pool_planes_f16(f0, cols, win, rows, pk, pmq, st))

    for k in libs:
        scene(k)()
    torch.cuda.synchronize()
    f0_equal = bool(torch.equal(ws["base"][off[0]:off[0] + 2 * n_f0], ws["new"][off[0]:off[0] + 2 * n_f0]))
    a, b = (ws[k][off[4]:off[4] + 2 * n_planes].view(torch.float16) for k in ("new", "base"))
    out = {"card": torch.cuda.get_device_name(0),
           "c1_conv0_map_bit_equal": f0_equal,
           "c1_pmq_bit_equal_fraction": float((a == b).float().mean()),
           "c1_pmq_max_fp16_ulps": fp16_ulps(a, b),
           "c1_pmq_nan": int(torch.isnan(a).sum()),
           "c1_labels_differing": int((labels["new"] != labels["base"]).sum())}
    print(json.dumps(out), flush=True)

    # ---- c5-shaped band for the w = 11 instantiation (random conv0 map; the kernel's time does not depend on values)
    R5, C5, w5 = 512, 8192, 11
    PR5, PC5 = R5 + w5 - 1, C5 + w5 - 1
    f05 = torch.randn(8 * PR5 * PC5 * 8, device=dev).half()
    sd5 = {k: v.to(dev) for k, v in O.basenet2_init(224, 16, conv_feat=256).items()}
    pk5 = ops.pack_basenet2(sd5, 224, 16, w5)
    pmq5 = torch.empty(9 * 4 * 8 * ((PR5 + 1) // 2) * ((PC5 + 1) // 2) * 8, dtype=torch.float16, device=dev)

    fns = {}
    for k in libs:
        fns[("c1_conv1_pool_ms", k)] = conv1(k, ws[k].data_ptr() + off[0], ws[k].data_ptr() + off[4], C, w, R,
                                             packed.data_ptr())
        fns[("c1_scene_ms", k)] = scene(k)
        fns[("c5band_conv1_pool_ms", k)] = conv1(k, f05.data_ptr(), pmq5.data_ptr(), C5, w5, R5, pk5.data_ptr())
    rounds = []
    for r in range(args.rounds):
        res = {}
        order = ["base", "new"] if r % 2 == 0 else ["new", "base"]
        for metric in ("c1_conv1_pool_ms", "c1_scene_ms", "c5band_conv1_pool_ms"):
            for k in order:
                res[f"{metric}_{k}"] = window(fns[(metric, k)], args.window_s)
        rounds.append(res)
        print(json.dumps({"round": r, **{k: round(v, 5) for k, v in res.items()}}), flush=True)
    summary = {}
    for metric in ("c1_conv1_pool_ms", "c1_scene_ms", "c5band_conv1_pool_ms"):
        bs = [x[f"{metric}_base"] for x in rounds]
        ns = [x[f"{metric}_new"] for x in rounds]
        d = [bb - nn for bb, nn in zip(bs, ns)]
        summary[metric] = {"base": bs, "new": ns, "base_minus_new_ms": d, "min_gain_fraction": min(dd / bb for dd, bb in zip(d, bs)),
                           "spread_base_ms": max(bs) - min(bs), "spread_new_ms": max(ns) - min(ns)}
    out["rounds"] = rounds
    out["summary"] = summary
    print(json.dumps(summary), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
