"""Timeline of one CTA of a scene kernel (clock64 stamps of its issuer / epilogue / loader warps).
Needs the instrumented library:  make -C cmlpl_b200/csrc trace   (-> scripts/_trace/libcmlpl_trace.so, git-ignored);
GPU box only, debugging aid -- nothing in the product loads that library.
usage: trace_kernel.py {conv2|conv1|spectral} [first_event] [n_events]"""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cmlpl_b200 import _lib, ops  # noqa: E402
from cmlpl_b200.tools.models import BaseNet2  # noqa: E402

_lib.require_device()
dev = torch.device("cuda")
which = sys.argv[1] if len(sys.argv) > 1 else "conv2"
R, C, B, K, w = 610, 340, 103, 9, 20
rng = np.random.default_rng(1088)
cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
torch.manual_seed(1088)
net = BaseNet2(num_features=B, dropout=0, num_classes=K).to(dev).eval()
packed = net.packed_weights(w)
ws = ops.scene_workspace(R, C, B, K, w, dev)
labels = torch.empty(R * C, dtype=torch.uint8, device=dev)
ops.scene_infer(cube, spectra, packed, K, w, workspace=ws, labels=labels)
torch.cuda.synchronize()
off = (ctypes.c_size_t * 12)()
_lib.call("cmlpl_scene_workspace_layout", R, C, B, K, w, off)
tl = ctypes.CDLL(os.path.join(ROOT, "scripts", "_trace", "libcmlpl_trace.so"))
st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
P, I, L = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
base = ws.data_ptr()
for _ in range(3):
    if which == "conv2":
        tl.cmlpl_conv2_scene_f16.argtypes = [P, I, I, I, P, P, P]
        rc = tl.cmlpl_conv2_scene_f16(base + off[4], C, w, R, packed.data_ptr(), base + off[5], st)
        names, export = ["mma", "epi0", "epi1", "load"], "cmlpl_debug_c2s_trace"
    elif which == "conv1":
        tl.cmlpl_conv1_pool_planes_f16.argtypes = [P, I, I, I, P, P, P]
        rc = tl.cmlpl_conv1_pool_planes_f16(base + off[0], C, w, R, packed.data_ptr(), base + off[4], st)
        names, export = ["mma", "epi0", "epi1", "-", "load"], "cmlpl_debug_c1p_trace"
    else:
        tl.cmlpl_spectral_logits_tc.argtypes = [P, L, I, I, I, P, P, P, P]
        rc = tl.cmlpl_spectral_logits_tc(spectra.data_ptr(), R * C, B, K, w, packed.data_ptr(), base + off[1], base + off[2], st)
        names, export = ["mma1", "mma2", "epi0", "epi1", "load"], "cmlpl_debug_spl_trace"
    assert rc == 0, rc
torch.cuda.synchronize()
buf = np.zeros((6, 4096), dtype=np.uint64)
assert getattr(tl, export)(buf.ctypes.data_as(ctypes.c_void_p)) == 0
t0 = int(min(buf[r, 0] for r in range(len(names)) if buf[r, 0]))
ev = []
for r in range(len(names)):
    for i in range(2047):
        c, tag = int(buf[r, 2 * i]), int(buf[r, 2 * i + 1])
        if c == 0:
            break
        ev.append((c - t0, names[r], tag))
ev.sort()
first = int(sys.argv[2]) if len(sys.argv) > 2 else len(ev) // 2
count = int(sys.argv[3]) if len(sys.argv) > 3 else 160
if which == "conv2":
    G = ["PA", "T1", "T2", "T3", "PB"]
    mma = [(c, t) for c, n, t in ev if n == "mma"]
    print("cycles per tile (MMA issue start to start):", [mma[(i + 1) * 50][0] - mma[i * 50][0] for i in range(min(12, len(mma) // 50 - 1))])

    def desc(n, t):
        if n == "mma":
            return f"kap{t >> 4} {G[(t & 15) >> 1]} {'issued' if t & 1 else 'start'}"
        if n == "load":
            return f"tma tile {t}"
        r = t >> 2
        return f"item kap{r // 3} it{r % 3} " + ["wait", "ready", "done"][t & 3]
elif which == "conv1":
    m = [c for c, n, t in ev if n == "mma" and t % 8 == 0]
    print("cycles per tile (MMA loop):", [m[i + 1] - m[i] for i in range(5, min(17, len(m) - 1))])

    def desc(n, t):
        if n == "mma":
            return f"tile {t // 8} half {(t // 4) % 2} " + ["loop", "slot free", "issued"][t & 3]
        if n == "load":
            return f"tile {t} tma issued"
        return f"tile {t // 32} pass {(t // 8) % 4} " + ["wait slot", "slot full", "in regs", "stored"][t & 7]
else:
    m1 = [c for c, n, t in ev if n == "mma1" and (t & 3) == 0]
    print("cycles per unit (MMA1 loop):", [m1[i + 1] - m1[i] for i in range(20, 40)])

    def desc(n, t):
        u, k = t >> 2, t & 3
        if n == "mma1":
            return f"unit {u} " + ["loop", "A tile in", "slot free", "issued"][k]
        if n == "mma2":
            return f"unit {u} " + ["loop", "", "H in", "issued"][k]
        if n == "load":
            return f"tile {t} copy issued"
        return f"unit {u} " + ["wait D1", "D1 full", "H slot free", "H written"][k]
lo = ev[first][0]
for c, n, t in ev[first:first + count]:
    print(f"{c - lo:7d} {n:5s} {desc(n, t)}")
