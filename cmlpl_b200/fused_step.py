"""The mutual-learning step of train.py:150-272 as ONE C-ABI call (``cmlpl_train_step``): 15 kernel launches for both
BaseNet2 peers -- patch gather + noise + conv0, conv1/conv2 with their pools, the spectral branch, classifier, every
loss of train.py:191-265 with the memory-bank update, the whole backward pass and both Adam updates -- optionally
captured in a CUDA graph.  Convolutions, their data gradients and weight gradients run on tcgen05 (fp16 operands,
fp32 accumulation; bar 1e-3 * max|ref| against ``cmlpl_b200.train.mutual_step``, which stays the fp32 reference).

torch only owns the memory: parameters stay the nn.Module's tensors (updated in place), gradients are views into one
flat block that ``p.grad`` points at, Adam moments live here.
"""
from __future__ import annotations

import ctypes
import math
from ctypes import c_float, c_int, c_size_t, c_ulonglong, c_void_p

import torch

from . import _lib

TENSORS = ("conv0.weight", "conv0.bias", "conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias",
           "feat_spe.weight", "feat_spe.bias", "classifier.weight", "classifier.bias")
HIST = ("lc", "total", "cls", "con", "acc", "total1", "cls1", "con1", "lc1")
CAT = 2624
# classifier input width per window: 64 pooled channels x (w // 4)^2 positions + the 1024 spectral features
CAT_OF_W = {20: CAT, 11: 64 * 2 * 2 + 1024}


class TrainNet(ctypes.Structure):
    _fields_ = [("p", c_void_p * 10), ("g", c_void_p * 10), ("m", c_void_p * 10), ("v", c_void_p * 10),
                ("queue_feats", c_void_p), ("queue_probs", c_void_p)]


class TrainParams(ctypes.Structure):
    _fields_ = [("noise_scale", c_float), ("dropout_p", c_float), ("temperature", c_float), ("alpha", c_float),
                ("adap_thr", c_float), ("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float),
                ("bc1", c_float), ("bc2_sqrt", c_float), ("smooth", c_int), ("queue_ptr", c_int * 2),
                ("seed", c_ulonglong), ("offset", c_ulonglong), ("grad_amax", c_float), ("pad_", c_int)]


class TrainIO(ctypes.Structure):
    _fields_ = [("bs", c_int), ("btu", c_int), ("bands", c_int), ("classes", c_int), ("w", c_int), ("queue", c_int),
                ("cube", c_void_p), ("scene_rows", c_int), ("cols", c_int),
                ("pix", c_void_p), ("patch_noise", c_void_p), ("spectra", c_void_p), ("spec_row", c_void_p),
                ("spec_noise", c_void_p), ("drop_mask", c_void_p), ("labels", c_void_p),
                ("net", TrainNet * 2), ("params", c_void_p),
                ("logits", c_void_p), ("feat", c_void_p), ("probs", c_void_p), ("mask", c_void_p), ("hist", c_void_p),
                ("grad_flat", c_void_p), ("grad_flat_bytes", c_size_t), ("work", c_void_p), ("work_bytes", c_size_t)]


def _ptr(t):
    return None if t is None else t.data_ptr()


class FusedMutualStep:
    """State + launcher of the fused step for two ``BaseNet2`` peers.

    ``step(...)`` runs one step on the current stream and returns the device tensor ``hist`` (f32 [12]: lc, total,
    cls, con, acc, total1, cls1, con1, lc1) without any host synchronisation.  Inputs either come from the PCA cube
    (``cube``, ``pix``; noise / dropout from the device Philox stream unless tensors are injected) or are passed
    assembled (``patches`` f32 [2, nb, 60, w, w], ``spectra`` f32 [2, nb, B]) -- the form the parity tests use.
    The window w (20, or 11 for the odd window of ExtractPatches_for_base) is the peers' ``BaseNet2.w``.
    """

    def __init__(self, Base, Base1, bs=128, btu=128, lr=5e-4, betas=(0.9, 0.999), eps=1e-8, temperature=0.3,
                 alpha=0.95, thr=1.0, num_epochs=20, queue_batch=17, noise=0.5, dropout=None, seed=1088,
                 queue_size=None, use_graph=False, param_slots=64):
        _lib.require_device()
        self.nets = (Base, Base1)
        dev = next(Base.parameters()).device
        self.dev = dev
        self.bs, self.btu, self.nb = bs, btu, bs + btu
        self.B, self.C = Base.num_features, Base.num_classes
        self.w = int(getattr(Base, "w", 20))
        if int(getattr(Base1, "w", 20)) != self.w:
            raise _lib.CmlplError(f"the two peers have different windows ({self.w} and {Base1.w})")
        if self.w not in CAT_OF_W:
            raise _lib.CmlplError(f"FusedMutualStep: w={self.w} unsupported (20 or 11)")
        self.cat = CAT_OF_W[self.w]
        self.lr, self.betas, self.eps = lr, betas, eps
        self.T, self.alpha, self.thr, self.num_epochs, self.queue_batch = temperature, alpha, thr, num_epochs, queue_batch
        self.noise = noise
        self.dropout = Base.dropout if dropout is None else dropout
        self.seed, self.offset = seed, 0
        self.queue = 5 * bs * 2 if queue_size is None else queue_size          # train.py:138,142
        self.queue_ptr, self.queue_ptr1 = 0, 0
        self.adam_step = 0
        self.params = [[dict(n.named_parameters())[k] for k in TENSORS] for n in self.nets]
        for ps in self.params:
            for p in ps:
                if p.dtype != torch.float32 or not p.is_contiguous() or p.device != dev:
                    raise _lib.CmlplError("FusedMutualStep needs contiguous float32 CUDA parameters")
        sizes = [p.numel() for p in self.params[0]]
        pad = lambda n: (n + 63) // 64 * 64                                      # keep every tensor 256-byte aligned
        total = sum(pad(n) for n in sizes)
        z = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
        self.grad_flat, self.m_flat, self.v_flat = z(2 * total), z(2 * total), z(2 * total)
        self.grads, self.ms, self.vs = [[], []], [[], []], [[], []]
        o = 0
        for e in range(2):
            for p, n in zip(self.params[e], sizes):
                self.grads[e].append(self.grad_flat[o:o + n].view_as(p))
                self.ms[e].append(self.m_flat[o:o + n].view_as(p))
                self.vs[e].append(self.v_flat[o:o + n].view_as(p))
                p.grad = self.grads[e][-1]
                o += pad(n)
        self.queue_feats = [z(self.queue, 1024), z(self.queue, 1024)]
        self.queue_probs = [z(self.queue, self.C), z(self.queue, self.C)]
        # outputs are allocated for the constructor's (largest) batch; a smaller last batch (train.py's DataLoader keeps
        # the partial batch) uses the head of the same buffers -- self.logits / feat / probs / mask are per-step views
        self._logits, self._feat = z(2 * self.nb * self.C), z(2 * self.nb * 1024)
        self._probs, self._mask = z(2 * btu * self.C), z(2 * btu)
        self.hist = z(12)
        self._views(bs, btu)
        lib = _lib.load()
        self.work = torch.zeros((lib.cmlpl_train_workspace_bytes(bs, btu, self.B, self.C, self.queue),),
                                dtype=torch.uint8, device=dev)
        # per-step scalars: a ring of pinned host blocks -- the H2D copy of step k is asynchronous and the host runs many
        # steps ahead of the device, so a block is only rewritten after the copy that read it has completed (its event)
        self._nslots = max(2, int(param_slots))
        psz = ctypes.sizeof(TrainParams)
        self.prm_ring = torch.zeros((self._nslots, psz), dtype=torch.uint8).pin_memory()
        self._prm_events = [None] * self._nslots
        self._slot = 0
        self.prm_dev = torch.zeros((psz,), dtype=torch.uint8, device=dev)
        self.prm = TrainParams.from_address(self.prm_ring[0].data_ptr())
        # static input buffers (CUDA-graph replays read the same addresses)
        self.pix = torch.zeros((self.nb,), dtype=torch.int64, device=dev)
        self.labels = torch.zeros((bs,), dtype=torch.int64, device=dev)
        self.use_graph = use_graph
        self._graphs = {}
        self._keep = None

    # ------------------------------------------------------------------ plumbing
    def _views(self, bs, btu):
        nb = bs + btu
        self.cur = (bs, btu)
        self.logits = self._logits[:2 * nb * self.C].view(2, nb, self.C)
        self.feat = self._feat[:2 * nb * 1024].view(2, nb, 1024)
        self.probs = self._probs[:2 * btu * self.C].view(2, btu, self.C)
        self.mask = self._mask[:2 * btu].view(2, btu)

    def _io(self, cube, patches, spectra, spec_row, patch_noise, spec_noise, drop_mask):
        io = TrainIO()
        io.bs, io.btu, io.bands, io.classes, io.w, io.queue = self.cur[0], self.cur[1], self.B, self.C, self.w, self.queue
        if cube is not None:
            io.cube, io.scene_rows, io.cols = cube.data_ptr(), cube.shape[0], cube.shape[1]
            io.pix = self.pix.data_ptr()
            io.patch_noise = _ptr(patch_noise)
        else:
            io.cube, io.scene_rows, io.cols = None, 0, 0
            io.pix = None
            io.patch_noise = patches.data_ptr()
        io.spectra, io.spec_row, io.spec_noise = spectra.data_ptr(), _ptr(spec_row), _ptr(spec_noise)
        io.drop_mask = _ptr(drop_mask)
        io.labels = self.labels.data_ptr()
        for e in range(2):
            for i in range(10):
                io.net[e].p[i] = self.params[e][i].data_ptr()
                io.net[e].g[i] = self.grads[e][i].data_ptr()
                io.net[e].m[i] = self.ms[e][i].data_ptr()
                io.net[e].v[i] = self.vs[e][i].data_ptr()
            io.net[e].queue_feats = self.queue_feats[e].data_ptr()
            io.net[e].queue_probs = self.queue_probs[e].data_ptr()
        io.params = self.prm_dev.data_ptr()
        io.logits, io.feat, io.probs = self.logits.data_ptr(), self.feat.data_ptr(), self.probs.data_ptr()
        io.mask, io.hist = self.mask.data_ptr(), self.hist.data_ptr()
        io.grad_flat, io.grad_flat_bytes = self.grad_flat.data_ptr(), self.grad_flat.numel() * 4
        io.work, io.work_bytes = self.work.data_ptr(), self.work.numel()
        return io

    def _set_params(self, epoch, batch_index, phases):
        slot = self._slot
        self._slot = (slot + 1) % self._nslots
        if self._prm_events[slot] is not None:
            self._prm_events[slot].synchronize()             # the copy issued _nslots steps ago has read this block
        p = self.prm = TrainParams.from_address(self.prm_ring[slot].data_ptr())
        nb = self.cur[0] + self.cur[1]
        p.noise_scale, p.dropout_p, p.temperature, p.alpha = self.noise, self.dropout, self.T, self.alpha
        p.adap_thr = self.thr * math.exp(-0.5 * ((epoch / self.num_epochs) ** 2))          # train.py:147-148,221
        p.smooth = 1 if (epoch > 0 or batch_index > self.queue_batch) else 0                # train.py:212
        p.queue_ptr[0], p.queue_ptr[1] = self.queue_ptr, self.queue_ptr1
        step = self.adam_step + 1
        p.lr, p.beta1, p.beta2, p.eps = self.lr, self.betas[0], self.betas[1], self.eps
        p.bc1 = 1.0 - self.betas[0] ** step
        p.bc2_sqrt = math.sqrt(1.0 - self.betas[1] ** step)
        p.seed, p.offset = self.seed, self.offset
        if self.queue_ptr + nb > self.queue or self.queue_ptr1 + nb > self.queue:
            # train.py:232 would raise on the shape mismatch of the slice assignment
            raise RuntimeError("memory-bank write [%d, %d) exceeds the queue of %d rows (train.py:232-237)"
                               % (max(self.queue_ptr, self.queue_ptr1), max(self.queue_ptr, self.queue_ptr1) + nb, self.queue))
        self.prm_dev.copy_(self.prm_ring[slot], non_blocking=True)
        if self._prm_events[slot] is None:
            self._prm_events[slot] = torch.cuda.Event()
        self._prm_events[slot].record()
        if phases & 2:
            self.queue_ptr = (self.queue_ptr + 256) % self.queue                            # train.py:234 (literal 256)
            self.queue_ptr1 = (self.queue_ptr + 256) % self.queue                           # train.py:237 (sic: reads queue_ptr)
        if phases & 8:
            self.adam_step = step
        self.offset += 1

    WS_FIELDS = ("x16", "a0", "p1", "m1", "m2", "cat", "dmask", "ynoisy", "norm", "dlogits", "dfeat", "dcat", "dhp",
                 "dz1", "da0", "S", "G", "dG", "probs_orig", "total")

    def workspace_layout(self):
        """{region: byte offset into self.work} (cmlpl_train_workspace_layout; tests and profiling).  The offsets do not
        depend on w; a w = 11 step packs each region at its own per-sample strides (include/cmlpl.h)."""
        off = (c_size_t * 20)()
        _lib.call("cmlpl_train_workspace_layout", self.bs, self.btu, self.B, self.C, self.queue, off)
        return dict(zip(self.WS_FIELDS, [int(v) for v in off]))

    def grad_scale(self):
        """The power-of-two scale the last backward pass applied to dz1 / da0 (reads the device params: syncs)."""
        prm = TrainParams.from_buffer_copy(bytes(self.prm_dev.cpu().numpy()))
        return 2.0 ** (12 - math.frexp(prm.grad_amax)[1]) if prm.grad_amax > 0 else 1.0

    @staticmethod
    def launches(phases=15):
        return _lib.load().cmlpl_train_step_launches(phases)

    # ------------------------------------------------------------------ one step
    def step(self, labels, epoch, batch_index, cube=None, pix=None, spectra=None, spec_row=None, patches=None,
             patch_noise=None, spec_noise=None, drop_masks=None, phases=15):
        """labels i64 [bs].  Cube mode: ``cube`` f32 [R, C, 60], ``pix`` i64 [nb] raster pixels ([labelled ; unlabelled]),
        ``spectra`` f32 [N, B] table (row ``spec_row[i]`` or ``pix[i]``).  Assembled mode: ``patches`` f32
        [2, nb, 60, w, w] and ``spectra`` f32 [2, nb, B] (train.py:174,184 after the noise was added).
        ``patch_noise`` [2, nb, 60, w, w], ``spec_noise`` [2, nb, B] and ``drop_masks`` [2, nb, cat] (scaled; cat = 2624,
        or 1280 at w = 11) inject the random draws; otherwise the device Philox stream (seed, step counter) is used."""
        def chk(t, shape, name):
            if t is None or not t.is_cuda or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
                raise _lib.CmlplError(f"{name}: expected a contiguous CUDA tensor of shape {tuple(shape)}, got "
                                      f"{None if t is None else tuple(t.shape)}")
        if (cube is None) == (patches is None):
            raise _lib.CmlplError("pass either cube+pix or assembled patches")
        bs = int(labels.numel())
        nb = int(pix.numel()) if cube is not None and pix is not None else (int(patches.shape[1]) if patches is not None else 0)
        if not (0 < bs <= self.bs and bs < nb and nb - bs <= self.btu):
            raise _lib.CmlplError(f"batch of {bs} labelled + {nb - bs} unlabelled rows does not fit the step built for "
                                  f"{self.bs} + {self.btu}")
        if (bs, nb - bs) != self.cur:
            self._views(bs, nb - bs)
        if cube is not None:
            chk(pix, (nb,), "pix")
            if (not cube.is_cuda or cube.dim() != 3 or cube.shape[2] != 60 or cube.dtype != torch.float32 or
                    not cube.is_contiguous()):
                raise _lib.CmlplError("cube must be a contiguous CUDA f32 [R, C, 60] tensor (there is no CPU path)")
            if (spectra is None or not spectra.is_cuda or spectra.dim() != 2 or spectra.shape[1] != self.B or
                    spectra.dtype != torch.float32 or not spectra.is_contiguous()):
                raise _lib.CmlplError("spectra must be a contiguous CUDA f32 [rows, B] tensor")
            self.pix[:nb].copy_(pix, non_blocking=True)
            if patch_noise is not None:
                chk(patch_noise, (2, nb, 60, self.w, self.w), "patch_noise")
            if spec_noise is not None:
                chk(spec_noise, (2, nb, self.B), "spec_noise")
        else:
            chk(patches, (2, nb, 60, self.w, self.w), "patches")
            chk(spectra, (2, nb, self.B), "spectra")
        chk(labels, (bs,), "labels")
        self.labels[:bs].copy_(labels, non_blocking=True)
        dm = None
        if drop_masks is not None:
            dm = drop_masks if isinstance(drop_masks, torch.Tensor) else torch.stack(list(drop_masks))
            chk(dm, (2, nb, self.cat), "drop_masks")
        self._set_params(epoch, batch_index, phases)
        stream = torch.cuda.current_stream().cuda_stream
        key = (phases, bs, nb, _ptr(cube), _ptr(patches), _ptr(spectra), _ptr(spec_row), _ptr(patch_noise), _ptr(spec_noise), _ptr(dm))
        if self.use_graph:
            if key not in self._graphs:
                io = self._io(cube, patches, spectra, spec_row, patch_noise, spec_noise, dm)
                _lib.call("cmlpl_train_step", ctypes.byref(io), phases, c_void_p(stream))     # this step, eagerly
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):                                                     # capture only (nothing runs)
                    _lib.call("cmlpl_train_step", ctypes.byref(io), phases,
                              c_void_p(torch.cuda.current_stream().cuda_stream))
                self._graphs[key] = (g, (cube, patches, spectra, spec_row, patch_noise, spec_noise, dm))
            else:
                self._graphs[key][0].replay()
        else:
            io = self._io(cube, patches, spectra, spec_row, patch_noise, spec_noise, dm)
            _lib.call("cmlpl_train_step", ctypes.byref(io), phases, c_void_p(stream))
            self._keep = (cube, patches, spectra, spec_row, patch_noise, spec_noise, dm)
        if phases & 8:
            # the kernels write through raw pointers: bump the version counters (one call, a LIST of tensors) so
            # that BaseNet2.packed_weights' cache and autograd's saved-tensor checks see the update
            torch._C._increment_version(self.params[0] + self.params[1])
        return self.hist
