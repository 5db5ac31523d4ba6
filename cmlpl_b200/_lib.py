"""ctypes binding of libcmlpl_sm100.so (the C ABI declared in include/cmlpl.h).

There is deliberately NO fallback: if the shared library is missing, cannot be loaded,
or a call fails, this module raises.  PyTorch is used by the callers only for device
memory and streams; every pointer handed over here is a raw device pointer.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcmlpl_sm100.so")

P, I, L, F, Z = c_void_p, c_int, c_int64, c_float, c_size_t

# name -> (restype, argtypes); mirrors include/cmlpl.h one to one
SIGNATURES = {
    "cmlpl_version": (I, []),
    "cmlpl_last_error": (c_char_p, []),
    "cmlpl_device_ok": (I, []),
    "cmlpl_memcpy2d_async": (I, [P, Z, P, Z, Z, Z, P]),
    "cmlpl_patch_gather_f32": (I, [P, I, I, I, I, I, I, I, P, L, L, P, F, P, P]),
    "cmlpl_sgemm_f32": (I, [I, I, I, F, P, L, L, P, L, L, P, F, P, L, L, I, P]),
    "cmlpl_conv2d_f32": (I, [P, P, P, P, P, I, I, I, I, I, I, I, I, P]),
    "cmlpl_conv2d_wgrad_f32": (I, [P, P, P, P, I, I, I, I, I, I, P]),
    "cmlpl_avgpool2_f32": (I, [P, P, L, I, I, P]),
    "cmlpl_avgpool2_bwd_f32": (I, [P, P, L, I, I, P]),
    "cmlpl_relu_bwd_f32": (I, [P, P, P, L, P]),
    "cmlpl_colsum_f32": (I, [P, P, L, L, P]),
    "cmlpl_l2norm_f32": (I, [P, P, P, L, L, F, P]),
    "cmlpl_l2norm_bwd_f32": (I, [P, P, P, P, L, L, F, P]),
    "cmlpl_packed_bytes": (Z, [I, I, I]),
    "cmlpl_pack_basenet2": (I, [P] * 10 + [I, I, I, P, P]),
    "cmlpl_scene_workspace_bytes": (Z, [I, I, I, I, I]),
    "cmlpl_scene_infer": (I, [P, I, I, I, I, P, I, I, I, I, I, P, P, Z, P, P, P]),
    "cmlpl_scene_infer_raw": (I, [P, I, I, I, I, I, I, I, I, I, I, P, P, P, P, P, P, Z, P, P, P]),
    "cmlpl_scene_infer_raw_masked": (I, [P, I, I, I, I, I, I, I, I, I, I, P, P, P, P, P, P, P, Z, P, P, P]),
    "cmlpl_valid_mask_u8": (I, [P, I, L, I, I, c_double, P, P, P, P]),
    "cmlpl_valid_mask_sel_u8": (I, [P, I, L, I, I, P, I, c_double, P, P, P, P]),
    "cmlpl_preprocess_fit_sel_f64": (I, [P, I, L, I, I, P, I, P, P, P, P, P]),
    "cmlpl_preprocess_apply_sel": (I, [P, I, L, I, P, I, I, P, P, P, P, P, P, P, P]),
    "cmlpl_scene_infer_raw_sel": (I, [P, I, I, I, I, I, I, P, I, I, I, I, I, P, P, P, P, P, P, P, Z, P, P, P]),
    "cmlpl_conv0_map_f16": (I, [P, I, I, I, I, I, I, I, P, P, P]),
    "cmlpl_patch_cnn_f16": (I, [P, I, I, I, P, P, P]),
    "cmlpl_scene_workspace_layout": (I, [I, I, I, I, I, P]),
    "cmlpl_conv1_pool_planes_f16": (I, [P, I, I, I, P, P, P]),
    "cmlpl_conv2_scene_f16": (I, [P, I, I, I, P, P, P]),
    "cmlpl_pool2_cls_f16": (I, [P, I, I, I, I, I, P, P, P]),
    "cmlpl_spectral_logits_tc": (I, [P, L, I, I, I, P, P, P, P]),
    "cmlpl_head_sum_lmap": (I, [P, P, I, I, I, I, I, P, P, P, P]),
    "cmlpl_argmax_u8": (I, [P, L, I, P, P]),
    "cmlpl_preprocess_fit_cube_f64": (I, [P, I, I, I, I, P, P, P]),
    "cmlpl_preprocess_fit_f64": (I, [P, I, L, I, P, P, P]),
    "cmlpl_preprocess_apply": (I, [P, I, L, I, I, P, P, P, P, P, P, P]),
    "cmlpl_preprocess_fit_masked_f64": (I, [P, I, L, I, I, P, P, P, P, P]),
    "cmlpl_preprocess_apply_masked": (I, [P, I, L, I, I, P, P, P, P, P, P, P, P]),
    "cmlpl_confusion_i64": (I, [P, P, L, I, P, P]),
    "cmlpl_ce_fwd_bwd_f32": (I, [P, P, P, P, L, I, F, P, P, P]),
    "cmlpl_softmax_entropy_f32": (I, [P, L, I, F, P, P]),
    "cmlpl_softmax_js_f32": (I, [P, P, L, I, F, P, P, P]),
    "cmlpl_sim_nt_tc_f32": (I, [P, P, I, I, I, P, P]),
    "cmlpl_set_loss_gemm_mode": (I, [I]),
    "cmlpl_set_scene_path_mode": (I, [I]),
    "cmlpl_bank_smooth_f32": (I, [P, P, P, P, L, I, I, L, F, F, I, F, P, P, P, P, P]),
    "cmlpl_graph_contrast_f32": (I, [P, P, P, P, L, I, I, F, I, F, P, P, P, P]),
    "cmlpl_ntxent_f32": (I, [P, L, I, F, P, P, P, P]),
    "cmlpl_adam_multi_f32": (I, [I, P, P, P, P, P, F, F, F, F, I, P]),
    "cmlpl_comm_unique_id": (I, [P]),
    "cmlpl_comm_init": (I, [I, I, P, P]),
    "cmlpl_comm_allgather_labels": (I, [P, P, L, P, P]),
    "cmlpl_comm_allreduce_confusion": (I, [P, P, I, P]),
    "cmlpl_comm_destroy": (I, [P]),
    "cmlpl_train_workspace_bytes": (Z, [I, I, I, I, I]),
    "cmlpl_train_workspace_layout": (I, [I, I, I, I, I, P]),
    "cmlpl_train_step": (I, [P, I, P]),
    "cmlpl_train_step_launches": (I, [I]),
}


class CmlplError(RuntimeError):
    pass


_lib = None


def load() -> ctypes.CDLL:
    """Load the library once.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CmlplError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  cmlpl_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def call(name: str, *args):
    """Call an int-returning entry point and raise CmlplError on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.cmlpl_last_error()
        raise CmlplError(f"{name} failed ({rc}): {msg.decode() if msg else '?'}")
    return rc


def require_device():
    """Fail loudly unless a CUDA device of compute capability 10.0 (B200) is current."""
    import torch

    if not torch.cuda.is_available():
        raise CmlplError("cmlpl_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    lib = load()
    torch.cuda.current_device()
    torch.cuda.init()
    ok = lib.cmlpl_device_ok()
    if ok != 1:
        raise CmlplError("cmlpl_b200 kernels are built for sm_100a (B200) only; current device is not sm_100")
