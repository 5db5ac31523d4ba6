"""The built library really contains the Blackwell instructions the design claims (no GPU needed: cuobjdump on the
in-tree .so, the same digest as profiles/r02_sass_digest.txt): tcgen05.mma (UTCHMMA) in every convolution / GEMM kernel
of the scene and training paths, tcgen05.st (STTM) where an epilogue hands data back through tensor memory, TMA tensor
loads (UTMALDG) in the scene kernels."""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "cmlpl_b200", "libcmlpl_sm100.so")
CUOBJDUMP = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP) or not os.path.exists(LIB), reason="needs cuobjdump and the built library")
def test_tcgen05_and_tma_instructions_present():
    env = dict(os.environ, PATH=os.path.dirname(CUOBJDUMP) + os.pathsep + os.environ.get("PATH", ""))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "sass_digest.py"), LIB], capture_output=True, text=True,
                         check=True, env=env).stdout
    rows = {}
    for line in out.splitlines():
        name = line[:62].strip()
        rows[name] = {k: int(v) for k, v in re.findall(r"(UTCHMMA|LDTM|STTM|UTMALDG|UBLKCP|REDG|FADD2)\s+(\d+)", line[62:])}

    def row(prefix):
        hits = [v for k, v in rows.items() if prefix in k]
        assert hits, f"{prefix} missing from the SASS digest"
        return hits

    for k in ("conv0_tc_kernel", "conv1_pool_kernel", "conv2_scene_kernel", "pool2_cls_kernel", "spectral_logits_kernel",
              "patch_cnn_kernel", "train_conv0_kernel", "train_conv_bwd_kernel", "train_conv0_bwd_kernel", "sim_tc_kernel"):
        for r in row(k):
            assert r["UTCHMMA"] > 0 and r["LDTM"] > 0, (k, r)
    for k in ("conv1_pool_kernel", "conv2_scene_kernel", "pool2_cls_kernel"):
        assert all(r["UTMALDG"] > 0 for r in row(k)), k
    for k in ("conv2_scene_kernel", "spectral_logits_kernel"):          # parked column partners / hidden tile as A operand
        assert all(r["STTM"] > 0 for r in row(k)), k
    assert all(r["REDG"] > 0 for r in row("train_conv_bwd_kernel"))      # vector reductions of the weight gradients
