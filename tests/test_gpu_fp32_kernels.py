"""The fp32 kernel library (fp32_ops.cu, losses.cu, the CUDA-core GEMM core of gemm_core.cuh, argmax) against float64
references at the shapes where tiled and warp-per-row kernels go wrong: M / N / K and rows off every tile and warp
multiple, all transpose and stride combinations, odd pooling sizes, grid-stride loops that wrap, 1-4096 classes, and
softmax rows that underflow.  -m gpu.

Every bar is an error bound, not a max-relative tolerance, so that a dropped or duplicated term fails (see
test_fp32_kernels_cpu.py for the bound's tightness):
  * products and convolutions with reduction length K: |got - ref64| <= K 2^-23 (|A|.|B|) elementwise, plus a few ulp
    of the epilogue's terms (alpha, bias, residual, beta*C);
  * the loss kernels: the same first-order analysis per element.  Each log-probability z - lse carries an absolute
    error of at most 2^-22 (C + 8 + 2|lse| + |max z| + |z - max z|) (`lp_err`), which is also the relative error of
    the probability; the bars propagate it through each loss's formula over absolute values.
The last test runs one fp32 mutual-learning step (`train.mutual_step`) at the WHU-Hi HongHu shape, 270 bands, 22
classes, w = 11, against the oracle's ref_step with the bars of test_gpu_train.py.
"""
import argparse
import copy
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from fused_step_harness import assembled, init_nets, make_inputs, oracle_step, random_banks, set_banks, thr_for
from oracle import cmlpl_oracle as O
from oracle import golden
from scene_harness import rel, relu_flips
from test_fp32_kernels_cpu import U, js_inputs, product_bound, softmax_js_loss_ref

pytestmark = pytest.mark.gpu

f64 = torch.float64


def gen(seed):
    return torch.Generator().manual_seed(seed)


def within(got, ref, tol, what=""):
    """|got - ref| <= tol elementwise; NaN or inf in got fails."""
    got = np.asarray(got.detach().cpu().double() if torch.is_tensor(got) else got, np.float64)
    ref = np.asarray(ref.detach().cpu() if torch.is_tensor(ref) else ref, np.float64)
    tol = np.broadcast_to(np.asarray(tol.detach().cpu() if torch.is_tensor(tol) else tol, np.float64), ref.shape)
    err = np.abs(got - ref)
    bad = ~(err <= tol)
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, np.nan_to_num(err - tol, nan=np.inf), -np.inf)), ref.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} outside the bound; at {i}: got {got[i]!r}, "
                             f"ref {ref[i]!r}, bound {tol[i]!r}")


def lp_err(z):
    """Per-element bound on the absolute error of z - lse as the kernels compute it (float64 z [rows, C])."""
    C = z.shape[1]
    mx = z.max(1, keepdim=True)[0]
    lse = torch.logsumexp(z, 1, keepdim=True)
    return 2 * U * (C + 8 + 2 * lse.abs() + mx.abs() + (z - mx).abs())


DENORM = 2.0 ** -148   # two fp32 denormal quanta: the absolute floor of a value that underflows, in or out of a kernel


# ------------------------------------------------------------------------------------------------ 1. GEMM core
GEMM_SHAPES = [(1, 1, 1), (15, 17, 16), (16, 16, 15), (17, 15, 17), (63, 65, 64), (64, 64, 63), (65, 63, 65),
               (130, 17, 1000), (1000, 15, 130), (17, 1000, 63), (1, 1000, 1000), (1000, 1, 17), (130, 130, 130),
               (64, 1000, 1), (1000, 65, 16)]


def strided(rows, cols, g, pad=5):
    """A [rows, cols] column slice of a wider matrix (row stride cols + pad)."""
    return torch.randn(rows, cols + pad, generator=g)[:, 2:2 + cols]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
def test_sgemm_shapes_and_transposes(dev, M, N, K):
    from cmlpl_b200 import ops
    g = gen(M * 1_000_003 + N * 1009 + K)
    for ta in (False, True):
        for tb in (False, True):
            A = strided(K, M, g) if ta else strided(M, K, g)
            B = strided(N, K, g) if tb else strided(K, N, g)
            # on the device: the same views of device copies of the wide matrices (strides kept)
            Ad = torch.zeros(A.shape[0], A.shape[1] + 5, device=dev)[:, 2:2 + A.shape[1]]
            Ad.copy_(A)
            Bd = torch.zeros(B.shape[0], B.shape[1] + 5, device=dev)[:, 2:2 + B.shape[1]]
            Bd.copy_(B)
            got = ops.sgemm(Ad, Bd, transA=ta, transB=tb)
            a, b = (A.t() if ta else A).to(f64), (B.t() if tb else B).to(f64)
            within(got, a @ b, product_bound(a.abs() @ b.abs(), K), f"sgemm {M}x{N}x{K} tA={ta} tB={tb}")
            # transposed views of the same storage (unit row stride)
            if M > 1 and K > 1:
                got_t = ops.sgemm(Ad.t(), Bd, transA=not ta, transB=tb)
                within(got_t, a @ b, product_bound(a.abs() @ b.abs(), K), f"sgemm via A^T view {M}x{N}x{K}")


@pytest.mark.parametrize("M,N,K", [(65, 130, 17), (1, 15, 1000), (130, 63, 64), (17, 1, 1)])
def test_sgemm_epilogue_into_strided_output(dev, M, N, K):
    """out = act(alpha A.B + bias + beta out) into a slice of a larger buffer (both row- and column-strided), whose
    other elements stay as they were."""
    from cmlpl_b200 import ops
    g = gen(7 * M + N + K)
    A, B = torch.randn(M, K, generator=g), torch.randn(K, N, generator=g)
    bias = torch.randn(N, generator=g)
    a, b = A.to(f64), B.to(f64)
    ab, absab = a @ b, a.abs() @ b.abs()
    for alpha, beta, act in ((-1.75, 0.625, 0), (0.3, -2.0, 1), (1.0, 1.0, 1)):
        for layout in ("rows", "cols"):
            if layout == "rows":
                buf = torch.randn(M + 3, N + 9, generator=g).to(dev)
                out = buf[1:1 + M, 3:3 + N]
            else:
                buf = torch.randn(N + 2, M + 4, generator=g).to(dev)
                out = buf[1:1 + N, 2:2 + M].t()
            before = buf.cpu().clone()
            C0 = out.cpu().to(f64)
            ops.sgemm(A.to(dev), B.to(dev), bias=bias.to(dev), act=act, out=out, alpha=alpha, beta=beta)
            ref = alpha * ab + bias.to(f64) + beta * C0
            if act:
                ref = ref.clamp_min(0)
            tol = abs(alpha) * product_bound(absab, K) + 3 * U * (abs(alpha) * absab + bias.to(f64).abs() + abs(beta) * C0.abs())
            within(out, ref, tol, f"sgemm epilogue alpha={alpha} beta={beta} act={act} {layout}")
            after = buf.cpu()
            keep = torch.ones_like(after, dtype=torch.bool)
            if layout == "rows":
                keep[1:1 + M, 3:3 + N] = False
            else:
                keep[1:1 + N, 2:2 + M] = False
            assert torch.equal(after[keep], before[keep]), "sgemm wrote outside its output view"


def test_sgemm_k0(dev):
    """K = 0: out = act(bias + beta out), also when the empty operands have no storage (null data pointers)."""
    from cmlpl_b200 import ops
    g = gen(11)
    M, N = 17, 65
    bias = torch.randn(N, generator=g)
    for A, B in ((torch.empty(M, 0, device=dev), torch.empty(0, N, device=dev)),
                 (torch.zeros(M, 3, device=dev)[:, :0], torch.zeros(3, N, device=dev)[:0])):
        for act, beta in ((0, 0.5), (1, -1.5), (0, 0.0)):
            C0 = torch.randn(M, N, generator=g)
            out = C0.to(dev)
            ops.sgemm(A, B, bias=bias.to(dev), act=act, out=out, alpha=3.0, beta=beta)
            ref = bias.to(f64) + beta * C0.to(f64)
            if act:
                ref = ref.clamp_min(0)
            within(out, ref, 2 * U * (bias.to(f64).abs() + abs(beta) * C0.to(f64).abs()), f"K=0 act={act} beta={beta}")


# ------------------------------------------------------------------------------------------------ 2. convolutions
#            b    ci  co   h   w
CONV_CASES = [(1, 60, 64, 20, 20), (3, 64, 64, 11, 11), (33, 3, 9, 10, 10), (128, 17, 70, 5, 5), (33, 60, 64, 2, 2),
              (1, 64, 64, 1, 1), (3, 17, 70, 7, 13), (128, 64, 64, 10, 10), (128, 3, 9, 20, 20), (33, 64, 64, 7, 13),
              (1, 3, 9, 11, 11), (3, 60, 64, 5, 5)]


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "b{}_{}to{}_{}x{}".format(*c))
def test_conv_fwd_dgrad_wgrad(dev, case, k):
    from cmlpl_b200 import ops
    b, ci, co, h, w = case
    g = gen(b * 131 + ci * 17 + co + h * 7 + w + k)
    pad = k // 2
    x = torch.randn(b, ci, h, w, generator=g)
    wt = torch.randn(co, ci, k, k, generator=g) / (ci * k * k) ** 0.5
    bias = torch.randn(co, generator=g)
    res = torch.randn(b, co, h, w, generator=g)
    dy = torch.randn(b, co, h, w, generator=g)
    rdx = torch.randn(b, ci, h, w, generator=g)
    x64, w64, b64, r64, dy64, rdx64 = (t.to(f64) for t in (x, wt, bias, res, dy, rdx))
    X, Wd, Bd, R, DY, RDX = (t.to(dev) for t in (x, wt, bias, res, dy, rdx))
    tag = f"b{b} {ci}->{co} {h}x{w} k{k}"
    # forward: plain, and + bias + residual + ReLU
    ref = F.conv2d(x64, w64, padding=pad)
    absref = F.conv2d(x64.abs(), w64.abs(), padding=pad)
    Kf = ci * k * k
    within(ops.conv2d(X, Wd), ref, product_bound(absref, Kf), "conv fwd " + tag)
    ref2 = (ref + b64.view(1, -1, 1, 1) + r64).clamp_min(0)
    tol2 = product_bound(absref, Kf) + 3 * U * (absref + b64.abs().view(1, -1, 1, 1) + r64.abs())
    within(ops.conv2d(X, Wd, Bd, res=R, relu=True), ref2, tol2, "conv fwd+bias+res+relu " + tag)
    # data gradient, without and with the residual branch's gradient
    Kd = co * k * k
    refd = torch.nn.grad.conv2d_input(x.shape, w64, dy64, padding=pad)
    absd = torch.nn.grad.conv2d_input(x.shape, w64.abs(), dy64.abs(), padding=pad)
    within(ops.conv2d_dgrad(DY, Wd), refd, product_bound(absd, Kd), "conv dgrad " + tag)
    within(ops.conv2d_dgrad(DY, Wd, res=RDX), refd + rdx64, product_bound(absd, Kd) + 2 * U * (absd + rdx64.abs()),
           "conv dgrad+res " + tag)
    # weight gradient (split-K atomics) and bias gradient (sample loop over b > 32)
    Kw = b * h * w
    dw, db = ops.conv2d_wgrad(X, DY, k)
    refw = torch.nn.grad.conv2d_weight(x64, wt.shape, dy64, padding=pad)
    absw = torch.nn.grad.conv2d_weight(x64.abs(), wt.shape, dy64.abs(), padding=pad)
    within(dw, refw, product_bound(absw, Kw), "conv wgrad " + tag)
    within(db, dy64.sum((0, 2, 3)), product_bound(dy64.abs().sum((0, 2, 3)), Kw), "conv bias grad " + tag)


# ------------------------------------------------------------------------------------------------ 3. elementwise
def _wrap_elems(dev):
    """Elements past which the grid-stride loops of fp32_ops.cu (16 CTAs of 256 threads per SM) wrap."""
    return 16 * torch.cuda.get_device_properties(dev).multi_processor_count * 256


@pytest.mark.parametrize("hw", [11, 5, 3])
def test_avgpool2_odd_sizes(dev, hw):
    """Floor pooling at odd sizes with enough planes that the grid-stride loop wraps: the forward is the window sum
    ((x00 + x01) + x10) + x11 over 4 bit for bit; the backward is exactly dy/4 on the pooled positions and exactly 0 on
    the dropped last row and column."""
    from cmlpl_b200 import ops
    oh = hw // 2
    planes = _wrap_elems(dev) // (oh * oh) + 999
    c = 64
    b = -(-planes // c)
    g = gen(hw)
    x = torch.randn(b, c, hw, hw, generator=g)
    y = ops.avgpool2(x.to(dev)).cpu()
    assert y.numel() > _wrap_elems(dev)
    xn = x.numpy()
    s00, s01 = xn[:, :, 0:2 * oh:2, 0:2 * oh:2], xn[:, :, 0:2 * oh:2, 1:2 * oh:2]
    s10, s11 = xn[:, :, 1:2 * oh:2, 0:2 * oh:2], xn[:, :, 1:2 * oh:2, 1:2 * oh:2]
    want = (((s00 + s01) + s10) + s11) / np.float32(4)
    assert np.array_equal(y.numpy(), want)
    ref64 = F.avg_pool2d(x.to(f64), 2, 2)
    within(y, ref64, 3 * U / 2 * F.avg_pool2d(x.to(f64).abs(), 2, 2), f"avgpool2 {hw}")
    dy = torch.randn(b, c, oh, oh, generator=g)
    dx = ops.avgpool2_bwd(dy.to(dev), hw, hw).cpu()
    assert dx.shape == (b, c, hw, hw)
    assert torch.equal(dx[:, :, 2 * oh:, :], torch.zeros_like(dx[:, :, 2 * oh:, :]))
    assert torch.equal(dx[:, :, :, 2 * oh:], torch.zeros_like(dx[:, :, :, 2 * oh:]))
    up = (dy / 4).repeat_interleave(2, 2).repeat_interleave(2, 3)
    assert torch.equal(dx[:, :, :2 * oh, :2 * oh], up)


def test_relu_bwd_exact(dev):
    from cmlpl_b200 import ops
    g = gen(12)
    n = _wrap_elems(dev) + 4099
    y = torch.randn(n, generator=g)
    y[::7] = 0.0
    y[3::7] = -0.0
    y[5::11] = 1e-45                                  # a denormal is > 0
    dy = torch.randn(n, generator=g)
    got = ops.relu_bwd(y.to(dev), dy.to(dev)).cpu()
    assert torch.equal(got, torch.where(y > 0, dy, torch.zeros_like(dy)))


@pytest.mark.parametrize("m", [1, 7, 9, 70000])
@pytest.mark.parametrize("n", [1, 33, 1023])
def test_colsum(dev, m, n):
    from cmlpl_b200 import ops
    g = torch.Generator(device=dev).manual_seed(m * 7 + n)
    x = torch.randn(m, n, generator=g, device=dev)
    got = ops.colsum(x)
    x64 = x.cpu().to(f64)
    within(got, x64.sum(0), product_bound(x64.abs().sum(0), m), f"colsum {m}x{n}")


@pytest.mark.parametrize("rows", [1, 9, 77])
@pytest.mark.parametrize("cols", [1, 7, 33, 1000])
def test_l2norm_and_backward(dev, rows, cols):
    from cmlpl_b200 import ops
    g = gen(rows * 1000 + cols)
    x = torch.randn(rows, cols, generator=g) * 3
    dy = torch.randn(rows, cols, generator=g)
    for eps in (0.0, 1e-12):
        y, nr = ops.l2norm(x.to(dev), eps)
        x64 = x.to(f64)
        n64 = x64.norm(dim=1)
        within(nr, n64, (cols + 4) * U * n64, f"l2norm norm {rows}x{cols}")
        within(y, x64 / n64[:, None], (cols + 4) * U * (x64 / n64[:, None]).abs(), f"l2norm y {rows}x{cols}")
        # backward on the kernel's own fp32 y and norm
        y64, nn64 = y.cpu().to(f64), nr.cpu().to(f64)[:, None]
        s = (dy.to(f64) * y64).sum(1, keepdim=True)
        ref = (dy.to(f64) - y64 * s) / nn64
        sabs = (dy.to(f64) * y64).abs().sum(1, keepdim=True)
        tol = (cols + 4) * U * (dy.to(f64).abs() + y64.abs() * sabs) / nn64
        within(ops.l2norm_bwd(y, nr, dy.to(dev), eps), ref, tol, f"l2norm_bwd {rows}x{cols}")


def test_l2norm_zero_row_eps(dev):
    """eps = 0 (models.py Normalize) keeps the reference's NaN on a zero row; eps = 1e-12 is F.normalize: the row is 0
    and its gradient is dy / eps, as torch's autograd of F.normalize gives."""
    from cmlpl_b200 import ops
    g = gen(13)
    x = torch.randn(9, 33, generator=g)
    x[4] = 0
    dy = torch.randn(9, 33, generator=g)
    y0, n0 = ops.l2norm(x.to(dev))
    assert torch.isnan(y0[4]).all() and torch.isfinite(y0[torch.arange(9) != 4]).all()
    y, nr = ops.l2norm(x.to(dev), 1e-12)
    xr = x.to(f64).requires_grad_(True)
    ref = F.normalize(xr, dim=1)
    ref.backward(dy.to(f64))
    assert torch.equal(y[4].cpu(), torch.zeros(33)) and float(nr[4]) == 0.0
    within(y, ref.detach(), 40 * U * ref.detach().abs(), "F.normalize forward")
    dx = ops.l2norm_bwd(y, nr, dy.to(dev), 1e-12)
    within(dx, xr.grad, 40 * U * xr.grad.abs() + 1e-6 * xr.grad.abs().max(1, keepdim=True)[0], "F.normalize backward")


# ------------------------------------------------------------------------------------------------ 4. loss kernels
LOSS_ROWS = [1, 5, 77, 129]
LOSS_C = [1, 2, 9, 16, 17, 22, 32, 4096]


def logits(rows, C, g):
    """N(0, 3^2) logits; the first row spans 200 (softmax underflows in fp32) where there is more than one class."""
    z = torch.randn(rows, C, generator=g) * 3
    if C > 1:
        z[0] = torch.linspace(100, -100, C)[torch.randperm(C, generator=g)]
    return z


@pytest.mark.parametrize("C", LOSS_C)
@pytest.mark.parametrize("rows", LOSS_ROWS)
def test_ce_hard_and_soft(dev, rows, C):
    from cmlpl_b200 import ops
    g = gen(rows * 10007 + C)
    z = logits(rows, C, g)
    z64 = z.to(f64)
    lp = F.log_softmax(z64, 1)
    p = lp.exp()
    e = lp_err(z64)
    scale = 0.7
    gsc = scale / rows
    m = (torch.rand(rows, generator=g) > 0.3).float()
    y = torch.randint(0, C, (rows,), generator=g)
    if rows >= 5:
        y[1], m[1] = 255, 0.0                          # ignore_index 255 with mask 0
        y[3], m[3] = 255, 1.0                          # with mask 1: out of range (nothing) below 256 classes
    m64 = m.to(f64)[:, None]
    # hard labels
    loss, dz = ops.ce_fwd_bwd(z.to(dev), labels=y.to(dev), mask=m.to(dev), scale=scale)
    valid = (y < C)[:, None]
    onehot = torch.zeros(rows, C, dtype=f64)
    onehot[valid[:, 0], y[valid[:, 0]]] = 1
    li = -(lp * onehot).sum(1, keepdim=True) * m64
    tol_li = m64 * (onehot * (e + U * lp.abs())).sum(1, keepdim=True)
    within(loss, gsc * li.sum(), gsc * (tol_li.sum() + (rows + 4) * U * li.abs().sum()) + 1e-30, f"ce hard loss {rows}x{C}")
    ref_dz = gsc * m64 * valid * (p - onehot)
    live = (m64 * valid) > 0
    within(dz, ref_dz, gsc * m64 * valid * (p * e + 4 * U * (p + onehot)) + live * DENORM, f"ce hard dz {rows}x{C}")
    zr = z64.clone().requires_grad_(True)        # the same against autograd of F.cross_entropy (labels outside [0, C) ignored)
    y_ref = torch.where(valid[:, 0], y, torch.full_like(y, -100))
    (scale * (F.cross_entropy(zr, y_ref, reduction="none") * m.to(f64)).mean()).backward()
    assert torch.allclose(zr.grad, ref_dz, rtol=0, atol=1e-12)
    # soft targets (rows need not sum to 1) with the mask
    t = torch.softmax(torch.randn(rows, C, generator=g) * 2, 1) * 0.9
    t64 = t.to(f64)
    loss, dz = ops.ce_fwd_bwd(z.to(dev), probs=t.to(dev), mask=m.to(dev), scale=scale)
    li = -(lp * t64).sum(1, keepdim=True) * m64
    tol_li = m64 * (t64 * (e + (C + 2) * U * lp.abs())).sum(1, keepdim=True)
    within(loss, gsc * li.sum(), gsc * (tol_li.sum() + (rows + 4) * U * li.abs().sum()) + 1e-30, f"ce soft loss {rows}x{C}")
    ts = t64.sum(1, keepdim=True)
    within(dz, gsc * m64 * (p * ts - t64), gsc * m64 * (p * ts * (e + (C + 2) * U) + 4 * U * (p * ts + t64)) + (m64 > 0) * DENORM,
           f"ce soft dz {rows}x{C}")
    zr = z64.clone().requires_grad_(True)
    (scale * O.soft_ce(zr, t64, m.to(f64))).backward()
    assert torch.allclose(zr.grad, gsc * m64 * (p * ts - t64), rtol=0, atol=1e-12)


@pytest.mark.parametrize("C", LOSS_C)
@pytest.mark.parametrize("rows", LOSS_ROWS)
def test_softmax_entropy(dev, rows, C):
    from cmlpl_b200 import ops
    g = gen(rows * 10009 + C)
    z = logits(rows, C, g)
    z64 = z.to(f64)
    p = torch.softmax(z64, 1)
    eps = float(np.float32(1e-10))
    terms = p * torch.log(p + eps)
    got = ops.softmax_entropy(z.to(dev))
    e = lp_err(z64)
    tol = (p * e * ((p + eps).log().abs() + 1) + (C + 4) * U * terms.abs()).sum(1) + C * 30 * DENORM
    within(got, -terms.sum(1), tol, f"softmax_entropy {rows}x{C}")


def js_bound(z64, t64, scale):
    """Bounds on js_kernel's loss and dz (formula of its header comment) by first-order propagation of lp_err."""
    rows, C = z64.shape
    lp = F.log_softmax(z64, 1)
    p = lp.exp()
    e = lp_err(z64)
    M = 0.5 * (p + t64)
    lM = torch.where(M > 0, torch.log(torch.where(M > 0, M, torch.ones_like(M))), torch.zeros_like(M))
    lt = torch.log(t64 + float(np.float32(1e-5)))
    dM = 0.5 * p * e + U * M + DENORM
    dlM = torch.where(M > 0, e + 2 * U + U * lM.abs(), torch.zeros_like(M))
    dlt = U * (lt.abs() + 2)
    h = lM + 1 - 0.5 * lp - 0.5 * lt
    dh = dlM + 0.5 * e + 0.5 * dlt + U * (lM.abs() + lp.abs() + lt.abs() + 4)
    Q = p * h.abs() + M
    dq = p * (e * h.abs() + dh) + dM + 2 * U * Q + (h.abs() + 2) * DENORM     # p and M may underflow in fp32
    cf = scale * 0.5 / (rows * C)
    tol_dz = cf * (dq + p * dq.sum(1, keepdim=True) + (e + (C + 4) * U) * p * Q.sum(1, keepdim=True) + 4 * U * Q) + DENORM
    li_abs = (M * ((lM - lp).abs() + (lM - lt).abs())).sum(1)
    tol_li = (dM * (2 * lM - lp - lt).abs() + M * (2 * dlM + e + dlt)).sum(1) + (C + 4) * U * li_abs
    tol_loss = cf * (tol_li.sum() + (rows + 4) * U * li_abs.sum()) + 1e-30
    return tol_loss, tol_dz


@pytest.mark.parametrize("C", LOSS_C)
@pytest.mark.parametrize("rows", LOSS_ROWS)
def test_softmax_js(dev, rows, C):
    """Includes rows whose softmax underflows in fp32 (spreads 120, 200, 1600) and targets with exact zeros: the
    parent's M/p gradient gave NaN on every such row."""
    from cmlpl_b200 import ops
    z, t = js_inputs(rows, C, rows * 10037 + C)
    z, t = z.float(), t.float()
    z64, t64 = z.to(f64), t.to(f64)
    scale = 1.3
    zr = z64.clone().requires_grad_(True)
    ref = scale * softmax_js_loss_ref(zr, t64)
    ref.backward()
    loss, dz = ops.softmax_js(z.to(dev), t.to(dev), scale)
    tol_loss, tol_dz = js_bound(z64, t64, scale)
    assert torch.isfinite(dz).all(), f"softmax_js dz not finite on rows {torch.where(~torch.isfinite(dz).all(1))[0].tolist()}"
    within(loss, ref.detach(), tol_loss, f"softmax_js loss {rows}x{C}")
    within(dz, zr.grad, tol_dz, f"softmax_js dz {rows}x{C}")


BANK_CASES = [(1, 33, 1024), (5, 1000, 7), (77, 1, 7), (129, 1279, 1024)]       # rows, queue, dim


@pytest.mark.parametrize("C", [1, 2, 9, 16, 17, 22, 32])
@pytest.mark.parametrize("rows,queue,dim", BANK_CASES)
def test_bank_smooth(dev, rows, queue, dim, C):
    """Both templates (C <= 16 and 17-32), queues that are not a multiple of 32, all-zero bank rows (their exp(0) = 1
    still counts); rows whose max probability lies within 1e-5 of thr are excluded from the mask comparison."""
    from cmlpl_b200 import ops
    g = gen(rows * 7919 + queue * 31 + dim + C)
    z = logits(rows, C, g)
    f = O.normalize(torch.randn(rows, dim, generator=g, dtype=f64)).float()
    qf = O.normalize(torch.randn(queue, dim, generator=g, dtype=f64)).float()
    qp = torch.softmax(torch.randn(queue, C, generator=g) * 2, 1)
    zq = queue // 5
    if zq:
        qf[-zq:] = 0
        qp[-zq:] = 0
    z64, f64_, qf64, qp64 = (t.to(f64) for t in (z, f, qf, qp))
    alpha, T = 0.95, 0.3
    ref_o = torch.softmax(z64, 1)
    tol_o = ref_o * lp_err(z64) + DENORM
    S = f64_ @ qf64.t()
    a = torch.exp(S / T)
    A = (a @ qp64) / a.sum(1, keepdim=True)
    dS = product_bound(f64_.abs() @ qf64.abs().t(), dim)
    ea = (dS / T + 2 * U * (1 + S.abs() / T)).max(1, keepdim=True)[0]
    for smooth in (False, True):
        ref = alpha * ref_o + (1 - alpha) * A if smooth else ref_o
        thr = float(ref.max(1)[0].median())
        po, pr, mk = ops.bank_smooth(z.to(dev), f.to(dev), qf.to(dev), qp.to(dev), alpha, T, smooth, thr)
        within(po, ref_o, tol_o, f"bank_smooth probs_orig {rows} q{queue} C{C}")
        tol = (alpha * tol_o + (1 - alpha) * A * (2 * ea + (queue + 8) * U) + 3 * U * ref) if smooth else tol_o
        within(pr, ref, tol, f"bank_smooth probs smooth={smooth} {rows} q{queue} C{C}")
        mx = ref.max(1)[0]
        keep = (mx - thr).abs() >= 1e-5
        assert torch.equal(mk.cpu()[keep], (mx >= thr).float()[keep])


def graph_probs(n, C, seed):
    """Sharp class probabilities whose products p1.p^T stay 1e-5 away from the thresholds 0.3 and 0.8 (so the masks
    are the reference's) and contain entries on both sides of each."""
    for s in range(seed, seed + 200):
        g = gen(s)
        p1 = torch.softmax(torch.randn(n, C, generator=g) * 4, 1)
        p = torch.softmax(torch.randn(n, C, generator=g) * 4, 1)
        p1[: n // 2] = p[: n // 2] * 0.7 + p1[: n // 2] * 0.3      # some pairs share a class: entries >= 0.8 too
        q = p1.to(f64) @ p.to(f64).t()
        off = ~torch.eye(n, dtype=torch.bool)
        qo = q[off]
        if ((qo - 0.3).abs().min() > 1e-5 and (qo - 0.8).abs().min() > 1e-5 and (qo >= 0.8).any() and (qo <= 0.3).any()
                and ((qo > 0.3) & (qo < 0.8)).any()):
            return p1, p
    raise AssertionError("no probabilities with a margin around the thresholds")


@pytest.mark.parametrize("dim", [7, 1024])
@pytest.mark.parametrize("n,C", [(5, 16), (77, 22), (129, 9)])
def test_graph_contrast(dev, n, C, dim):
    from cmlpl_b200 import ops
    g = gen(n * 13 + dim)
    fs = O.normalize(torch.randn(n, dim, generator=g, dtype=f64)).float()
    fw = O.normalize(torch.randn(n, dim, generator=g, dtype=f64)).float()
    p1, p = graph_probs(n, C, 100 * n + C)
    q0 = p1.to(f64) @ p.to(f64).t()
    off = ~torch.eye(n, dtype=torch.bool)
    assert (q0[off] - 0.3).abs().min() > 1e-5 and (q0[off] - 0.8).abs().min() > 1e-5
    fs64, fw64 = fs.to(f64), fw.to(f64)
    Q, Qn = O.graph_targets(p1.to(f64), p.to(f64))
    T = 0.3
    # the loss's error bound, and dG = dL/dG (the matrix the kernel hands to the last GEMM) over absolute values
    G = fs64 @ fw64.t()
    dG_in = product_bound(fs64.abs() @ fw64.abs().t(), dim)
    l = G / T
    lz = torch.logsumexp(l, 1, keepdim=True)
    sp = torch.exp(l - lz)
    lsp = l - lz
    e = dG_in / T + (dG_in / T).max(1, keepdim=True)[0] + U * (n + 8 + 2 * l.abs() + lz.abs())
    er = (C + n + 4) * U
    Li = -(Q * lsp).sum(1) + (Qn * torch.log(sp + 1)).sum(1)
    Li_abs = (Q * lsp.abs() + Qn * torch.log(sp + 1)).sum(1)
    tol_Li = (Q * (e + er * lsp.abs()) + Qn * (sp * e + er * torch.log(sp + 1))).sum(1) + (n + 4) * U * Li_abs
    tol_L = tol_Li.sum() / n + (n + 4) * U * Li.abs().sum() / n + 1e-30
    wv = -Q + Qn * sp / (sp + 1)
    dG = (wv - sp * wv.sum(1, keepdim=True)) / (T * n)
    D = Q + Qn * sp / (sp + 1)
    kap = 2 * e.max(1, keepdim=True)[0] + (C + 2 * n + 8) * U
    tol_dG = kap * (D + sp * D.sum(1, keepdim=True)) / (T * n) + n * U * dG.abs()
    for side in (0, 1):
        a, b = fs64.clone().requires_grad_(side == 0), fw64.clone().requires_grad_(side == 1)
        ref = O.graph_contrast(a, b, Q, Qn, T)
        ref.backward()
        loss, df = ops.graph_contrast(fs.to(dev), fw.to(dev), p1.to(dev), p.to(dev), T, side)
        within(loss, ref.detach(), tol_L, f"graph_contrast loss n{n} dim{dim} side{side}")
        if side == 0:
            want, tol = a.grad, tol_dG @ fw64.abs()
            assert torch.allclose(dG @ fw64, want, rtol=0, atol=1e-12 * want.abs().max())
        else:
            want, tol = b.grad, tol_dG.t() @ fs64.abs()
            assert torch.allclose(dG.t() @ fs64, want, rtol=0, atol=1e-12 * want.abs().max())
        within(df, want, tol, f"graph_contrast dfeat n{n} dim{dim} side{side}")


def ntxent_ref(z, bs, T):
    """models.py:22-39 on unit rows z (restated on z, so that autograd gives dL/dz)."""
    n = 2 * bs
    S = z @ z.t()
    pos = torch.cat([torch.diag(S, bs), torch.diag(S, -bs)], 0)
    neg = 1.0 - torch.eye(n, dtype=S.dtype)
    den = (neg * torch.exp(S / T)).sum(1)
    return torch.sum(-torch.log(torch.exp(pos / T) / den)) / n


@pytest.mark.parametrize("dim", [7, 1024])
@pytest.mark.parametrize("bs", [5, 77, 129])
def test_ntxent(dev, bs, dim):
    from cmlpl_b200 import ops
    n, T = 2 * bs, 0.5
    z = O.normalize(torch.randn(n, dim, generator=gen(bs * 3 + dim), dtype=f64)).float()
    z64 = z.to(f64)
    zr = z64.clone().requires_grad_(True)
    ref = ntxent_ref(zr, bs, T)
    ref.backward()
    loss, dz = ops.ntxent(z.to(dev), bs, T)
    S = z64 @ z64.t()
    dS_in = product_bound(z64.abs() @ z64.abs().t(), dim)
    eye = torch.eye(n, dtype=torch.bool)
    ex = torch.where(eye, torch.zeros_like(S), torch.exp(S / T))
    den = ex.sum(1, keepdim=True)
    soft = ex / den
    part = torch.roll(torch.eye(n, dtype=f64), bs, 1)
    e = ((dS_in / T).masked_fill(eye, 0).max(1, keepdim=True)[0] * 2 + U * (n + 8 + 2 * S.abs().max(1, keepdim=True)[0] / T
                                                                           + den.log().abs()))
    Li = -(S * part).sum(1) / T + den[:, 0].log()
    tol_L = (e[:, 0] + (dS_in * part).sum(1) / T + U * (S * part).abs().sum(1) / T).sum() / n + (n + 4) * U * Li.abs().sum() / n
    within(loss, ref.detach(), tol_L, f"ntxent loss bs{bs} dim{dim}")
    dS = (soft - part) / (n * T)
    tol_dS = (soft * 2 * e + 2 * U * (soft + part)) / (n * T)
    dSs = dS + dS.t()
    tol_s = tol_dS + tol_dS.t() + U * dSs.abs()
    assert torch.allclose(dSs @ z64, zr.grad, rtol=0, atol=1e-12 * zr.grad.abs().max())
    within(dz, zr.grad, (tol_s + n * U * dSs.abs()) @ z64.abs(), f"ntxent dz bs{bs} dim{dim}")


def test_contrastive_loss_zero_row(dev):
    """ContrastiveLoss normalises like the reference's F.normalize: an all-zero embedding row gives the reference's
    finite loss and gradients (its gradient is dL/dz / 1e-12), not NaN."""
    from cmlpl_b200.tools.models import ContrastiveLoss
    bs, dim = 24, 64
    g = gen(14)
    ei, ej = torch.randn(bs, dim, generator=g), torch.randn(bs, dim, generator=g)
    ei[3] = 0
    a, b = ei.to(f64).requires_grad_(True), ej.to(f64).requires_grad_(True)
    ref = O.nt_xent(a, b, 0.5)
    ref.backward()
    assert torch.isfinite(ref) and torch.isfinite(a.grad).all() and torch.isfinite(b.grad).all()
    ad, bd = ei.to(dev).requires_grad_(True), ej.to(dev).requires_grad_(True)
    l = ContrastiveLoss(bs, device=dev, temperature=0.5)(ad, bd)
    l.backward()
    assert abs(float(l) - float(ref)) <= 1e-5 * abs(float(ref))
    zero = torch.zeros(bs, dtype=torch.bool)
    zero[3] = True
    for got, want, rows in ((ad.grad, a.grad, zero), (bd.grad, b.grad, torch.zeros(bs, dtype=torch.bool))):
        got = got.cpu().to(f64)
        for sel in (rows, ~rows):                         # the zero row's gradient is ~1e12 times the others'
            if sel.any():
                assert (got[sel] - want[sel]).abs().max() <= 1e-4 * want[sel].abs().max()


@pytest.mark.parametrize("C", [1, 33, 255])
def test_argmax_u8_ties(dev, C):
    """First index on exact ties (logits drawn from 7 values), all-equal rows, n off the 256-thread block and past the
    grid-stride wrap."""
    from cmlpl_b200 import ops
    g = gen(C)
    n = 8 * torch.cuda.get_device_properties(dev).multi_processor_count * 256 + 1077
    z = torch.randint(-3, 4, (n, C), generator=g).float()
    z[::97] = 1.5
    z[5::101] = float("-inf")
    got = ops.argmax_u8(z.to(dev)).cpu().numpy()
    assert np.array_equal(got, np.argmax(z.numpy(), 1).astype(np.uint8))


# ------------------------------------------------------------------------------------------------ 5. Adam
def test_fused_adam_many_tensors_empty_and_late(dev):
    """FusedAdam over 40 tensors (three table chunks of 16), with empty tensors, tensors that never get a gradient, and
    one whose gradient first appears at step 3 (its own launch at its own step count), over 10 steps against float64
    Adam.  Per tensor, the device result's largest distance from float64 is at most twice that of torch's own fp32
    Adam(foreach=False), plus 2 ulp.  (Per element the two fp32 results round differently -- the kernel rounds the bias
    corrections to fp32 and contracts to FMA -- so an element where torch happens to land on float64 can be a few ulp
    from the kernel's.)"""
    from cmlpl_b200.losses import FusedAdam
    g = gen(15)
    shapes = [(0,), (1,), (7,), (300,), (64, 60, 1, 1), (1000, 3), (0, 5), (33,), (1024,), (9,)] * 4
    never = {5, 17, 33}
    late = 21
    init = [torch.randn(s, generator=g) for s in shapes]
    p64 = [t.to(f64).requires_grad_(True) for t in init]
    p32 = [t.clone().requires_grad_(True) for t in init]
    pd = [t.to(dev).requires_grad_(True) for t in init]
    lr = 1e-3
    o64 = torch.optim.Adam(p64, lr=lr, foreach=False)
    o32 = torch.optim.Adam(p32, lr=lr, foreach=False)
    od = FusedAdam(pd, lr=lr)
    for step in range(1, 11):
        for i, s in enumerate(shapes):
            if i in never or (i == late and step < 3):
                continue
            gr = torch.randn(s, generator=g) * 10.0 ** -(step % 3)
            p64[i].grad, p32[i].grad, pd[i].grad = gr.to(f64), gr.clone(), gr.to(dev)
        o64.step(); o32.step(); od.step()
    ratios = []
    for i in range(len(shapes)):
        want = p64[i].detach().numpy()
        got = pd[i].detach().cpu().numpy().astype(np.float64)
        if i in never:
            assert np.array_equal(got, init[i].numpy())
            continue
        if want.size == 0:
            continue
        err = np.abs(got - want).max()
        err32 = np.abs(p32[i].detach().numpy().astype(np.float64) - want).max()
        ulp = float(np.spacing(np.float32(np.abs(want).max())))
        ratios.append(err / max(err32, 1e-30))
        assert err <= 2 * err32 + 2 * ulp, (i, err, err32, ulp)
    print("max |device - fp64| / max |torch fp32 - fp64| per tensor: max %.3f, median %.3f" % (max(ratios), np.median(ratios)))
    assert od.state[pd[late]]["step"] == 8 and od.state[pd[0]]["step"] == 10


# ------------------------------------------------------------------------------------------------ 6. fp32 mutual step
def test_mutual_step_fp32_honghu_w11(dev, golden_dir):
    """One --fp32_step step at the WHU-Hi HongHu shape (270 bands, 22 classes) on 11 x 11 windows: train.mutual_step
    against the oracle's ref_step, with the bars of test_gpu_train.py (scene_harness.relu_flips's docstring)."""
    from cmlpl_b200 import train as T
    B, K, bs, btu, epoch, batch_index, ptrs, seed = 270, 22, 128, 128, 1, 5, (512, 768), 2711
    ti = golden.load(os.path.join(golden_dir, "train_infer.npz"))
    g = gen(seed)
    inp = make_inputs(ti, bs, btu, B, K, g, 11)
    sd, sd1 = init_nets(B, K, seed, 11)
    sa = O.StepArgs(num_epochs=20, labeled_batch_size=bs)
    ost = O.make_state(sd, sd1, K, sa)
    queues = random_banks(5 * bs * 2, K, g)
    set_banks(ost, queues, ptrs)
    sa.thr = thr_for(oracle_step(copy.deepcopy(ost), inp, epoch, batch_index, sa), epoch, sa.num_epochs)
    args = argparse.Namespace(temperature=sa.temperature, thr=sa.thr, num_epochs=sa.num_epochs, queue_batch=sa.queue_batch,
                              alpha=sa.alpha, lr=sa.lr, labeled_batch_size=bs, dropout=0, noise=sa.noise)
    st = T.make_state(B, K, args, dev, w=11)
    st.Base.load_state_dict({k: v.detach() for k, v in sd.items()}, strict=False)
    st.Base1.load_state_dict({k: v.detach() for k, v in sd1.items()}, strict=False)
    for dst, src in zip((st.queue_feats, st.queue_probs, st.queue_feats1, st.queue_probs1), queues):
        dst.copy_(src)
    st.queue_ptr, st.queue_ptr1 = ptrs
    st.extras["keep_grads"] = True
    r = oracle_step(ost, inp, epoch, batch_index, sa)
    patches, spectra = assembled(inp, sa.noise)
    dd = lambda t: t.to(dev).contiguous()
    hist, aux = T.mutual_step(st, dd(patches[0]), dd(spectra[0]), dd(patches[1]), dd(spectra[1]), dd(inp["Y_l"]), epoch,
                              batch_index, args, drop_masks=(dd(inp["masks"][0]), dd(inp["masks"][1])))
    hist = hist.cpu().numpy()
    assert np.abs(hist - r["hist"]).max() <= 1e-4 * np.abs(r["hist"]).max(), (hist, r["hist"])
    assert rel(aux["logits"].cpu(), r["logits"]) < 1e-5 and rel(aux["logits1"].cpu(), r["logits1"]) < 1e-5
    assert rel(aux["probs"].cpu(), r["probs"]) < 1e-5 and rel(aux["probs1"].cpu(), r["probs1"]) < 1e-5
    assert torch.equal(aux["mask"].cpu(), r["mask"]) and torch.equal(aux["masks"].cpu(), r["masks"])
    assert 0.05 <= float(r["mask"].mean()) <= 0.95 and 0.05 <= float(r["masks"].mean()) <= 0.95
    for name in ("total1", "lc1", "con1", "cls1"):
        assert abs(float(aux[name]) - r[name]) <= 1e-4 * max(1.0, abs(r[name])), name
    with torch.no_grad():
        flips = (relu_flips(sd, patches[0], spectra[0], dev),
                 relu_flips(sd1, patches[1], spectra[1], dev))
    bars = [1e-4 if f == 0 else 5e-3 for f in flips]
    print("ReLU mask disagreements (net0, net1):", flips)
    for k in O.LIVE_KEYS:
        assert rel(aux["grads"][k].cpu(), r["grads"][k]) < bars[0], (k, flips)
        assert rel(aux["grads1"][k].cpu(), r["grads1"][k]) < bars[1], (k, flips)
        new = dict(st.Base.named_parameters())[k].detach().cpu().numpy()
        gk = r["grads"][k].numpy()
        gz = np.abs(gk) > 1e-3 * np.abs(gk).max()
        assert np.abs(new - ost.sd[k].detach().numpy())[gz].max() < (1e-6 if flips[0] == 0 else 5e-5), k
    assert (st.queue_ptr, st.queue_ptr1) == (ost.queue_ptr, ost.queue_ptr1)
    assert rel(st.queue_feats.cpu(), ost.queue_feats) < 1e-5 and rel(st.queue_probs1.cpu(), ost.queue_probs1) < 1e-5
