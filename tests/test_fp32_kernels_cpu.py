"""The algebra and the error bars behind tests/test_gpu_fp32_kernels.py, checked without a GPU.

  * softmax_js gradient: js_kernel computes dz_j = cf (p_j h_j - M_j - p_j sum_k (p_k h_k - M_k)),
    h = log M + 1 - log(p)/2 - log(t + 1e-5)/2, the form without M/p.  Here that formula, in float64 numpy, equals torch
    autograd of the reference's softmax_js_loss (trian_CCT.py:76-84), also on rows whose softmax underflows, where the
    old form's M/p is inf or 0/0.
  * the product bound |got - ref64| <= K 2^-23 (|A|.|B|) holds for an fp32 product in any summation order and fails for
    a product with one k-term dropped.
"""
import numpy as np
import torch
import torch.nn.functional as F

U = 2.0 ** -23          # one ulp of 1.0 in fp32 (twice the unit roundoff): the unit of every bar


def softmax_js_loss_ref(inputs, targets):
    """trian_CCT.py:76-84 restated (oracle/make_golden.py compiles the same function from the reference's source)."""
    epsilon = 1e-5
    M = (F.softmax(inputs, dim=1) + targets) * 0.5
    kl1 = F.kl_div(F.log_softmax(inputs, dim=1), M, reduction='mean')
    kl2 = F.kl_div(torch.log(targets + epsilon), M, reduction='mean')
    return (kl1 + kl2) * 0.5


def js_grad_np(z, t, scale=1.0):
    """js_kernel's gradient formula in float64 numpy (xlogy convention log M := 0 where M = 0, as the kernel)."""
    z = np.asarray(z, np.float64); t = np.asarray(t, np.float64)
    rows, C = z.shape
    lp = z - z.max(1, keepdims=True)
    lp = lp - np.log(np.exp(lp).sum(1, keepdims=True))
    p = np.exp(lp)
    M = 0.5 * (p + t)
    with np.errstate(divide="ignore"):
        lM = np.where(M > 0, np.log(np.where(M > 0, M, 1.0)), 0.0)
    h = lM + 1.0 - 0.5 * lp - 0.5 * np.log(t + 1e-5)
    q = p * h - M
    cf = scale * 0.5 / (rows * C)
    return cf * (q - p * q.sum(1, keepdims=True))


def js_grad_np_old(z, t):
    """The parent's form, p (g - sum g p) with g = h - M/p, in float64 (for the record of what it did)."""
    z = np.asarray(z, np.float64); t = np.asarray(t, np.float64)
    rows, C = z.shape
    lp = z - z.max(1, keepdims=True)
    lp = lp - np.log(np.exp(lp).sum(1, keepdims=True))
    p = np.exp(lp)
    M = 0.5 * (p + t)
    with np.errstate(divide="ignore", invalid="ignore"):
        lM = np.where(M > 0, np.log(np.where(M > 0, M, 1.0)), 0.0)
        g = lM + 1.0 - 0.5 * lp - M / p - 0.5 * np.log(t + 1e-5)
        gp = (g * p).sum(1, keepdims=True)
        return 0.5 / (rows * C) * p * (g - gp)


def js_inputs(rows, C, seed):
    """Logits and targets with the edges of js_kernel: ordinary rows, rows whose softmax underflows in fp32 (spread 120
    and 200) and in float64 (spread 1600, row 2), targets with exact zeros (row 0, also where its softmax underflows in
    fp32).  Row 2's targets have no zeros: where the softmax underflows in float64 too and the target is 0, the
    reference's own autograd is NaN (d xlogy(M, M)/dM = log M + 1 at M = 0)."""
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(rows, C, generator=g, dtype=torch.float64) * 2
    t = torch.softmax(torch.randn(rows, C, generator=g, dtype=torch.float64) * 3, 1)
    if C >= 2:
        for r, spread in ((0, 120.0), (1, 200.0), (2, 1600.0)):
            if r < rows:
                z[r] = torch.linspace(0, -spread, C, dtype=torch.float64)[torch.randperm(C, generator=g)]
        t[0] = 0.0; t[0, -1] = 1.0                  # exact zeros, also at entries whose softmax is 0 in fp32
        if rows > 3:
            t[3, : C // 2] = 0.0
            t[3] = t[3] / t[3].sum()
    return z, t


def test_js_gradient_formula_matches_reference_autograd():
    for rows, C, seed in ((5, 9, 1), (7, 22, 2), (4, 2, 3), (3, 1, 4), (6, 300, 5)):
        z, t = js_inputs(rows, C, seed)
        zr = z.clone().requires_grad_(True)
        loss = softmax_js_loss_ref(zr, t)
        loss.backward()
        want = zr.grad.numpy()
        assert np.isfinite(want).all() and np.isfinite(float(loss))
        got = js_grad_np(z.numpy(), t.numpy())
        assert np.abs(got - want).max() <= 1e-13 * max(np.abs(want).max(), 1e-300), (rows, C)
        got_s = js_grad_np(z.numpy(), t.numpy(), scale=-3.5)
        assert np.abs(got_s + 3.5 * want).max() <= 1e-13 * 3.5 * np.abs(want).max()


def test_js_old_form_is_nan_where_the_softmax_underflows():
    """The row with spread 1600 underflows even in float64: there the parent's M/p form gives NaN for the whole row, and
    the new form the reference's finite gradient.  (In fp32 the same happens from a spread of about 88 on.)"""
    z, t = js_inputs(5, 9, 1)
    old = js_grad_np_old(z.numpy(), t.numpy())
    assert np.isnan(old[2]).all() and np.isfinite(old[3:]).all()
    assert np.isfinite(js_grad_np(z.numpy(), t.numpy())).all()


def product_bound(absprod, K):
    """|got - ref64| <= K 2^-23 (|A|.|B|): any order of an fp32 sum of K products (also split-K partials added with
    atomics) stays inside it; 2^-23 is twice fp32's unit roundoff."""
    return K * U * absprod


def test_product_bound_holds_for_fp32_and_catches_a_dropped_term():
    g = np.random.default_rng(7)
    for M, N, K in ((17, 33, 1000), (64, 65, 130), (5, 7, 16)):
        A = g.standard_normal((M, K)).astype(np.float32)
        B = g.standard_normal((K, N)).astype(np.float32)
        ref = A.astype(np.float64) @ B.astype(np.float64)
        tol = product_bound(np.abs(A).astype(np.float64) @ np.abs(B).astype(np.float64), K)
        got = A @ B                                               # fp32 BLAS, its own order
        assert (np.abs(got - ref) <= tol).all()
        seq = np.zeros((M, N), np.float32)                        # one k at a time, fp32 rounding at every add
        for k in range(K):
            seq = seq + np.outer(A[:, k], B[k]).astype(np.float32)
        assert (np.abs(seq - ref) <= tol).all()
        dropped = seq - np.outer(A[:, K // 2], B[K // 2]).astype(np.float32)
        assert (np.abs(dropped - ref) > tol).mean() > 0.5, (M, N, K)
