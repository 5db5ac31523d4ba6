"""Sensor-like scenes on the CPU: the conditioning of ``oracle.sensor_scene``, and the error bounds that
test_gpu_sensor_scenes.py holds the device preprocessing and the folded raw conv0 to, checked against numpy emulations
of the kernels' arithmetic.  Each bound must hold for the emulated kernel and fail for a known mistake.

The bounds are first-order error analyses of the kernels, evaluated from their actual operands (u = 2^-24):

* ``preprocess_apply_kernel`` (preprocess.cu): c_b = fl(x_b - mu32_b), cube_k = fl(sum_b c_b * Us32_bk (fma chain) -
  shift_k).  |cube - ref64| <= (B + 4) u sum_b |x_b - mu32_b| |Us32_bk| + sum_b |mu32_b - mu_b| |Us32_bk| + 2u |shift_k|:
  one rounding per fma, one for c_b, one for Us32, one for the subtraction of the shift, plus the f32 band means'
  own rounding, which the kernel cannot undo (it is a bias of the centred value, not a relative error).
* the raw conv0 (conv0_sm100.cu, all three variants): z = fl(fl(x - mu32) * inv_sigma32), w = fl(wf32 * fl(1 / inv_sigma32));
  both split into fp16 hi + lo, and each 16-band K-step adds hi.hi + hi.lo + lo.hi into an f32 accumulator, + bias,
  stored as fp16.  Before the fp16 store the error is at most
      sum_k |z_k||w_k| (3 * 2^-22 + 16 * 2^-23 + 8u)      split: lo rounded to fp16, lo.lo dropped (2^-22 each);
                                                           a 16-product MMA (15 roundings, 2^-23 to allow truncation);
                                                           f32 rounding of z, w and of the folded weights
      + 2^-23 * 3 * sum_j |S_j|                            the accumulator after each K-step j (S_j the exact prefix sum)
      + sum_k |mu32_k - mu_k| |wf_k|                       the f32 band means
      + 2^-25 (sum_k |z_k| + sum_k |w_k|)                  a lo part in fp16's subnormal range (absolute 2^-25)
      + u (|F| + |bias|)                                   the bias add
  and the fp16 store adds half an fp16 ulp.  sum |z||w| is the cancellation: on a sensor-like scene it is up to 1e5 to 1e7
  times |F0|, because the trailing PCA components are small differences of large band values."""
import numpy as np
import pytest

from oracle import cmlpl_oracle as O

U = 2.0 ** -24
f16, f32, f64 = np.float16, np.float32, np.float64


# ------------------------------------------------------------------------------------------- bounds (shared with -m gpu)
def apply_bound(X, mu32, mu64, Us32, shift64):
    """Per pixel and component: the bound on |preprocess.apply's PCA cube - float64| (module docstring)."""
    X = np.asarray(X, f64)
    aUs = np.abs(np.asarray(Us32, f64))
    B = X.shape[1]
    mu32 = np.asarray(mu32, f64)
    return ((B + 4) * U * (np.abs(X - mu32) @ aUs) + (np.abs(mu32 - mu64) @ aUs)[None]
            + 2 * U * np.abs(shift64)[None])


def conv0_operands(X, mu32, inv_sigma32, wf32):
    """z [n, B] and w [B, 64] as the raw conv0 kernels form them in f32 before the hi / lo split."""
    z = ((np.asarray(X, f32) - mu32).astype(f32) * inv_sigma32).astype(f32)
    w = (wf32 * (f32(1) / inv_sigma32)[:, None]).astype(f32)
    return z, w


def conv0_bar(X, mu32, mu64, inv_sigma32, wf32, wf64, bf64, ref):
    """Per position and output channel: the bound on |conv0 map (fp16) - float64| (module docstring)."""
    z, w = conv0_operands(X, mu32, inv_sigma32, wf32)
    z, w = z.astype(f64), w.astype(f64)
    T = np.abs(z) @ np.abs(w)
    S, acc = np.zeros_like(T), np.zeros_like(T)
    for j in range(0, z.shape[1], 16):
        acc += z[:, j:j + 16] @ w[j:j + 16]
        S += 3 * np.abs(acc)
    E = (T * (3 * 2.0 ** -22 + 16 * 2.0 ** -23 + 8 * U) + 2.0 ** -23 * S
         + (np.abs(np.asarray(mu32, f64) - mu64) @ np.abs(wf64))[None]
         + 2.0 ** -25 * (np.abs(z).sum(1, keepdims=True) + np.abs(w).sum(0)[None])
         + U * (np.abs(ref) + np.abs(bf64)[None]))
    half_ulp = 0.5 * np.spacing(np.minimum(np.abs(ref) + E, 65504).astype(f16)).astype(f64)
    return half_ulp + E, T


# ------------------------------------------------------------------------------------------- kernel emulations
def emulate_apply(X, mu32, Us32, shift32, acc_dtype=f32):
    """preprocess_apply_kernel in numpy: f32 centring, an fma chain over the bands (exact product, one rounding)."""
    c = (np.asarray(X, f32) - mu32).astype(f32).astype(f64)
    acc = np.zeros((c.shape[0], Us32.shape[1]), acc_dtype)
    Us = np.asarray(Us32, f64)
    for b in range(c.shape[1]):
        acc = (acc.astype(f64) + c[:, b:b + 1] * Us[b]).astype(acc_dtype)
    return (acc.astype(f32) - shift32).astype(f32)


def emulate_conv0(X, mu32, inv_sigma32, wf32, bf32, lo=True):
    """The raw conv0 in numpy: hi / lo fp16 operands, hi.hi + hi.lo + lo.hi per 16-band K-step into f32, + bias, fp16.
    ``lo=False``: hi.hi only."""
    z, w = conv0_operands(X, mu32, inv_sigma32, wf32)
    zh, wh = z.astype(f16), w.astype(f16)
    zl, wl = (z - zh.astype(f32)).astype(f16), (w - wh.astype(f32)).astype(f16)
    terms = [(zh, wh), (zh, wl), (zl, wh)] if lo else [(zh, wh)]
    acc = np.zeros((z.shape[0], w.shape[1]), f32)
    for j in range(0, z.shape[1], 16):
        for a, b in terms:
            acc = (acc.astype(f64) + a[:, j:j + 16].astype(f64) @ b[j:j + 16].astype(f64)).astype(f32)
    return (acc + bf32).astype(f32).astype(f16).astype(f64)


def folded_reference(pp, seed=0):
    """A conv0 of BaseNet2's init range folded with ``pp`` in float64, and its f32 copies as Preproc.folded_conv0 makes them."""
    rng = np.random.default_rng(seed)
    W0 = rng.uniform(-1, 1, (64, 60)) / np.sqrt(60)
    b0 = rng.uniform(-1, 1, 64) / np.sqrt(60)
    Us = pp["U"] / pp["pca_sigma"][None]
    wf, bf = Us @ W0.T, b0 - W0 @ (pp["pca_mu"] / pp["pca_sigma"])
    return wf, bf


# (B, K, noise DN, sample, DC offset): the GPU tests' scene kinds
CASES = [(103, 9, 8.0, "u16", 20000.0), (103, 9, 1.0, "u16", 0.0), (224, 16, 1.0, "u16", 20000.0),
         (270, 22, 8.0, "i16", 0.0), (512, 32, 1.0, "f32", 0.0)]


def _scene(B, K, nd, sample, dc, R=48, C=40):
    cube, _ = O.sensor_scene(R, C, B, K, nd, seed=B + int(nd), sample=sample, dc=dc)
    return cube, cube.reshape(-1, B).astype(f64), O.preprocess_params(cube, 60)


@pytest.mark.parametrize("B,K,nd,sample,dc", CASES + [(103, 9, 0.5, "u16", 20000.0)])
def test_sensor_scene_is_what_its_name_says(B, K, nd, sample, dc):
    """lambda_1 / lambda_60 of the band covariance >= 1e5 at 8 DN and >= 1e7 at 1 DN or less; no zero-variance band;
    the sample type's range (DC offset, negative int16 values, reflectance)."""
    cube, X, pp = _scene(B, K, nd, sample, dc)
    ev = np.linalg.eigvalsh(np.cov((X - X.mean(0)).T))[::-1]
    ratio = ev[0] / ev[59]
    print("B = %d, %s, %.1f DN: lambda_1 / lambda_60 = %.1e, smallest band std %.3g" % (B, sample, nd, ratio,
                                                                                        pp["sigma"].min()))
    assert ratio >= (1e5 if nd >= 8 else 1e7)
    assert pp["sigma"].min() > 0.05 * pp["sigma"].max()
    assert cube.dtype == {"u16": np.uint16, "i16": np.int16, "f32": np.float32}[sample]
    if sample == "u16" and dc:
        assert X.min() > dc and pp["mu"].min() > 5 * pp["sigma"].max()
    if sample == "i16":
        assert (X < 0).mean() > 0.01
    if sample == "f32":
        assert 0 < X.min() and X.max() < 1.5


@pytest.mark.parametrize("B,K,nd,sample,dc", CASES)
def test_apply_bound_holds_for_f32_and_catches_fp16(B, K, nd, sample, dc):
    """The apply bound against the emulated kernel; the same bound fails when the band means are taken as fp16 or the
    projection accumulates in fp16."""
    _, X, pp = _scene(B, K, nd, sample, dc)
    Us64, sh64 = pp["U"] / pp["pca_sigma"][None], pp["pca_mu"] / pp["pca_sigma"]
    mu32, Us32, sh32 = pp["mu"].astype(f32), Us64.astype(f32), sh64.astype(f32)
    ref = (X - pp["mu"]) @ Us64 - sh64
    bound = apply_bound(X, mu32, pp["mu"], Us32, sh64)
    ratio = lambda got: float((np.abs(got - ref) / bound).max())
    ok = ratio(emulate_apply(X, mu32, Us32, sh32))
    mu16 = ratio(emulate_apply(X, pp["mu"].astype(f16).astype(f32), Us32, sh32))
    acc16 = ratio(emulate_apply(X, mu32, Us32, sh32, acc_dtype=f16))
    print("B = %d, %s, %.0f DN: apply error / bound: f32 %.3f, fp16 mu %.1f, fp16 accumulator %.1f" % (B, sample, nd, ok,
                                                                                                     mu16, acc16))
    assert ok <= 1.0 and mu16 > 1.0 and acc16 > 1.0


@pytest.mark.parametrize("B,K,nd,sample,dc", CASES)
def test_conv0_bound_holds_for_split_operands_and_catches_a_dropped_lo(B, K, nd, sample, dc):
    """The conv0 map bound against the emulated hi / lo kernel; the same bound fails for hi.hi alone.  The emulated error
    also stays under the outer bar of 1e-3 of the largest |F0|."""
    _, X, pp = _scene(B, K, nd, sample, dc)
    wf, bf = folded_reference(pp, seed=B)
    mu32, is32 = pp["mu"].astype(f32), (1.0 / pp["sigma"]).astype(f32)
    ref = (X - pp["mu"]) @ wf + bf
    bar, T = conv0_bar(X, mu32, pp["mu"], is32, wf.astype(f32), wf, bf, ref)
    got = emulate_conv0(X, mu32, is32, wf.astype(f32), bf.astype(f32))
    hi = emulate_conv0(X, mu32, is32, wf.astype(f32), bf.astype(f32), lo=False)
    ok, bad = float((np.abs(got - ref) / bar).max()), float((np.abs(hi - ref) / bar).max())
    outer = float(np.abs(got - ref).max() / np.abs(ref).max())
    print("B = %d, %s, %.0f DN: conv0 error / bar: split %.3f, hi only %.1f; error / max|F0| %.1e; sum|z||w| / |F0| up to"
          " %.1e" % (B, sample, nd, ok, bad, outer, (T / np.maximum(np.abs(ref), 1e-3 * np.abs(ref).max())).max()))
    assert ok <= 1.0 and bad > 1.0 and outer < 1e-3
