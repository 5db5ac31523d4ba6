"""Helpers shared by the GPU scene, preprocessing and training tests: the relative error every bar is stated in, the
near-tie rule for labels, the scene path mode, the random nets and synthetic raw scenes the scene tests run, the raw
layouts, the device fit's moments and the fp32 step's ReLU-mask flips.  Imported as a plain module (pytest puts
tests/ on sys.path); it holds no tests."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O


def rel(a, b):
    """max|a - b| / max|b| in float64; a and b may be numpy arrays or tensors on any device (two tensors on one device
    are compared there).  NaN in a gives NaN, which fails every bar."""
    if torch.is_tensor(a) and torch.is_tensor(b) and a.device == b.device:
        a, b = a.detach().double(), b.detach().double()
        return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    a = np.asarray(a.detach().cpu() if torch.is_tensor(a) else a, dtype=np.float64)
    b = np.asarray(b.detach().cpu() if torch.is_tensor(b) else b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def near_ties_only(lab, lab_ref, log_ref, bar=2e-3):
    """every label that differs from the reference sits on a reference top-2 margin below the bar"""
    lab, lab_ref, log_ref = np.asarray(lab), np.asarray(lab_ref), np.asarray(log_ref, dtype=np.float64)
    diff = lab != lab_ref
    srt = np.sort(log_ref, 1)
    return bool(np.all((srt[diff, -1] - srt[diff, -2]) <= bar * np.abs(log_ref).max()))


class path_mode:
    """cmlpl_set_scene_path_mode for a block (the mode is per host thread; 1 is the default)"""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        from cmlpl_b200 import _lib
        _lib.call("cmlpl_set_scene_path_mode", self.mode)

    def __exit__(self, *exc):
        from cmlpl_b200 import _lib
        _lib.call("cmlpl_set_scene_path_mode", 1)


def scene_net(B, K, w, seed, dev):
    """random-init BaseNet2 (w = 11: the 1280-input classifier of the odd-window variant) and its cpu state dict"""
    from cmlpl_b200.tools.models import BaseNet2
    torch.manual_seed(seed)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    return net, {k: v.detach().cpu() for k, v in net.state_dict().items()}


def raw_scene(dev, R, C, B, K, seed):
    """synthetic raw scene, its float64 oracle preprocessing, and the device preprocessing with the oracle's PCA signs"""
    from cmlpl_b200 import preprocess, synth
    cube_u16, _ = synth.synth_scene(R, C, B, K, seed=seed)
    ref_cube, ref_spec = O.preprocess(cube_u16, 60)
    raw = torch.from_numpy(cube_u16.reshape(-1, B).copy()).to(dev)
    pp = preprocess.fit(raw, 60)
    cube, _ = preprocess.apply(raw, pp, want_spectra=False)
    sgn = np.sign((cube.cpu().numpy().reshape(R, C, 60) * ref_cube).sum((0, 1)))   # singular vectors: up to sign
    pp.U = pp.U * sgn[None, :]
    pp._dev = None
    return cube_u16, raw, pp, ref_cube.astype(np.float32), ref_spec.astype(np.float32)


def as_layout(cube, interleave, dev):
    """[rows, cols, B] numpy cube -> contiguous device tensor in the layout."""
    a = {"bip": cube.reshape(-1, cube.shape[2]), "bil": cube.transpose(0, 2, 1), "bsq": cube.transpose(2, 0, 1)}[interleave]
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def fit_moments(raw, code, rows, cols, B):
    """Band means and the full (symmetrised) Gram matrix of the device fit: cmlpl_preprocess_fit_f64 when cols is None
    (BIP rows), cmlpl_preprocess_fit_cube_f64 otherwise."""
    from cmlpl_b200 import _lib
    mean = torch.empty(B, dtype=torch.float64, device=raw.device)
    gram = torch.empty(B, B, dtype=torch.float64, device=raw.device)
    if cols is None:
        _lib.call("cmlpl_preprocess_fit_f64", raw.data_ptr(), code, rows, B, mean.data_ptr(), gram.data_ptr(),
                  torch.cuda.current_stream().cuda_stream)
    else:
        _lib.call("cmlpl_preprocess_fit_cube_f64", raw.data_ptr(), code, rows, cols, B, mean.data_ptr(), gram.data_ptr(),
                  torch.cuda.current_stream().cuda_stream)
    g = gram.cpu().numpy()
    return mean.cpu().numpy(), np.triu(g) + np.triu(g, 1).T


def relu_flips(sd, x, y, dev):
    """Number of ReLU inputs whose sign differs between the CUDA fp32 forward and torch CPU fp32.
    Summation order moves activations by ~2e-6; an activation that is zero to within that flips its
    ReLU mask, and ONE flip moves a conv weight gradient (a sum of ~1e5 signed terms) by ~1e-3 of its
    max.  Gradient bars are therefore 1e-4 when no mask differs and 5e-3 otherwise."""
    from cmlpl_b200 import ops
    d = lambda t: t.detach().to(dev).contiguous()
    a0 = F.conv2d(x, sd["conv0.weight"], sd["conv0.bias"])
    a1 = F.relu(F.conv2d(a0, sd["conv1.weight"], sd["conv1.bias"], padding=1) + a0)
    p1 = F.avg_pool2d(a1, 2, 2)
    a2 = F.relu(F.conv2d(p1, sd["conv2.weight"], sd["conv2.bias"], padding=1) + p1)
    h = F.relu(F.linear(y, sd["feat_spe.weight"], sd["feat_spe.bias"]))
    m0 = ops.conv2d(d(x), d(sd["conv0.weight"]), d(sd["conv0.bias"]))
    m1 = ops.conv2d(m0, d(sd["conv1.weight"]), d(sd["conv1.bias"]), res=m0, relu=True)
    mp1 = ops.avgpool2(m1)
    m2 = ops.conv2d(mp1, d(sd["conv2.weight"]), d(sd["conv2.bias"]), res=mp1, relu=True)
    mh = ops.sgemm(d(y), d(sd["feat_spe.weight"]), transB=True, bias=d(sd["feat_spe.bias"]), act=1)
    assert rel(m1.cpu(), a1) < 1e-5 and rel(m2.cpu(), a2) < 1e-5 and rel(mh.cpu(), h) < 1e-5
    return sum(int(((m.cpu() > 0) != (a > 0)).sum()) for m, a in ((m1, a1), (m2, a2), (mh, h)))
