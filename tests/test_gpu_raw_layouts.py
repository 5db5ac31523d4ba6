"""Raw cubes in BIL and BSQ and int16 samples on the GPU (-m gpu).

Nothing after conv0's loader and the spectral branch's input conversion depends on the layout, and both loaders produce
the same operands from every layout, so every claim here is exact (torch.equal):
  * cmlpl_scene_infer_raw from BIL and BSQ against BIP, labels and logits, on every path the raw entry point runs: dense
    (<= 16 and 17-32 classes, w = 20 and 11), path mode 0, conv0_tc + the CUDA-core head (240 bands), the K-sliced conv0
    + the CUDA-core head (270, 425 bands); and in row bands with slab_row0 > 0, where a BSQ plane stride taken from the
    scene instead of the slab would read the wrong rows;
  * int16 against the same values in float32 (negative ones included), and uint16 against the same values in int16;
  * cmlpl_preprocess_fit_cube_f64 in every layout and sample type against numpy float64 (1e-12 of the largest entry:
    float64 atomics reorder the sums);
  * StreamedRawScene from BIL / BSQ host cubes against the BIP one.
One Preproc, fitted on the BIP cube, serves every layout.
"""

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

LAYOUTS = ("bip", "bil", "bsq")


def as_layout(cube, interleave, dev):
    """[rows, cols, B] numpy cube -> contiguous device tensor in the layout."""
    a = {"bip": cube.reshape(-1, cube.shape[2]), "bil": cube.transpose(0, 2, 1), "bsq": cube.transpose(2, 0, 1)}[interleave]
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def scene(dev, R, C, B, K, w, seed):
    from cmlpl_b200 import preprocess, synth
    from cmlpl_b200.tools.models import BaseNet2
    cube, _ = synth.synth_scene(R, C, B, K, seed=seed)
    pp = preprocess.fit(as_layout(cube, "bip", dev), 60)
    torch.manual_seed(seed)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    return cube, pp.folded_conv0(sd["conv0.weight"], sd["conv0.bias"], dev), net.packed_weights(w)


def infer(raw, il, folded, packed, K, C, w, **kw):
    from cmlpl_b200 import ops
    return ops.scene_infer_raw(raw, folded, packed, K, C, w, want_logits=True, interleave=il, **kw)


def assert_same(got, want):
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


#   id              B    K   w   path mode
SHAPES = {
    "b103_k9":      (103, 9, 20, 1),      # dense path
    "b103_k9_pm0":  (103, 9, 20, 0),      # per-pixel kernels + tensor-core spectral branch
    "b200_k16_w11": (200, 16, 11, 1),
    "b103_k20":     (103, 20, 20, 1),     # NC = 32
    "b240_k16":     (240, 16, 20, 1),     # conv0_tc + CUDA-core spectral head
    "b270_k22":     (270, 22, 20, 1),     # K-sliced conv0 + CUDA-core spectral head
    "b425_k16":     (425, 16, 20, 1),
}


@pytest.mark.parametrize("dtype", ["u16", "f32"])
@pytest.mark.parametrize("case", list(SHAPES))
def test_bil_and_bsq_match_bip(dev, case, dtype):
    from cmlpl_b200 import _lib
    B, K, w, mode = SHAPES[case]
    R, C = 29, 37
    cube, folded, packed = scene(dev, R, C, B, K, w, seed=B + K + w)
    cube = cube if dtype == "u16" else cube.astype(np.float32)
    _lib.call("cmlpl_set_scene_path_mode", mode)
    try:
        ref = infer(as_layout(cube, "bip", dev), "bip", folded, packed, K, C, w)
        for il in ("bil", "bsq"):
            assert_same(infer(as_layout(cube, il, dev), il, folded, packed, K, C, w), ref)
        # row bands at the top edge, in the middle and at the bottom edge, each from its own halo slab
        lo, hi = w // 2, w - w // 2 - 1
        for a, b in [(0, 6), (6, 17), (17, 29)]:
            s0, s1 = max(0, a - lo), min(R, b + hi)
            want = (ref[0][a * C:b * C], ref[1][a * C:b * C])
            for il in LAYOUTS:
                got = infer(as_layout(cube[s0:s1], il, dev), il, folded, packed, K, C, w, band_row0=a, band_rows=b - a,
                            scene_rows=R, slab_row0=s0)
                assert_same(got, want)
    finally:
        _lib.call("cmlpl_set_scene_path_mode", 1)


@pytest.mark.parametrize("B,K", [(103, 9), (240, 16), (270, 22)])
def test_int16_matches_the_same_values(dev, B, K):
    """int16 with negative values == the same values as float32; uint16 below 32768 == the same values as int16."""
    R, C, w = 29, 37, 20
    cube, folded, packed = scene(dev, R, C, B, K, w, seed=B * 3 + K)
    signed = (cube.astype(np.int32) - 3000).astype(np.int16)
    assert signed.min() < 0 and cube.max() < 32768
    for il in LAYOUTS:
        assert_same(infer(as_layout(signed, il, dev), il, folded, packed, K, C, w),
                    infer(as_layout(signed.astype(np.float32), il, dev), il, folded, packed, K, C, w))
        assert_same(infer(as_layout(cube, il, dev), il, folded, packed, K, C, w),
                    infer(as_layout(cube.astype(np.int16), il, dev), il, folded, packed, K, C, w))


def fit_moments(raw, code, rows, cols, B):
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


@pytest.mark.parametrize("B", [103, 270])
def test_fit_cube_matches_numpy(dev, B):
    from cmlpl_b200 import synth
    from cmlpl_b200.preprocess import INTERLEAVE
    R, C = 41, 53
    u16, _ = synth.synth_scene(R, C, B, 9, seed=B)
    cubes = {0: u16, 1: u16.astype(np.float32) * 0.37, 2: (u16.astype(np.int32) - 3000).astype(np.int16)}
    for code, cube in cubes.items():
        x = cube.reshape(-1, B).astype(np.float64)
        mu = x.mean(0)
        gram = (x - mu).T @ (x - mu)
        bar_m, bar_g = 1e-12 * np.abs(mu).max(), 1e-12 * np.abs(gram).max()
        m, g = fit_moments(as_layout(cube, "bip", dev), code, R * C, None, B)
        assert np.abs(m - mu).max() <= bar_m and np.abs(g - gram).max() <= bar_g, ("fit_f64", code)
        for il in LAYOUTS:
            m, g = fit_moments(as_layout(cube, il, dev), code | INTERLEAVE[il], R, C, B)
            err_m, err_g = np.abs(m - mu).max() / np.abs(mu).max(), np.abs(g - gram).max() / np.abs(gram).max()
            print("B = %d, sample %d, %s: mean %.1e, gram %.1e (relative to the largest entry)" % (B, code, il, err_m, err_g))
            assert err_m <= 1e-12 and err_g <= 1e-12, (code, il)


def pinned(cube, il):
    a = {"bip": cube.reshape(-1, cube.shape[2]), "bil": cube.transpose(0, 2, 1), "bsq": cube.transpose(2, 0, 1)}[il]
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


@pytest.mark.parametrize("nsplit", [1, 2, 3])
def test_streamed_raw_scene_from_bil_and_bsq(dev, nsplit):
    """The rank's slab [s0, s1) lies strictly inside the scene, so a BSQ copy pitch or offset taken from the scene instead
    of the slab would misplace rows.  After every call the device slab must hold the host cube exactly, the labels must
    be the one-call labels of the same rows, and h2d_bytes (summed from the copies issued) the host cube's size."""
    from cmlpl_b200._lib import CmlplError
    from cmlpl_b200.tools.hyper_tools import StreamedRawScene
    R, C, B, K, w = 60, 37, 103, 9, 20
    cube, folded, packed = scene(dev, R, C, B, K, w, seed=nsplit)
    row0, rows = 15, 25
    s0, s1 = max(0, row0 - w // 2), min(R, row0 + rows + w - w // 2 - 1)
    assert 0 < s0 and s1 < R
    ref = infer(as_layout(cube, "bip", dev), "bip", folded, packed, K, C, w)[0][row0 * C:(row0 + rows) * C].cpu()
    cubes = {torch.uint16: cube[s0:s1], torch.int16: cube[s0:s1].astype(np.int16),
             torch.float32: cube[s0:s1].astype(np.float32)}
    nbytes = {}
    for dt, c in cubes.items():
        for il in LAYOUTS:
            st = StreamedRawScene(None, R, C, B, K, w, nsplit=nsplit, row0=row0, rows=rows, raw_dtype=dt, interleave=il)
            host = pinned(c, il)
            for _ in range(3):                        # both buffer sets, then the first one again
                st(packed, host, folded=folded)
                got = st.wait().clone()
                assert torch.equal(got, ref), (dt, il)
                assert torch.equal(st.sets[(st.calls - 1) & 1]["raw"].cpu(), host), (dt, il)
                assert st.h2d_bytes == host.nbytes
            nbytes[dt, il] = st.h2d_bytes
            if il != "bip":
                with pytest.raises(CmlplError):
                    st(packed, host)                  # preprocess.apply + cmlpl_scene_infer read BIP only
    for il in LAYOUTS:
        assert nbytes[torch.int16, il] * 2 == nbytes[torch.float32, il] == (s1 - s0) * C * B * 4
