"""The intermediate tensors of the dense scene path, stage by stage (tools/models.py:133-150 for all pixels at once):
the conv0 map F0, the pooled conv1 parity planes  PM[A][B]  that conv1_pool_kernel writes, the half-pooled conv2 maps
YP[Al][Be]  that conv2_scene_kernel writes (border halves of the 2x2 pool added in its epilogue), the row maps
M[I] = sum_J L[I][J](., x + 2J)  that pool2_cls_kernel writes and the quarter partials of spectral_logits_kernel, each
against the float64 references of tests/dense_refs.py on the kernel's own fp16 inputs, entry by entry within the
elementwise bound of fp16 output rounding plus fp32 accumulation (dense_refs.bound), and with the max-relative bars:
fp16-rounded maps 1e-3 * max|ref| (one rounding, 4.9e-4 relative), fp32 class partial maps 1e-4, spectral partials
5e-4 * max|ref|, logits 1e-3 * max|ref| (north_star).  Outputs are NaN-prefilled; the entries checked are the ones the
head depends on (dense_refs.consumed).

Small scenes (one tile per CTA) also go through the per-pixel kernels (path mode 0) and the CPU oracle.  The many-tile
cases (dense_refs.CASES: the whole PaviaU scene, c5 bands of an 8192 x 8192 scene at w = 11, a Houston-2018 band at
32 classes, w = 11 at 32 classes) run every persistent kernel over many tiles per CTA, so their rings wrap, their
accumulator stages and phases repeat and their tile orders matter; there the head's conv logits are also checked
against a per-pixel float64 tower and the driver (ops.scene_infer) against the stage chain bit for bit."""
import time

import numpy as np
import pytest
import torch

import dense_refs as D
from oracle import cmlpl_oracle as O
from scene_harness import rel

pytestmark = pytest.mark.gpu


def slab_of(SR, r0, R, w):
    """scene rows [s0, s1) the mirrored halo of band rows [r0, r0 + R) reads"""
    rows = D.mirror(r0 + np.arange(R + w - 1) - w // 2, SR)
    return int(rows.min()), int(rows.max()) + 1


def stage_chain(cube, spectra, sd, packed, SR, s0, r0, R, B, K, w, perturb=False):
    """Every stage through its entry point on NaN-prefilled outputs, each against its float64 reference within its
    bound on the entries the head consumes.  Returns the results, the kernel's tensors and the worst ratios."""
    from cmlpl_b200 import _lib
    dev = cube.device
    C = cube.shape[1]
    st = torch.cuda.current_stream().cuda_stream
    PR, PC = R + w - 1, C + w - 1
    PR2, PC2 = (R + w) // 2, (C + w) // 2
    n = R * C
    NC = 16 if K <= 16 else 32
    ncls, ncell = D.nclass(w), D.GEOM[w]["ncell"]
    res, ratios = {}, {}
    nan = float("nan")
    f0 = torch.full((8 * PR * PC * 8,), nan, dtype=torch.float16, device=dev)
    pmq = torch.full((9, 4, 8, PR2, PC2, 8), nan, dtype=torch.float16, device=dev)
    yq = torch.full((9, 4, 8, PR2, PC2, 8), nan, dtype=torch.float16, device=dev)
    lmap = torch.full((4, 5, NC // 4, PR2, PC2, 4), nan, dtype=torch.float32, device=dev)
    mt, kc = (n + 127) // 128, ((B + 15) // 16) * 2
    x16 = torch.full((mt * kc * 1024,), nan, dtype=torch.float16, device=dev)
    part = torch.full((4, mt * 128, NC), nan, dtype=torch.float32, device=dev)
    _lib.call("cmlpl_spectral_logits_tc", spectra.data_ptr(), n, B, K, w, packed.data_ptr(), x16.data_ptr(), part.data_ptr(), st)
    _lib.call("cmlpl_conv0_map_f16", cube.data_ptr(), SR, C, s0, cube.shape[0], w, r0, R, packed.data_ptr(), f0.data_ptr(), st)
    _lib.call("cmlpl_conv1_pool_planes_f16", f0.data_ptr(), C, w, R, packed.data_ptr(), pmq.data_ptr(), st)
    _lib.call("cmlpl_conv2_scene_f16", pmq.data_ptr(), C, w, R, packed.data_ptr(), yq.data_ptr(), st)
    _lib.call("cmlpl_pool2_cls_f16", yq.data_ptr(), C, w, R, B, K, packed.data_ptr(), lmap.data_ptr(), st)
    torch.cuda.synchronize()
    m_use, yp_use, pm_use = (torch.from_numpy(a).to(dev) for a in D.consumed(R, C, w))
    T = D.tile_constants()

    # ---- conv0 map on the mirrored slab
    F0k = D.dense_f0(f0, PR, PC)
    ref, a = D.conv0_map(cube, sd["conv0.weight"], sd["conv0.bias"], SR, s0, r0, R, w)
    bnd = D.bound(ref, a, D.N_CONV0, True)
    ratios["conv0"] = D.ratio(F0k, ref, bnd)
    res["f0_nan"], res["f0_rel"] = int(torch.isnan(F0k).sum()), rel(F0k, ref)
    if perturb:                                         # channels 24-31 of the first position of conv0's second tile
        at = (slice(24, 32), 128 // PC, 128 % PC)
        frm = (slice(24, 32), 127 // PC, 127 % PC)
        res["perturbed"] = {"conv0": D.ratio(moved(F0k, at, frm), ref, bnd)}
    del ref, a, bnd
    # ---- conv1 + pool planes: every stored class, the cells and the zeros
    q, pm_ref, pm_a, cell = D.check_conv1_planes(f0, pmq, sd, w, PR, PC)
    res.update({"planes_" + k: v for k, v in q.items() if k != "ratio"})
    PMk = D.dense_planes(pmq, PR2, PC2)
    use = pm_use[:, :, None].expand(9, 4, 64, PR2, PC2)
    res["planes_consumed_nan"] = int(torch.isnan(PMk[use]).sum())
    bnd = D.bound(pm_ref, pm_a, D.N_CONV1, True)
    ratios["conv1_pool"] = max(D.ratio(PMk, pm_ref, bnd, use), q["ratio"])    # consumed / every stored class
    if perturb:                                         # class 4 (mid / mid), plane 0, first row of tile row 1: a tile's
        row = T["c1p_OH"] // 2                          # OH pooled rows are OH / 2 rows of each parity plane
        assert bool(pm_use[4, 0, row, 1])
        res["perturbed"]["conv1_pool"] = D.ratio(moved(PMk, (4, 0, slice(24, 32), row, 1), (4, 0, slice(24, 32), row - 1, 1)),
                                                 pm_ref, bnd, use)
    del pm_ref, pm_a, bnd
    # ---- conv2: half-pooled maps from the kernel's own planes
    PMd = torch.nan_to_num(PMk.to(D.F64))
    yp_ref, yp_a = D.conv2_ref(PMd, D.h16(sd["conv2.weight"]), sd["conv2.bias"].to(D.F64), w)
    del PMd
    YPk = D.dense_planes(yq, PR2, PC2)
    use = yp_use[:, :, None].expand(9, 4, 64, PR2, PC2)
    res["half_pooled_nan"] = int(torch.isnan(YPk[use]).sum())
    bnd = D.bound(yp_ref, yp_a, D.N_CONV2, True)
    ratios["conv2"] = D.ratio(YPk, yp_ref, bnd, use)
    res["half_pooled_rel"] = rel(YPk[use], yp_ref[use])
    for Al in range(ncls if w == 20 else 0):            # and every row a map produces (rows y' < rho of class rho are not)
        r0a = [0, 2, 3][Al]
        sl = (slice(Al * 3, Al * 3 + ncls), slice(None), slice(None), slice(r0a, PR2 - 1), slice(0, PC2 - 1))
        res["half_pooled_rel"] = max(res["half_pooled_rel"], rel(torch.nan_to_num(YPk[sl]), yp_ref[sl]))
    if perturb:
        # first row of tile row 1, class 4 (mid / mid), plane 0, column 4 (pool2_cls reads the middle columns of the
        # mid / mid map from column 2J >= 2 on)
        row = T["c2s_TH"]
        assert bool(yp_use[4, 0, row, 4])
        res["perturbed"]["conv2"] = D.ratio(moved(YPk, (4, 0, slice(24, 32), row, 4), (4, 0, slice(24, 32), row - 1, 4)),
                                            yp_ref, bnd, use)
    del yp_ref, yp_a, bnd
    # ---- pool2 + classifier row maps from the kernel's own half-pooled maps
    cf, nn_ = D.GEOM[w]["conv_feat"], D.GEOM[w]["ncell"]
    Wconv = sd["classifier.weight"][:, :cf].reshape(K, 64, nn_, nn_)
    M_ref, M_a = D.pool2_ref(torch.nan_to_num(YPk.to(D.F64)), Wconv, w, K)
    Mk = D.dense_lmap(lmap, NC, PR2, PC2)[:, :ncell, :K]
    use = m_use[:, :, None].expand(4, ncell, K, PR2, PC2)
    res["row_maps_nan"] = int(torch.isnan(Mk[use]).sum())
    bnd = D.bound(M_ref, M_a, D.N_POOL2, False)
    ratios["pool2_cls"] = D.ratio(Mk, M_ref, bnd, use)
    res["row_maps_rel"] = rel(Mk[use], M_ref[use])
    for I in range(ncell if w == 20 else 0):            # and wherever every input of map I exists
        sl = (slice(None), I, slice(None), slice(2 * I, PR2 - 1), slice(0, PC2 - 2 * ncell))
        res["row_maps_rel"] = max(res["row_maps_rel"], rel(Mk[sl], M_ref[sl]))
    if perturb:
        row = T["p2c_TH"]                               # first row of tile row 1, row map 1, plane 0, classes 0-7
        assert bool(m_use[0, 1, row, 1])
        res["perturbed"]["pool2_cls"] = D.ratio(moved(Mk, (0, 1, slice(0, 8), row, 1), (0, 1, slice(0, 8), row - 1, 1)),
                                                M_ref, bnd, use)
    del M_ref, M_a, bnd, YPk
    # ---- spectral branch: quarter partials on the kernel's own fp16 input tiles
    check_spectral(res, ratios, x16, part, spectra, sd, n, B, K, perturb)
    return res, ratios, dict(F0=F0k, part=part, lmap=lmap, n=n, NC=NC, mt=mt)


def moved(t, at, frm):
    """A copy of a kernel output in which the entries t[at] (one 8-channel chunk at a tile seam) hold the values of
    t[frm] (the same chunk one row or position before the seam): a wrong-but-plausible tile-edge error."""
    t = t.clone()
    t[at] = t[frm]
    return t


def check_spectral(res, ratios, x16, part, spectra, sd, n, B, K, perturb=False):
    x, pad = D.dense_x16(x16, n, B)
    res["x16_pad_zero"] = bool((pad == 0).all())
    res["x16_equal"] = bool(torch.equal(x, spectra.half()))
    ref, bnd = D.spectral_ref(x, sd["feat_spe.weight"], sd["feat_spe.bias"], sd["classifier.weight"][:, -1024:])
    got = part[:, :n, :K]
    res["spectral_nan"] = int(torch.isnan(got).sum())
    ratios["spectral"] = D.ratio(got, ref, bnd)
    res["spectral_rel"] = rel(got.sum(0), ref.sum(0))
    if perturb:                                         # quarter 1, first pixel of the second 128-pixel tile, classes 0-7
        res["perturbed"]["spectral"] = D.ratio(moved(got, (1, 128, slice(0, 8)), (1, 127, slice(0, 8))), ref, bnd)


def assert_stages(res, ratios):
    assert res["f0_nan"] == 0 and res["f0_rel"] <= 1e-3, res
    assert res["planes_nan"] == 0 and res["planes_consumed_nan"] == 0 and res["planes_noncell_zero"], res
    assert res["planes_rel"] <= 1e-3 and res["planes_bit_equal"] >= 0.999, res
    assert res["half_pooled_nan"] == 0 and res["half_pooled_rel"] < 1e-3, res
    assert res["row_maps_nan"] == 0 and res["row_maps_rel"] < 1e-4, res
    assert res["x16_pad_zero"] and res["x16_equal"], res
    assert res["spectral_nan"] == 0 and res["spectral_rel"] <= 5e-4, res
    assert all(q <= 1.0 for q in ratios.values()), ratios


def weights(B, K, w, seed, dev):
    from cmlpl_b200 import ops
    torch.manual_seed(seed)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K, conv_feat=D.GEOM[w]["conv_feat"]).items()}
    return sd, ops.pack_basenet2(sd, B, K, w)


def head(lmap, part, C, R, B, K, w, packed, dev):
    from cmlpl_b200 import _lib
    lab = torch.empty(R * C, dtype=torch.uint8, device=dev)
    lg = torch.empty(R * C, K, dtype=torch.float32, device=dev)
    _lib.call("cmlpl_head_sum_lmap", part.data_ptr(), lmap.data_ptr(), C, R, B, K, w, packed.data_ptr(), lab.data_ptr(),
              lg.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return lab, lg


@pytest.mark.parametrize("R,C,B,K,seed", [(37, 45, 103, 9, 1), (24, 75, 144, 15, 2), (50, 61, 200, 16, 5)])
def test_dense_stages_match_torch_per_pixel_path_and_oracle(dev, R, C, B, K, seed):
    from cmlpl_b200 import _lib, ops
    w = 20
    rng = np.random.default_rng(seed)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
    torch.manual_seed(seed)
    sd_cpu = O.basenet2_init(B, K)
    sd = {k: v.to(dev) for k, v in sd_cpu.items()}
    packed = ops.pack_basenet2(sd, B, K, w)
    res, ratios, _ = stage_chain(cube, spectra, sd, packed, R, 0, 0, R, B, K, w)
    print(f"[{R}x{C}] {res}\n   worst error / bound {ratios}")
    assert_stages(res, ratios)
    labels, logits = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    _lib.call("cmlpl_set_scene_path_mode", 0)
    try:
        lab2, log2 = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    finally:
        _lib.call("cmlpl_set_scene_path_mode", 1)
    torch.cuda.synchronize()
    assert rel(logits, log2) < 1e-3 and bool((labels == lab2).all())
    lab_ref, log_ref = O.test_whole(sd_cpu, cube.cpu().numpy(), spectra.cpu().numpy(), w, return_logits=True)
    assert rel(logits.cpu(), torch.from_numpy(log_ref)) < 1e-3


def test_comparison_flags_a_perturbed_chunk_at_a_tile_seam(dev):
    """The bound comparisons are sensitive: in a copy of one kernel output at a time (F0, PM, YP, M, the spectral
    partials), one 8-channel chunk of one map at a tile seam takes the values of the row (position) before the seam,
    and the comparison flags it, while the kernel's own tensors meet their bounds."""
    R, C, B, K, w = 37, 45, 103, 9, 20
    rng = np.random.default_rng(3)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
    sd, packed = weights(B, K, w, 3, dev)
    res, ratios, _ = stage_chain(cube, spectra, sd, packed, R, 0, 0, R, B, K, w, perturb=True)
    print(ratios, res["perturbed"])
    assert_stages(res, ratios)
    assert all(q > 1.0 for q in res["perturbed"].values()), res["perturbed"]


@pytest.mark.parametrize("case", D.CASES, ids=[c[0] for c in D.CASES])
def test_many_tile_stages_match_float64(dev, case):
    """Every persistent dense kernel over many tiles per CTA (dense_refs.CASES), against the float64 references within
    their bounds on every consumed entry; the head's conv logits against the per-pixel float64 tower on the band's first
    and last rows and columns and 2000 random pixels at 1e-3 * max|ref|; the driver bit-identical to the stage chain."""
    from cmlpl_b200 import ops
    name, SR, C, r0, R, B, K, w = case
    t_start = time.time()
    per = D.tiles_per_cta(D.tile_constants(), R, C, w, R * C, torch.cuda.get_device_properties(dev).multi_processor_count)
    T = D.tile_constants()
    assert per["conv1_pool"] > T["c1p_NBUF"] and per["conv2"] >= 3 and per["pool2_cls"] >= 3 and per["spectral"] > 8, per
    s0, s1 = slab_of(SR, r0, R, w)
    gen = torch.Generator(device=dev)
    gen.manual_seed(SR + C + r0 + B)
    cube = torch.randn((s1 - s0, C, 60), device=dev, generator=gen)
    spectra = torch.randn((R * C, B), device=dev, generator=gen)
    sd, packed = weights(B, K, w, B + K, dev)
    res, ratios, k = stage_chain(cube, spectra, sd, packed, SR, s0, r0, R, B, K, w)
    assert_stages(res, ratios)
    # ---- the head on the conv partials alone against the per-pixel float64 tower
    zero = torch.zeros_like(k["part"])
    _, lg_conv = head(k["lmap"], zero, C, R, B, K, w, packed, dev)
    g = np.random.default_rng(r0 + R)
    pix = np.concatenate([np.arange(C), (R - 1) * C + np.arange(C), np.arange(R) * C, np.arange(R) * C + C - 1,
                          g.integers(0, R * C, 2000)])
    pr = torch.from_numpy(pix // C).to(dev)
    pc = torch.from_numpy(pix % C).to(dev)
    tower = D.tower_logits(k["F0"], pr, pc, sd, w)
    tower_rel = rel(lg_conv[torch.from_numpy(pix).to(dev)], tower)
    assert tower_rel < 1e-3, tower_rel
    # ---- the driver: same labels and logits, bit for bit
    lab, lg = head(k["lmap"], k["part"], C, R, B, K, w, packed, dev)
    lab_d, lg_d = ops.scene_infer(cube, spectra, packed, K, w, band_row0=r0, band_rows=R, scene_rows=SR, slab_row0=s0,
                                  want_logits=True)
    torch.cuda.synchronize()
    assert torch.equal(lab, lab_d) and torch.equal(lg, lg_d)
    print(f"[{name}] tiles per CTA {per}; worst error / bound {ratios}; tower rel {tower_rel:.2e}; "
          f"{time.time() - t_start:.1f} s")


@pytest.mark.parametrize("B,K", D.SPECTRAL_CASES)
def test_spectral_partials_many_tiles(dev, B, K):
    """spectral_logits_kernel alone on 60 001 pixels (> 8 tiles per CTA) at every input-ring depth (B = 103 / 150 /
    204 / 224: nA = 4 / 3 / 2 / 1) and both class widths: the fp16 tiles equal the rounded spectra with exact zero
    padding in NaN-prefilled scratch, and the quarter partials meet their bound."""
    from cmlpl_b200 import _lib
    n, w = D.SPECTRAL_N, 20
    T = D.tile_constants()
    assert D.tiles_per_cta(T, 1, 1, w, n, torch.cuda.get_device_properties(dev).multi_processor_count)["spectral"] > 8
    gen = torch.Generator(device=dev)
    gen.manual_seed(B * 100 + K)
    spectra = torch.randn((n, B), device=dev, generator=gen)
    sd, packed = weights(B, K, w, B + K, dev)
    NC = 16 if K <= 16 else 32
    mt, kc = (n + 127) // 128, ((B + 15) // 16) * 2
    x16 = torch.full((mt * kc * 1024,), float("nan"), dtype=torch.float16, device=dev)
    part = torch.full((4, mt * 128, NC), float("nan"), dtype=torch.float32, device=dev)
    _lib.call("cmlpl_spectral_logits_tc", spectra.data_ptr(), n, B, K, w, packed.data_ptr(), x16.data_ptr(), part.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    res, ratios = {}, {}
    check_spectral(res, ratios, x16, part, spectra, sd, n, B, K)
    print(f"[B={B} K={K} nA={D.spectral_nA(T, B, NC)}] {res} worst error / bound {ratios['spectral']:.3f}")
    assert res["x16_pad_zero"] and res["x16_equal"] and res["spectral_nan"] == 0, res
    assert res["spectral_rel"] <= 5e-4 and ratios["spectral"] <= 1.0, (res, ratios)


@pytest.mark.parametrize("B,sample,dc,layout", [(103, "u16", 20000.0, "bip"), (103, "i16", 0.0, "bil"),
                                              (103, "f32", 0.0, "bsq"), (270, "i16", 0.0, "bil")])
def test_raw_conv0_loaders_many_tiles(dev, B, sample, dc, layout):
    """The raw conv0 loaders (pixel-major, band-major BIL / BSQ, and the K-sliced ring of 64-band slices at 270 bands)
    on a PaviaU-size sensor-like scene, 12 tiles per CTA: the conv0 map within conv0_bar per position and channel, and
    1e-3 of its largest entry (dense_refs.raw_conv0_map_check, the comparison of test_gpu_sensor_scenes.py)."""
    R, C, K, w = 610, 340, 9, 20
    per = D.tiles_per_cta(D.tile_constants(), R, C, w, R * C, torch.cuda.get_device_properties(dev).multi_processor_count)
    assert per["conv0"] > 2, per                        # more tiles than TMEM accumulator slots
    t0 = time.time()
    q, e = D.raw_conv0_map_check(dev, R, C, B, K, w, 1.0, sample, dc, layout)
    print(f"[B={B} {sample} {layout}] conv0 tiles per CTA {per['conv0']}: error / max|F0| {e:.1e}, worst error / bar "
          f"{q:.3f}; {time.time() - t0:.1f} s")
    assert q <= 1.0
    assert e < 1e-3


def test_conv1_pool_planes_match_torch(dev):
    """conv1_pool_kernel (the 9 conv1 border-class variants pooled in its epilogue) on a 41 x 67 scene at w = 20 and
    w = 11, against the float64 planes on the kernel's own conv0 map.  w = 11 stores only the top / mid classes of
    both directions."""
    from cmlpl_b200 import _lib
    R, C, B, K = 41, 67, 103, 9
    st = torch.cuda.current_stream().cuda_stream
    for w in (20, 11):
        rng = np.random.default_rng(11)
        cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
        sd, packed = weights(B, K, w, 11, dev)
        PR, PC = R + w - 1, C + w - 1
        PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
        f0 = torch.empty(8 * PR * PC * 8, dtype=torch.float16, device=dev)
        pmq = torch.full((9, 4, 8, PR2, PC2, 8), float("nan"), dtype=torch.float16, device=dev)
        _lib.call("cmlpl_conv0_map_f16", cube.data_ptr(), R, C, 0, R, w, 0, R, packed.data_ptr(), f0.data_ptr(), st)
        _lib.call("cmlpl_conv1_pool_planes_f16", f0.data_ptr(), C, w, R, packed.data_ptr(), pmq.data_ptr(), st)
        torch.cuda.synchronize()
        q = D.check_conv1_planes(f0, pmq, sd, w, PR, PC)[0]
        print(f"[w = {w}] {q}")
        assert q["nan"] == 0 and q["noncell_zero"] and q["rel"] <= 1e-3 and q["bit_equal"] >= 0.999 and q["ratio"] <= 1.0, q
