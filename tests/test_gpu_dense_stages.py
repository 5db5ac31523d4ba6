"""The intermediate tensors of the dense scene path, stage by stage (tools/models.py:133-150 for all pixels at once):
the pooled conv1 parity planes  PM[A][B]  that conv1_pool_kernel writes, the half-pooled conv2 maps  YP[Al][Be]  that
conv2_scene_kernel writes (border halves of the 2x2 pool added in its epilogue), the row maps  M[I] = sum_J L[I][J](., x + 2J)
that pool2_cls_kernel writes and the quarter partials of spectral_logits_kernel, each against a plain torch fp32
evaluation of the same formula on the kernel's own fp16 inputs, then the whole path against the per-pixel kernels
(path mode 0) and the CPU oracle.  Bars: fp16-rounded maps 1e-3 * max|ref| (one rounding, 4.9e-4 relative), fp32 class
partial maps 1e-4, spectral partials 5e-4 * max|ref|, logits 1e-3 * max|ref| (north_star), labels identical on these
sizes."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O

pytestmark = pytest.mark.gpu
REP = [0, 1, 4, 8, 9]
cls = lambda i: 0 if i == 0 else (2 if i == 9 else 1)
S = ((1, 2), (0, 1, 2), (0, 1))     # conv1 taps dy (dx) a top / mid / bottom (left / mid / right) patch border keeps
AB = ((0, 1), (1, 1), (1, 2))       # conv1 border class of the two rows (columns) of a top / mid / bottom pooled cell


def rel(a, b):
    a = a.float(); b = b.float()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def conv1_pool_planes_ref(f0, W1, b1, PR, PC):
    """torch fp32 evaluation of what cmlpl_conv1_pool_planes_f16 stores, from the conv0 map f0 f16 [8][PR][PC][8]:
        G[a][b][p]       = relu(b1 + F0[p] + sum_{dy in S_a, dx in S_b} W1[dy,dx] . F0[p + (dy-1, dx-1)])
        PM[A][B][pr,pc]  = 1/4 sum_{u,v in {0,1}} G[a(A,u)][b(B,v)][pr+u, pc+v]          (pr < PR-1, pc < PC-1)
    scattered into the parity planes [9 = A*3+B][4 = (pr&1)*2+(pc&1)][8 chunks][PR2][PC2][8].  Returns the planes (0
    where no pooled cell exists) and the [4][PR2][PC2] mask of the entries that hold a pooled cell."""
    PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
    F0 = f0.view(8, PR, PC, 8).permute(0, 3, 1, 2).reshape(64, PR, PC).float()
    Fp = F.pad(F0, (1, 1, 1, 1))                                      # the kernel's tile loads zero-fill outside the map
    T = [[torch.einsum("oc,cyx->oyx", W1[:, :, dy, dx], Fp[:, dy:dy + PR, dx:dx + PC]) for dx in range(3)] for dy in range(3)]
    base = b1.view(64, 1, 1) + F0
    G = [[(base + sum(T[dy][dx] for dy in S[a] for dx in S[b])).clamp_min(0) for b in range(3)] for a in range(3)]
    planes = torch.zeros(9, 4, 8, PR2, PC2, 8, device=f0.device)
    cell = torch.zeros(4, PR2, PC2, dtype=torch.bool, device=f0.device)
    for A in range(3):
        for B in range(3):
            pm = sum(G[AB[A][u]][AB[B][v]][:, u:u + PR - 1, v:v + PC - 1] for u in range(2) for v in range(2)) / 4
            for p in range(2):
                for q in range(2):
                    sub = pm[:, p::2, q::2]
                    h, w_ = sub.shape[1], sub.shape[2]
                    planes[A * 3 + B, p * 2 + q, :, :h, :w_, :] = sub.reshape(8, 8, h, w_).permute(0, 2, 3, 1)
                    cell[p * 2 + q, :h, :w_] = True
    return planes, cell


def compare_conv1_pool_planes(pmq, ref, cell, ncls):
    """The kernel's planes (pre-filled with NaN) against conv1_pool_planes_ref on the ncls x ncls stored classes."""
    idx = [A * 3 + B for A in range(ncls) for B in range(ncls)]
    got, want = pmq[idx].float(), ref[idx]
    off = ~cell.view(1, 4, 1, cell.shape[1], cell.shape[2], 1).expand_as(got)
    d = (got - want).abs()
    _, e = torch.frexp(want.half().float())                              # |x| in [2^(e-1), 2^e)
    e = torch.where(want.half() == 0, torch.full_like(e, -24), e - 11).clamp_min(-24)
    ulp = torch.ldexp(torch.ones_like(want), e)                          # fp16 ulp of the reference (2^-24 below 2^-14)
    res = dict(planes_nan=int(torch.isnan(got).sum()), planes_noncell_zero=bool((got[off] == 0).all()),
               planes_rel=float(torch.nan_to_num(d, nan=float("inf")).max() / want.abs().max()),
               planes_bit_equal=float((pmq[idx] == want.half()).float().mean()),
               planes_ulps=float(torch.nan_to_num(d / ulp, nan=float("inf")).max()))
    print(f"   conv1_pool planes vs torch: nan={res['planes_nan']} non-cell entries zero={res['planes_noncell_zero']} "
          f"max|d|/max|ref| {res['planes_rel']:.2e}, bit-equal to the fp16 reference {res['planes_bit_equal']:.5f}, "
          f"largest difference {res['planes_ulps']:.2f} fp16 ulps")
    return res


def run(R, C, B, K, seed):
    from cmlpl_b200 import _lib, ops
    dev = torch.device("cuda", 0)
    w = 20
    res = {}
    rng = np.random.default_rng(seed)
    cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
    spectra = torch.from_numpy(rng.standard_normal((R * C, B)).astype(np.float32)).to(dev)
    torch.manual_seed(seed)
    sd = O.basenet2_init(B, K)
    sdd = {k: v.to(dev) for k, v in sd.items()}
    packed = ops.pack_basenet2(sdd, B, K, w)
    st = torch.cuda.current_stream().cuda_stream
    PR, PC = R + w - 1, C + w - 1
    PR2, PC2 = (R + w) // 2, (C + w) // 2
    n = R * C
    f0 = torch.empty(8 * PR * PC * 8, dtype=torch.float16, device=dev)
    pmq = torch.full((9, 4, 8, PR2, PC2, 8), float("nan"), dtype=torch.float16, device=dev)
    yq = torch.full((9, 4, 8, PR2, PC2, 8), float("nan"), dtype=torch.float16, device=dev)
    lmap = torch.full((4, 5, 4, PR2, PC2, 4), float("nan"), dtype=torch.float32, device=dev)
    _lib.call("cmlpl_conv0_map_f16", cube.data_ptr(), R, C, 0, R, w, 0, R, packed.data_ptr(), f0.data_ptr(), st)
    _lib.call("cmlpl_conv1_pool_planes_f16", f0.data_ptr(), C, w, R, packed.data_ptr(), pmq.data_ptr(), st)
    torch.cuda.synchronize()
    print(f"[{R}x{C}]")
    # ---- stage 1: conv1 + pool planes
    ref, cell = conv1_pool_planes_ref(f0, sdd["conv1.weight"].half().float(), sdd["conv1.bias"], PR, PC)
    res.update(compare_conv1_pool_planes(pmq, ref, cell, 3))
    # dense planes [9][4][64][PR2][PC2] f32 of the kernel's own pmq
    PMd = pmq.permute(0, 1, 2, 5, 3, 4).reshape(9, 4, 64, PR2, PC2).float()
    # ---- stage 2: conv2 variants
    _lib.call("cmlpl_conv2_scene_f16", pmq.data_ptr(), C, w, R, packed.data_ptr(), yq.data_ptr(), st)
    torch.cuda.synchronize()
    W2 = sdd["conv2.weight"].half().float()
    b2 = sdd["conv2.bias"]
    Yd = torch.zeros(25, 4, 64, PR2, PC2, device=dev)
    for rho in range(5):
        for kap in range(5):
            acc = PMd[cls(REP[rho]) * 3 + cls(REP[kap])].clone() + b2.view(1, 64, 1, 1)
            for dy in range(3):
                i2 = REP[rho] + dy - 1
                if i2 < 0 or i2 > 9: continue
                for dx in range(3):
                    j2 = REP[kap] + dx - 1
                    if j2 < 0 or j2 > 9: continue
                    src = PMd[cls(i2) * 3 + cls(j2)]                                 # [4, 64, PR2, PC2]
                    sh = F.pad(src, (1, 1, 1, 1))[:, :, dy:dy + PR2, dx:dx + PC2]    # value at (y+dy-1, x+dx-1)
                    acc += torch.einsum("oc,pcyx->poyx", W2[:, :, dy, dx], sh)
            Yd[rho * 5 + kap] = acc.clamp_min(0)
    # the kernel stores 9 half-pooled maps: border classes averaged with their partner (rho 0 with rho 1 one row down, ...)
    ycl = lambda c, u: u if c == 0 else (2 if c == 1 else 3 + u)
    yq_d = yq.permute(0, 1, 2, 5, 3, 4).reshape(9, 4, 64, PR2, PC2).float()
    worst, nan_y = 0.0, 0
    for Al in range(3):
        for Be in range(3):
            us = [0, 1] if Al != 1 else [0]
            vs = [0, 1] if Be != 1 else [0]
            ref = torch.zeros(4, 64, PR2, PC2, device=dev)
            for u in us:
                for v in vs:
                    src = Yd[ycl(Al, u) * 5 + ycl(Be, v)]
                    ref += F.pad(src, (0, 1, 0, 1))[:, :, u:u + PR2, v:v + PC2] / (len(us) * len(vs))
            r0 = [0, 2, 3][Al]                                   # rows y' < rho of row class rho are never produced
            got = yq_d[Al * 3 + Be][:, :, r0:PR2 - 1, :PC2 - 1]
            nan_y += int(torch.isnan(got).sum())
            e = rel(torch.nan_to_num(got), ref[:, :, r0:PR2 - 1, :PC2 - 1])
            worst = max(worst, e)
            if not e < 5e-3:
                print("      map Al=%d Be=%d rel %.2e" % (Al, Be, e))
    res["half_pooled_rel"], res["half_pooled_nan"] = worst, nan_y
    print(f"   half-pooled conv2 maps: worst rel err {worst:.2e} (fp16 output rounding ~5e-4) nan={nan_y}")
    # ---- stage 3: pooled classifier partial maps from the kernel's own yq
    _lib.call("cmlpl_pool2_cls_f16", yq.data_ptr(), C, w, R, B, K, packed.data_ptr(), lmap.data_ptr(), st)
    torch.cuda.synchronize()
    Wc = sdd["classifier.weight"][:, :1600].reshape(K, 64, 5, 5).half().float()
    yz = torch.nan_to_num(yq_d)
    # the kernel sums the pooled columns: M[I][y, x] = sum_J L[I][J][y, x + 2J]
    worst = 0.0
    for I in range(5):
        Al = 0 if I == 0 else (2 if I == 4 else 1)
        ref = torch.zeros(4, K, PR2, PC2, device=dev)
        for J in range(5):
            Be = 0 if J == 0 else (2 if J == 4 else 1)
            us = [0, 1] if Al == 1 else [0]
            vs = [0, 1] if Be == 1 else [0]
            for u in us:
                for v in vs:
                    sh = F.pad(yz[Al * 3 + Be], (0, 2 * J + 1, 0, 1))[:, :, u:u + PR2, 2 * J + v:2 * J + v + PC2]
                    ref += torch.einsum("kc,pcyx->pkyx", Wc[:, :, I, J], sh) / (len(us) * len(vs))
        got = lmap[:, I].permute(0, 1, 4, 2, 3).reshape(4, 16, PR2, PC2)[:, :K]
        # map I is read at y' = r' + 2I >= 2I, x' = c' <= PC2 - 11 only; compare where every input exists
        e = rel(got[:, :, 2 * I:PR2 - 1, :PC2 - 10], ref[:, :, 2 * I:PR2 - 1, :PC2 - 10])
        worst = max(worst, e)
    res["row_maps_rel"] = worst
    print(f"   class-partial row maps: worst rel err {worst:.2e}")
    # ---- spectral branch: quarter partials Wc_spe . relu(Wspe . x + b) on the kernel's own fp16 input tiles; the kernel
    # packs the hidden tile as fp16 before the classifier MMA
    mt, kc = (n + 127) // 128, ((B + 15) // 16) * 2
    x16 = torch.empty(mt * kc * 1024, dtype=torch.float16, device=dev)
    part = torch.full((4, mt * 128, 16), float("nan"), dtype=torch.float32, device=dev)
    _lib.call("cmlpl_spectral_logits_tc", spectra.data_ptr(), n, B, K, w, packed.data_ptr(), x16.data_ptr(), part.data_ptr(), st)
    torch.cuda.synchronize()
    x = x16.view(mt, kc, 128, 8).permute(0, 2, 1, 3).reshape(mt * 128, kc * 8)[:n, :B].float()
    hidden = (x @ sdd["feat_spe.weight"].half().float().t() + sdd["feat_spe.bias"]).clamp_min(0).half().float()
    ref = hidden @ sdd["classifier.weight"][:, 1600:].half().float().t()
    res["spectral_rel"] = rel(part.sum(0)[:n, :K], ref)
    print(f"   spectral quarter partials vs torch: rel {res['spectral_rel']:.2e}")
    # ---- stage 4: whole path vs per-pixel path (path mode 0) vs oracle
    labels, logits = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    _lib.call("cmlpl_set_scene_path_mode", 0)
    try:
        lab2, log2 = ops.scene_infer(cube, spectra, packed, K, w, want_logits=True)
    finally:
        _lib.call("cmlpl_set_scene_path_mode", 1)
    torch.cuda.synchronize()
    res["dense_vs_pixel_rel"], res["labels_equal"] = rel(logits, log2), float((labels == lab2).float().mean())
    print(f"   logits dense vs per-pixel path: rel {res['dense_vs_pixel_rel']:.2e}, labels equal {res['labels_equal']:.5f}")
    if n <= 4000:
        lab_ref, log_ref = O.test_whole(sd, cube.cpu().numpy(), spectra.cpu().numpy(), w, return_logits=True)
        res["dense_vs_oracle_rel"] = rel(logits.cpu(), torch.from_numpy(log_ref))
        print(f"   logits dense vs oracle: rel {res['dense_vs_oracle_rel']:.2e}; per-pixel vs oracle {rel(log2.cpu(), torch.from_numpy(log_ref)):.2e}")
    return res


def assert_conv1_pool_planes(res):
    assert res["planes_nan"] == 0 and res["planes_noncell_zero"], res
    assert res["planes_rel"] <= 1e-3 and res["planes_bit_equal"] >= 0.999, res


@pytest.mark.parametrize("R,C,B,K,seed", [(37, 45, 103, 9, 1), (24, 75, 144, 15, 2), (50, 61, 200, 16, 5)])
def test_dense_stages_match_torch_per_pixel_path_and_oracle(dev, R, C, B, K, seed):
    res = run(R, C, B, K, seed)
    assert_conv1_pool_planes(res)
    assert res["half_pooled_nan"] == 0 and res["half_pooled_rel"] < 1e-3, res
    assert res["row_maps_rel"] < 1e-4, res
    assert res["spectral_rel"] <= 5e-4, res
    assert res["dense_vs_pixel_rel"] < 1e-3 and res["labels_equal"] == 1.0, res
    assert res["dense_vs_oracle_rel"] < 1e-3, res


def test_conv1_pool_planes_match_torch(dev):
    """conv1_pool_kernel (the 9 conv1 border-class variants pooled in its epilogue) on a 41 x 67 scene at w = 20 and
    w = 11, against conv1_pool_planes_ref on the kernel's own conv0 map.  w = 11 stores only the top / mid classes of
    both directions."""
    from cmlpl_b200 import _lib, ops
    R, C, B, K = 41, 67, 103, 9
    st = torch.cuda.current_stream().cuda_stream
    for w in (20, 11):
        rng = np.random.default_rng(11)
        cube = torch.from_numpy(rng.standard_normal((R, C, 60)).astype(np.float32)).to(dev)
        torch.manual_seed(11)
        sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K, conv_feat=1600 if w == 20 else 256).items()}
        packed = ops.pack_basenet2(sd, B, K, w)
        PR, PC = R + w - 1, C + w - 1
        PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
        f0 = torch.empty(8 * PR * PC * 8, dtype=torch.float16, device=dev)
        pmq = torch.full((9, 4, 8, PR2, PC2, 8), float("nan"), dtype=torch.float16, device=dev)
        _lib.call("cmlpl_conv0_map_f16", cube.data_ptr(), R, C, 0, R, w, 0, R, packed.data_ptr(), f0.data_ptr(), st)
        _lib.call("cmlpl_conv1_pool_planes_f16", f0.data_ptr(), C, w, R, packed.data_ptr(), pmq.data_ptr(), st)
        torch.cuda.synchronize()
        print(f"[w = {w}]")
        ref, cell = conv1_pool_planes_ref(f0, sd["conv1.weight"].half().float(), sd["conv1.bias"], PR, PC)
        assert_conv1_pool_planes(compare_conv1_pool_planes(pmq, ref, cell, 3 if w == 20 else 2))
