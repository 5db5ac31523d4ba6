"""The float64 references and elementwise bounds of tests/dense_refs.py, without a GPU:
  * every bound holds for an fp16-operand / fp32-accumulate emulation of the stage (each contraction summed in fp32,
    one term at a time, in a shuffled order; fp16 outputs rounded once), at both windows and class widths;
  * every bound fails when one tap or one k-term of the stage is dropped;
  * the consumed-entry maps agree with a direct per-pixel walk of the index maps;
  * the many-tile cases of the stage test reach, at 148 SMs and with the tile constants read from the CUDA sources,
    more than 2 conv0 tiles and more than NBUF conv1_pool tiles per CTA, >= 3 conv2 / pool2_cls tiles, > 8 spectral tiles, every spectral ring
    depth 1-4 at both class widths, both windows, both class widths and a partial class quad."""
import numpy as np
import pytest
import torch

import dense_refs as D
from scene_harness import rel

SMS = 148


def emulated_contract(seed):
    """fp16 operands, fp32 accumulation one term at a time in a shuffled order of the contracted index"""
    g = torch.Generator().manual_seed(seed)

    def contract(eq, a, b):
        ins, out = eq.split("->")
        ia, ib = ins.split(",")
        k = next(c for c in ia if c in ib and c not in out)
        a32, b32 = a.float(), b.float()
        acc = None
        for j in torch.randperm(a.shape[ia.index(k)], generator=g).tolist():
            t = torch.einsum(eq.replace(k, ""), a32.select(ia.index(k), j), b32.select(ib.index(k), j))
            acc = t if acc is None else acc + t
        return acc.to(D.F64)
    return contract


def stage_inputs(w, seed):
    g = torch.Generator().manual_seed(seed)
    R, C = 5, 11                                     # the mirrored halo needs >= w/2 columns
    PR, PC = R + w - 1, C + w - 1
    rn = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc)
    sd = {"conv0.weight": rn(64, 60, 1, 1, sc=0.13), "conv0.bias": rn(64, sc=0.1),
          "conv1.weight": rn(64, 64, 3, 3, sc=0.04), "conv1.bias": rn(64, sc=0.04),
          "conv2.weight": rn(64, 64, 3, 3, sc=0.04), "conv2.bias": rn(64, sc=0.04)}
    return g, R, C, PR, PC, sd


def run_stages(w, seed, K=9, drop=None, up=None):
    """every stage reference, each from the float64 output of the one before rounded as the kernel stores it (or from
    the stage inputs of `up`, another run's result)"""
    g, R, C, PR, PC, sd = stage_inputs(w, seed)
    cube = torch.randn(PR + 3, C, 60, generator=g)
    W0 = sd["conv0.weight"].clone()
    W1, W2 = D.h16(sd["conv1.weight"]), D.h16(sd["conv2.weight"])
    Wc = torch.randn(K, 64, D.GEOM[w]["ncell"], D.GEOM[w]["ncell"], generator=g) * 0.05
    if drop == "conv0":
        W0[:, 7] = 0
    if drop == "conv1":
        W1[:, :, 0, 2] = 0
    if drop == "conv2":
        W2[:, :, 2, 1] = 0
    if drop == "pool2":
        Wc[:, 5] = 0
    f0, f0a = D.conv0_map(cube, W0, sd["conv0.bias"], PR + 3, 0, 1, R, w)
    F0 = f0.half().to(D.F64) if up is None else up["F0"]
    pm, pma, cell = D.conv1_ref(F0, W1, sd["conv1.bias"].to(D.F64))
    PM = pm.half().to(D.F64) if up is None else up["PM"]
    yp, ypa = D.conv2_ref(PM, W2, sd["conv2.bias"].to(D.F64), w)
    YP = yp.half().to(D.F64) if up is None else up["YP"]
    M, Ma = D.pool2_ref(YP, Wc, w, K)
    return dict(f0=(f0, f0a), pm=(pm, pma), yp=(yp, ypa), M=(M, Ma), F0=F0, PM=PM, YP=YP)


def spectral_inputs(B, K, seed, drop=False):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(300, B, generator=g).half()
    Wspe = torch.randn(1024, B, generator=g) / B ** 0.5
    b = torch.randn(1024, generator=g) * 0.1
    Wcs = torch.randn(K, 1024, generator=g) / 32
    if drop:
        Wspe[:, B // 2] = 0
    return x, Wspe, b, Wcs


STAGES = (("f0", D.N_CONV0, True), ("pm", D.N_CONV1, True), ("yp", D.N_CONV2, True), ("M", D.N_POOL2, False))


@pytest.mark.parametrize("w", [20, 11])
@pytest.mark.parametrize("seed", [1, 2])
def test_bounds_hold_for_fp32_accumulation_in_shuffled_order(w, seed, monkeypatch):
    ref = run_stages(w, seed)
    monkeypatch.setattr(D, "contract", emulated_contract(seed))
    emu = run_stages(w, seed, up=ref)
    for name, n, fp16 in STAGES:
        r, a = ref[name]
        got = emu[name][0].float()
        if fp16:
            got = got.half()
        q = D.ratio(got, r, D.bound(r, a, n, fp16))
        print(f"w={w} {name}: worst |emulated - ref| / bound {q:.3f}")
        assert q <= 1.0, (name, q)


@pytest.mark.parametrize("w", [20, 11])
def test_bounds_fail_when_a_tap_or_k_term_is_dropped(w):
    ref = run_stages(w, 3)
    for name, n, fp16 in STAGES:
        stage = {"f0": "conv0", "pm": "conv1", "yp": "conv2", "M": "pool2"}[name]
        bad = run_stages(w, 3, drop=stage, up=ref)[name][0]
        r, a = ref[name]
        got = bad.float().half() if fp16 else bad.float()
        assert D.ratio(got, r, D.bound(r, a, n, fp16)) > 1.0, name


@pytest.mark.parametrize("B,K", [(103, 13), (224, 24)])
def test_spectral_bound_holds_and_fails_on_a_dropped_band(B, K, monkeypatch):
    x, Wspe, b, Wcs = spectral_inputs(B, K, B)
    ref, bnd = D.spectral_ref(x.double(), Wspe, b, Wcs)
    with monkeypatch.context() as m:
        m.setattr(D, "contract", emulated_contract(B))
        emu, _ = D.spectral_ref(x.double(), Wspe, b, Wcs)
    q = D.ratio(emu.float(), ref, bnd)
    print(f"B={B}: worst |emulated - ref| / bound {q:.3f}")
    assert q <= 1.0
    bad, _ = D.spectral_ref(x.double(), *spectral_inputs(B, K, B, drop=True)[1:])
    assert D.ratio(bad.float(), ref, bnd) > 1.0


def test_tower_matches_the_border_class_decomposition():
    """The per-pixel float64 tower (no border classes) against the stage references composed through the head's
    gathers, on every pixel of a small band at both windows: the class tables and index maps agree."""
    for w in (20, 11):
        g, R, C, PR, PC, sd = stage_inputs(w, 7)
        K = 5
        n = D.GEOM[w]["ncell"]
        sd["classifier.weight"] = torch.randn(K, 64 * n * n + 1024, generator=g) * 0.05
        sd["classifier.bias"] = torch.randn(K, generator=g) * 0.1
        F0 = torch.randn(64, PR, PC, generator=g, dtype=D.F64)
        pm, _ = D.conv1_planes(F0, D.h16(sd["conv1.weight"]), sd["conv1.bias"].to(D.F64))
        yp = D.conv2_maps(pm, D.h16(sd["conv2.weight"]), sd["conv2.bias"].to(D.F64), w)
        M = D.pool2_maps(yp, sd["classifier.weight"][:, :64 * n * n].reshape(K, 64, n, n), w, K)
        rr, cc = torch.meshgrid(torch.arange(R), torch.arange(C), indexing="ij")
        rr, cc = rr.reshape(-1), cc.reshape(-1)
        pl = (rr & 1) * 2 + (cc & 1)
        got = sd["classifier.bias"].to(D.F64) + sum(M[pl, I, :, (rr >> 1) + 2 * I, cc >> 1] for I in range(n))
        ref = D.tower_logits(F0, rr, cc, sd, w)
        # pool2_cls's weights are fp16(Wc / d), the tower's fp16(Wc): equal but for the subnormal range
        assert rel(got, ref) < 1e-6, w


@pytest.mark.parametrize("w", [20, 11])
def test_consumed_maps_match_a_per_pixel_walk(w):
    R, C = 6, 9
    m, yp, pm = D.consumed(R, C, w)
    PR2, PC2 = (R + w) // 2, (C + w) // 2
    rep, npool, ncell = D.GEOM[w]["rep"], D.GEOM[w]["npool"], D.GEOM[w]["ncell"]
    m2, yp2, pm2 = np.zeros_like(m), np.zeros_like(yp), np.zeros_like(pm)
    for r in range(R):
        for c in range(C):
            p = (r & 1) * 2 + (c & 1)
            for I in range(ncell):
                for J in range(ncell):
                    y, x = (r >> 1) + 2 * I, c >> 1
                    m2[p, I, y, x] = True
                    Al, Be = D.al_of(I), D.al_of(J)
                    for u in ([0, 1] if Al == 1 else [0]):
                        for v in ([0, 1] if Be == 1 else [0]):
                            y1, x1 = y + u, x + 2 * J + v
                            if y1 >= PR2 or x1 >= PC2:
                                continue
                            yp2[Al * 3 + Be, p, y1, x1] = True
                            for u2 in ([0, 1] if Al != 1 else [0]):
                                for v2 in ([0, 1] if Be != 1 else [0]):
                                    y2, x2 = y1 + u2, x1 + v2
                                    if y2 >= PR2 or x2 >= PC2:
                                        continue
                                    i, j = rep[D.ycl(Al, u2)], rep[D.ycl(Be, v2)]
                                    pm2[D.cls1(w, i) * 3 + D.cls1(w, j), p, y2, x2] = True
                                    for dy in range(3):
                                        for dx in range(3):
                                            ii, jj, y3, x3 = i + dy - 1, j + dx - 1, y2 + dy - 1, x2 + dx - 1
                                            if 0 <= ii < npool and 0 <= jj < npool and 0 <= y3 < PR2 and 0 <= x3 < PC2:
                                                pm2[D.cls1(w, ii) * 3 + D.cls1(w, jj), p, y3, x3] = True
    assert (m == m2).all() and (yp == yp2).all() and (pm == pm2).all()


def test_cases_reach_many_tiles_every_ring_depth_and_class_width():
    T = D.tile_constants()
    assert T["c1p_NBUF"] >= 2 and T["p2c_NSLOT"] == {16: 8, 32: 6}, T
    seen = set()
    for name, SR, C, r0, R, B, K, w in D.CASES:
        t = D.tiles_per_cta(T, R, C, w, R * C, SMS)
        print(name, t)
        assert t["conv0"] > 2 and t["conv1_pool"] > T["c1p_NBUF"], (name, t)
        assert t["conv2"] >= 3 and t["pool2_cls"] >= 3, (name, t)
        assert t["spectral"] > 8, (name, t)
        NC = 16 if K <= 16 else 32
        seen |= {("w", w), ("nc", NC), ("nA", NC, D.spectral_nA(T, B, NC))}
        if K % 4:
            seen.add(("partial quad", NC))
        if r0 == 0:
            seen.add("top mirror")
        if r0 + R == SR and r0 > 0:
            seen.add("bottom mirror from a slab")
        if r0 > 0 and r0 + R < SR:
            seen.add("interior band")
    assert {("w", 20), ("w", 11), ("nc", 16), ("nc", 32), ("partial quad", 16), ("partial quad", 32), "top mirror",
            "bottom mirror from a slab", "interior band"} <= seen, seen
    for B, K in D.SPECTRAL_CASES:
        NC = 16 if K <= 16 else 32
        seen.add(("nA", NC, D.spectral_nA(T, B, NC)))
        assert D.tiles_per_cta(T, 1, 1, 20, D.SPECTRAL_N, SMS)["spectral"] > 8
    assert {("nA", nc, a) for nc in (16, 32) for a in (1, 2, 3, 4)} <= seen, seen
