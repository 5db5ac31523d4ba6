"""float64 references of the dense scene path, stage by stage, and the elementwise error bounds the stage tests hold
the kernels to.  Imported as a plain module (pytest puts tests/ on sys.path); it holds no tests.

Every reference starts from the kernel's own fp16 inputs and the fp16-rounded weights, on either window (w = 20, 11)
and class width (NC = 16, 32), and returns the value and the same formula on |weights| and |inputs| (sum|terms|), from
which `bound` forms the elementwise bar:
    fp16 outputs (F0, PM, YP)   |got - ref| <= 1/2 ulp16(|ref| + acc) + acc,  acc = n 2^-24 sum|terms|
    fp32 outputs (M, partials)  |got - ref| <= acc
for n the terms of the output's fp32 sum in any order.  The spectral partials also carry the fp16 rounding of each
hidden feature through |Wc|.  Layouts (DESIGN 3): the kernels' chunked tensors are turned dense by the `dense_*`
helpers, the references work on dense [.., 64, rows, cols] maps.

The module also holds the many-tile case list of tests/test_gpu_dense_stages.py and the tile arithmetic of the
persistent kernels, with their tile constants parsed from the CUDA sources, so that a retiled kernel cannot leave the
cases behind unnoticed (tests/test_dense_refs_cpu.py)."""
import os
import re

import numpy as np
import torch
import torch.nn.functional as F

from scene_harness import rel

U = 2.0 ** -24                  # unit roundoff of fp32
F64 = torch.float64

# per window: conv2 row representatives (DESIGN 4.1: rho in {i=0, 1, 2..7, 8, 9}; w = 11: {0, 1, 2..3}, 4.5), pooled
# conv1 rows, pooled cells per side (row maps), classifier conv columns
GEOM = {20: dict(rep=[0, 1, 4, 8, 9], npool=10, ncell=5, conv_feat=1600),
        11: dict(rep=[0, 1, 2], npool=5, ncell=2, conv_feat=256)}
S = ((1, 2), (0, 1, 2), (0, 1))     # conv1 taps dy (dx) a top / mid / bottom (left / mid / right) patch border keeps
AB = ((0, 1), (1, 1), (1, 2))       # conv1 border class of the two rows (columns) of a top / mid / bottom pooled cell

# terms of one output's fp32 sum (products, bias, residual, pool adds and scales)
N_CONV0 = 60 + 2
N_CONV1 = 9 * 64 + 2 + 4 + 1
N_CONV2 = 9 * 64 + 2 + 2 + 1
N_POOL2 = 5 * 4 * 64 + 1


def cls1(w, i):
    """border class of pooled conv1 row (column) i of the window: top 0, mid 1, bottom 2 (w = 11: no bottom)"""
    return 0 if i == 0 else (2 if w == 20 and i == GEOM[w]["npool"] - 1 else 1)


def nclass(w):
    """row (column) classes of the pooled conv1 planes and of the half-pooled conv2 maps"""
    return 3 if w == 20 else 2


def ycl(Al, u):
    """conv2 representative pooled into half-pooled class Al (with its partner u rows down)"""
    return u if Al == 0 else (2 if Al == 1 else 3 + u)


def al_of(I):
    """half-pooled class of pooled cell row (column) I"""
    return 0 if I == 0 else (2 if I == 4 else 1)


# ---------------------------------------------------------------------------------------------- bounds
def contract(eq, a, b):
    """torch.einsum of two operands; tests/test_dense_refs_cpu.py replaces it with an fp32 sum in shuffled order"""
    return torch.einsum(eq, a, b)


def half_ulp16(x):
    """1/2 fp16 ulp of |x| (float64; 2^-25 in the subnormal range)"""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -14))
    return torch.ldexp(torch.ones_like(x), e - 12)


def bound(ref, terms, n, fp16):
    acc = n * U * terms
    return half_ulp16(ref.abs() + acc) + acc if fp16 else acc


def ratio(got, ref, bnd, mask=None):
    """max |got - ref| / bound over the mask: inf where got is NaN, 0 where got equals ref (a zero bound included)"""
    e = torch.nan_to_num((got.to(F64) - ref).abs(), nan=float("inf"))
    d = torch.where(e == 0, torch.zeros_like(e), e / bnd)
    if mask is not None:
        d = d[mask]
    return float(d.max()) if d.numel() else 0.0


# ---------------------------------------------------------------------------------------------- layouts
def dense_f0(f0, PR, PC):
    """conv0 map f16 [8 chunks][PR][PC][8] -> float64 [64][PR][PC]"""
    return f0.view(8, PR, PC, 8).permute(0, 3, 1, 2).reshape(64, PR, PC).to(F64)


def dense_planes(q, PR2, PC2):
    """PM / YP f16 [9][4][8][PR2][PC2][8] -> [9][4][64][PR2][PC2] (dtype kept)"""
    return q.view(9, 4, 8, PR2, PC2, 8).permute(0, 1, 2, 5, 3, 4).reshape(9, 4, 64, PR2, PC2)


def dense_lmap(lmap, NC, PR2, PC2):
    """M f32 [4][5][NC/4][PR2][PC2][4] -> [4][5][NC][PR2][PC2] (dtype kept)"""
    return lmap.view(4, 5, NC // 4, PR2, PC2, 4).permute(0, 1, 2, 5, 3, 4).reshape(4, 5, NC, PR2, PC2)


def dense_x16(x16, n, B):
    """spectral tiles f16 [mt][KC][128][8] -> [n][B] (dtype kept) and the padding: k >= B of every row, rows >= n"""
    mt, kc = (n + 127) // 128, ((B + 15) // 16) * 2
    x = x16.view(mt, kc, 128, 8).permute(0, 2, 1, 3).reshape(mt * 128, kc * 8)
    return x[:n, :B], torch.cat([x[:, B:].reshape(-1), x[n:, :B].reshape(-1)])


def h16(t):
    """fp16-rounded weights as float64"""
    return t.detach().half().to(F64)


# ---------------------------------------------------------------------------------------------- references
def mirror(o, n):
    """single reflection (hyper_tools.py:35-55), as common.cuh mirror_index"""
    return np.where(o < 0, -o - 1, np.where(o >= n, 2 * n - 1 - o, o))


def conv0_map(cube, W0, b0, scene_rows, slab_row0, band_row0, band_rows, w):
    """F0 = W0 . x + b0 on the mirror-padded band of the PCA cube slab cube [slab_rows, cols, 60] (rows slab_row0.. of a
    scene_rows-row scene); the mirror applies at true scene edges only.  -> (F0, sum|terms|) float64 [64][PR][PC]"""
    cols = cube.shape[1]
    lo = -(w // 2)
    PR, PC = band_rows + w - 1, cols + w - 1
    rows = torch.from_numpy(mirror(band_row0 + np.arange(PR) + lo, scene_rows) - slab_row0).to(cube.device)
    cc = torch.from_numpy(mirror(np.arange(PC) + lo, cols)).to(cube.device)
    x = cube.half().to(F64)[rows][:, cc]                                  # [PR][PC][60], the kernel's fp16 operand
    W = h16(W0.reshape(64, 60))
    b = b0.detach().to(F64).view(64, 1, 1)
    f = contract("ok,pqk->opq", W, x) + b
    a = contract("ok,pqk->opq", W.abs(), x.abs()) + b.abs()
    return f, a


def conv1_planes(F0, W1, b1, relu=True):
    """The pooled border-class planes of conv1_pool_kernel from the conv0 map F0 float64 [64][PR][PC]:
        G[a][b][p]       = relu(b1 + F0[p] + sum_{dy in S_a, dx in S_b} W1[dy,dx] . F0[p + (dy-1, dx-1)])
        PM[A][B][pr,pc]  = 1/4 sum_{u,v in {0,1}} G[a(A,u)][b(B,v)][pr+u, pc+v]          (pr < PR-1, pc < PC-1)
    on the parity planes [9 = A*3+B][4 = (pr&1)*2+(pc&1)][64][PR2][PC2] (0 where no pooled cell exists), and the mask
    [4][PR2][PC2] of the entries that hold a pooled cell.  W1 (fp16-rounded) [64][64][3][3]."""
    _, PR, PC = F0.shape
    PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
    Fp = F.pad(F0, (1, 1, 1, 1))                                      # the kernel's tile loads zero-fill outside the map
    T = [[contract("oc,cyx->oyx", W1[:, :, dy, dx], Fp[:, dy:dy + PR, dx:dx + PC]) for dx in range(3)] for dy in range(3)]
    base = b1.view(64, 1, 1) + F0
    G = [[base + sum(T[dy][dx] for dy in S[a] for dx in S[b]) for b in range(3)] for a in range(3)]
    if relu:
        G = [[g.clamp_min(0) for g in row] for row in G]
    del T
    planes = torch.zeros(9, 4, 64, PR2, PC2, dtype=F64, device=F0.device)
    cell = torch.zeros(4, PR2, PC2, dtype=torch.bool, device=F0.device)
    for A in range(3):
        for B in range(3):
            pm = sum(G[AB[A][u]][AB[B][v]][:, u:u + PR - 1, v:v + PC - 1] for u in range(2) for v in range(2)) / 4
            for p in range(2):
                for q in range(2):
                    sub = pm[:, p::2, q::2]
                    planes[A * 3 + B, p * 2 + q, :, :sub.shape[1], :sub.shape[2]] = sub
                    cell[p * 2 + q, :sub.shape[1], :sub.shape[2]] = True
    return planes, cell


def conv1_ref(F0, W1, b1):
    """(PM, sum|terms|, cell) of conv1_planes"""
    pm, cell = conv1_planes(F0, W1, b1)
    pa, _ = conv1_planes(F0.abs(), W1.abs(), b1.abs(), relu=False)
    return pm, pa, cell


def conv2_maps(PM, W2, b2, w, relu=True):
    """The half-pooled conv2 maps YP[Al*3+Be] [9][4][64][PR2][PC2] of conv2_scene_kernel from the planes PM (float64
    [9][4][64][PR2][PC2], the kernel's own): the conv2 variant of representative rows rho / columns kap
        Y[rho][kap] = relu(b2 + PM[cls(rep rho)][cls(rep kap)] + sum_{taps inside the pooled map} W2 . PM[cls][cls](shifted))
    with the border halves of the 2x2 pool averaged (rho 0 with rho 1 one row down, rho 3 with rho 4; same for kap).
    Maps of classes the window does not have (w = 11: Al, Be = 2) stay 0."""
    rep, npool = GEOM[w]["rep"], GEOM[w]["npool"]
    nr = len(rep)
    _, _, _, PR2, PC2 = PM.shape
    Pp = F.pad(PM, (1, 1, 1, 1))
    sh = {}                                                            # W2[dy,dx] . PM[class] shifted by (dy-1, dx-1)

    def tap(c, dy, dx):
        if (c, dy, dx) not in sh:
            sh[(c, dy, dx)] = contract("oc,pcyx->poyx", W2[:, :, dy, dx], Pp[c, :, :, dy:dy + PR2, dx:dx + PC2])
        return sh[(c, dy, dx)]

    Y = {}
    for rho in range(nr):
        for kap in range(nr):
            i, j = rep[rho], rep[kap]
            acc = PM[cls1(w, i) * 3 + cls1(w, j)] + b2.view(1, 64, 1, 1)
            for dy in range(3):
                if not 0 <= i + dy - 1 < npool:
                    continue
                for dx in range(3):
                    if not 0 <= j + dx - 1 < npool:
                        continue
                    acc = acc + tap(cls1(w, i + dy - 1) * 3 + cls1(w, j + dx - 1), dy, dx)
            Y[(rho, kap)] = acc.clamp_min(0) if relu else acc
    sh.clear()
    yp = torch.zeros(9, 4, 64, PR2, PC2, dtype=F64, device=PM.device)
    for Al in range(nclass(w)):
        for Be in range(nclass(w)):
            us = [0, 1] if Al != 1 else [0]
            vs = [0, 1] if Be != 1 else [0]
            for u in us:
                for v in vs:
                    yp[Al * 3 + Be] += F.pad(Y[(ycl(Al, u), ycl(Be, v))], (0, 1, 0, 1))[:, :, u:u + PR2, v:v + PC2] / (len(us) * len(vs))
    return yp


def conv2_ref(PM, W2, b2, w):
    """(YP, sum|terms|)"""
    return conv2_maps(PM, W2, b2, w), conv2_maps(PM.abs(), W2.abs(), b2.abs(), w, relu=False)


def pool2_weight(Wc, I, J, d):
    """pool2_cls_kernel's block weight of cell (I, J) for a map averaged over d variants: fp16(Wc / d) (pack.cu)"""
    return (Wc[:, :, I, J].detach().float() / d).half().to(F64)


def pool2_maps(YP, Wconv, w, K, absw=False):
    """The row maps M[I][p][k][y, x] = sum_J L[I][J][p][k][y, x + 2J] of pool2_cls_kernel [4][ncell][K][PR2][PC2] from
    the half-pooled maps YP (float64 [9][4][64][PR2][PC2], the kernel's own), with the remaining 2x2 pool of the middle
    classes; Wconv = the classifier's conv columns [K][64][n][n] (fp32)."""
    ncell = GEOM[w]["ncell"]
    _, _, _, PR2, PC2 = YP.shape
    M = torch.zeros(4, ncell, K, PR2, PC2, dtype=F64, device=YP.device)
    for I in range(ncell):
        Al = al_of(I)
        us = [0, 1] if Al == 1 else [0]
        for J in range(ncell):
            Be = al_of(J)
            vs = [0, 1] if Be == 1 else [0]
            Wt = pool2_weight(Wconv, I, J, len(us) * len(vs))
            if absw:
                Wt = Wt.abs()
            src = F.pad(YP[Al * 3 + Be], (0, 2 * J + 1, 0, 1))
            for u in us:
                for v in vs:
                    M[:, I] += contract("kc,pcyx->pkyx", Wt, src[:, :, u:u + PR2, 2 * J + v:2 * J + v + PC2])
    return M


def pool2_ref(YP, Wconv, w, K):
    """(M, sum|terms|)"""
    return pool2_maps(YP, Wconv, w, K), pool2_maps(YP.abs(), Wconv, w, K, absw=True)


def spectral_ref(x, Wspe, bspe, Wcs):
    """Quarter partials of spectral_logits_kernel from its own fp16 input rows x [n][B]: part[q] = Wc_spe[:, q] .
    fp16(relu(Wspe[q] . x + b[q])) for the hidden quarter q = features 256 q .. 256 q + 255.  -> (part float64
    [4][n][K], bound [4][n][K]): the fp32 sums of both GEMMs and one fp16 rounding of each hidden feature through |Wc|."""
    x = x.to(F64)
    B = x.shape[1]
    W1, W2, b = h16(Wspe), h16(Wcs), bspe.detach().to(F64)
    parts, bnds = [], []
    for q in range(4):
        s = slice(256 * q, 256 * q + 256)
        h = contract("nk,ok->no", x, W1[s]) + b[s]
        acc1 = (B + 2) * U * (x.abs() @ W1[s].abs().t() + b[s].abs())
        hr = h.clamp_min(0).half().to(F64)
        eh = 2 * half_ulp16(h.clamp_min(0) + acc1) + acc1                # kernel's fp16(h32) vs fp16(h64)
        del h
        parts.append(contract("nj,kj->nk", hr, W2[:, s]))
        bnds.append(256 * U * (hr.abs() @ W2[:, s].abs().t()) + eh @ W2[:, s].abs().t())
    return torch.stack(parts), torch.stack(bnds)


def tower_logits(F0, pix_r, pix_c, sd, w, chunk=512):
    """Per-pixel float64 conv tower (tools/models.py:133-150 without the spectral branch) on the w x w windows of the
    kernel's conv0 map F0 float64 [64][PR][PC] at band pixels (pix_r, pix_c): conv1 + residual, ReLU, floor 2x2 pool,
    conv2 + residual, ReLU, pool, the classifier's conv columns + bias.  No border classes: it checks the class tables.
    -> [npix][K] float64"""
    W1, W2 = h16(sd["conv1.weight"]), h16(sd["conv2.weight"])
    b1, b2 = sd["conv1.bias"].to(F64), sd["conv2.bias"].to(F64)
    cf = GEOM[w]["conv_feat"]
    Wc, bc = h16(sd["classifier.weight"][:, :cf]), sd["classifier.bias"].to(F64)
    d = torch.arange(w, device=F0.device)
    out = []
    for s in range(0, len(pix_r), chunk):
        r, c = pix_r[s:s + chunk], pix_c[s:s + chunk]
        X = F0[:, (r[:, None] + d)[:, :, None], (c[:, None] + d)[:, None, :]].permute(1, 0, 2, 3)   # [n][64][w][w]
        x = F.relu(F.conv2d(X, W1, b1, padding=1) + X)
        x = F.avg_pool2d(x, 2, 2)
        x = F.relu(F.conv2d(x, W2, b2, padding=1) + x)
        x = F.avg_pool2d(x, 2, 2)
        out.append(x.reshape(x.shape[0], -1) @ Wc.t() + bc)
    return torch.cat(out)


def check_conv1_planes(f0, pmq, sd, w, PR, PC):
    """conv1_pool_kernel's planes pmq (NaN-prefilled) against conv1_ref on its own conv0 map f0, on the classes the
    window stores (w = 11: top / mid of both directions): NaN count, entries without a pooled cell exactly 0, max
    relative error, share bit-equal to the fp16-rounded reference, worst error / bound.  Also returns the reference,
    its sum|terms| and the cell mask on all 9 classes."""
    PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
    ref, a, cell = conv1_ref(dense_f0(f0, PR, PC), h16(sd["conv1.weight"]), sd["conv1.bias"].to(F64))
    idx = [A * 3 + B for A in range(nclass(w)) for B in range(nclass(w))]
    got, want = dense_planes(pmq, PR2, PC2)[idx], ref[idx]
    off = ~cell.view(1, 4, 1, PR2, PC2).expand_as(got)
    q = dict(nan=int(torch.isnan(got).sum()), noncell_zero=bool((got[off] == 0).all()), rel=rel(got, want),
             bit_equal=float((got == want.half()).float().mean()), ratio=ratio(got, want, bound(want, a[idx], N_CONV1, True)))
    return q, ref, a, cell


def raw_conv0_map_check(dev, R, C, B, K, w, nd, sample, dc, layout):
    """The conv0 map of cmlpl_scene_infer_raw (workspace offset 0, chunk-planar fp16 [8][R+w-1][C+w-1][8]) on an
    oracle.sensor_scene cube in `layout`, against the folded 1x1 conv in float64 on the mirror-padded scene, per
    position and channel within test_sensor_scenes_cpu.conv0_bar (half an fp16 ulp + the hi / lo cancellation term).
    -> (worst error / bar, error / max|F0|)"""
    from cmlpl_b200 import ops, preprocess
    from cmlpl_b200.tools.models import BaseNet2
    from oracle import cmlpl_oracle as O
    from scene_harness import as_layout
    from test_sensor_scenes_cpu import conv0_bar
    cube, _ = O.sensor_scene(R, C, B, K, nd, seed=B + K, sample=sample, dc=dc)
    pp = preprocess.fit(as_layout(cube, "bip", dev), 60)
    torch.manual_seed(B)
    net = BaseNet2(B, 0, K, w=w).to(dev).eval()
    folded = pp.folded_conv0(net.conv0.weight, net.conv0.bias, dev)
    W0 = net.conv0.weight.detach().double().cpu().numpy().reshape(64, 60)
    wf64 = (pp.U / pp.pca_sigma[None]) @ W0.T
    bf64 = net.conv0.bias.detach().double().cpu().numpy() - W0 @ (pp.pca_mu / pp.pca_sigma)
    ws = ops.scene_workspace(R, C, B, K, w, dev)
    ws.fill_(255)                                                        # NaN fp16 everywhere
    ops.scene_infer_raw(as_layout(cube, layout, dev), folded, net.packed_weights(w), K, C, w, workspace=ws,
                        interleave=layout)
    torch.cuda.synchronize()
    PR, PC = R + w - 1, C + w - 1
    got = ws[:8 * PR * PC * 16].view(torch.float16).view(8, PR, PC, 8).permute(1, 2, 0, 3).reshape(-1, 64).double().cpu().numpy()
    rr = mirror(np.arange(PR) - w // 2, R)
    cc = mirror(np.arange(PC) - w // 2, C)
    Xp = cube[rr][:, cc].reshape(-1, B).astype(np.float64)
    ref = (Xp - pp.mu) @ wf64 + bf64
    bar, _ = conv0_bar(Xp, folded["mu"].cpu().numpy(), pp.mu, folded["inv_sigma"].cpu().numpy(),
                       folded["wf"].cpu().numpy(), wf64, bf64, ref)
    err = np.nan_to_num(np.abs(got - ref), nan=np.inf)
    return float((err / bar).max()), float(err.max() / np.abs(ref).max())


# ---------------------------------------------------------------------------------------------- consumed entries
def shift_or(dst, src, dy, dx):
    """dst[..., y+dy, x+dx] |= src[..., y, x] where the target lies inside dst"""
    H, W = src.shape[-2:]
    if dy >= H or dx >= W:
        return
    dst[..., dy:, dx:] |= src[..., :H - dy, :W - dx]


def shift_or_back(dst, src, dy, dx):
    """dst[..., y+dy, x+dx] |= src[..., y, x] for dy, dx in -1..1 (conv2 taps), inside dst"""
    H, W = src.shape[-2:]
    ys, yd = (slice(0, H - dy), slice(dy, H)) if dy >= 0 else (slice(-dy, H), slice(0, H + dy))
    xs, xd = (slice(0, W - dx), slice(dx, W)) if dx >= 0 else (slice(-dx, W), slice(0, W + dx))
    dst[..., yd, xd] |= src[..., ys, xs]


def consumed(R, C, w):
    """Entries of M [4][ncell][PR2][PC2], YP [9][4][PR2][PC2] and PM [9][4][PR2][PC2] that the head of an R x C band
    depends on, composing the index maps of the consumers:
        head_sum reads   M[(r&1)*2+(c&1)][I][(r>>1)+2I][c>>1]
        pool2_cls reads  YP[Al(I)][Be(J)][y+u][x+2J+v]
        conv2 reads      PM at its taps (and the residual) of the representatives pooled into YP."""
    PR2, PC2 = (R + w) // 2, (C + w) // 2
    ncell, rep, npool = GEOM[w]["ncell"], GEOM[w]["rep"], GEOM[w]["npool"]
    m = np.zeros((4, ncell, PR2, PC2), bool)
    for p in range(4):
        nr, nc = (R - (p >> 1) + 1) // 2, (C - (p & 1) + 1) // 2
        for I in range(ncell):
            m[p, I, 2 * I:2 * I + nr, :nc] = True
    yp = np.zeros((9, 4, PR2, PC2), bool)
    for I in range(ncell):
        Al = al_of(I)
        for J in range(ncell):
            Be = al_of(J)
            for u in ([0, 1] if Al == 1 else [0]):
                for v in ([0, 1] if Be == 1 else [0]):
                    shift_or(yp[Al * 3 + Be], m[:, I], u, 2 * J + v)
    yd = {}
    for Al in range(nclass(w)):
        for Be in range(nclass(w)):
            for u in ([0, 1] if Al != 1 else [0]):
                for v in ([0, 1] if Be != 1 else [0]):
                    k = (ycl(Al, u), ycl(Be, v))
                    yd.setdefault(k, np.zeros((4, PR2, PC2), bool))
                    shift_or(yd[k], yp[Al * 3 + Be], u, v)
    pm = np.zeros((9, 4, PR2, PC2), bool)
    for (rho, kap), mask in yd.items():
        i, j = rep[rho], rep[kap]
        pm[cls1(w, i) * 3 + cls1(w, j)] |= mask
        for dy in range(3):
            if not 0 <= i + dy - 1 < npool:
                continue
            for dx in range(3):
                if 0 <= j + dx - 1 < npool:
                    shift_or_back(pm[cls1(w, i + dy - 1) * 3 + cls1(w, j + dx - 1)], mask, dy - 1, dx - 1)
    return m, yp, pm


# ---------------------------------------------------------------------------------------------- tile coverage
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "cmlpl_b200", "csrc")


def _ns(src, name):
    a = src.index("namespace %s {" % name)
    return src[a:src.index("}  // namespace %s" % name, a)]


def _const(block, name):
    return int(re.search(r"\b%s\s*=\s*(\d+)\b" % name, block).group(1))


def tile_constants():
    """The tile constants of the persistent dense kernels, read from their CUDA sources."""
    read = lambda f: open(os.path.join(CSRC, f)).read()
    c1, c2, hd = read("conv1_scene_sm100.cu"), read("conv2_scene_sm100.cu"), read("head_sm100.cu")
    b1, b2, b3 = _ns(c1, "c1p"), _ns(c2, "c2s"), _ns(c2, "p2c")
    nslot = re.search(r"NSLOT\s*=\s*NC\s*==\s*16\s*\?\s*(\d+)\s*:\s*(\d+)", b3)
    plan = re.search(r"static bool spectral_logits_plan.*?const size_t b = (.*?);\s*if \(b <= (\d+)\)", hd, re.S)
    wcb = re.search(r"wc_bytes\(int NC\)\s*\{\s*return (.*?);", hd).group(1)
    kc = re.search(r"kc_spe_in = (.*?);", read("common.cuh")).group(1)
    return dict(c1p_OH=_const(b1, "OH"), c1p_OW=_const(b1, "OW"), c1p_NBUF=_const(b1, "NBUF"),
                c2s_TH=_const(b2, "TH"), c2s_TW=_const(b2, "TW"), p2c_TH=_const(b3, "TH"), p2c_TW=_const(b3, "TW"),
                p2c_NSLOT={16: int(nslot.group(1)), 32: int(nslot.group(2))},
                spl_bytes=re.sub(r"size_t\((\w+)\)", r"\1", plan.group(1)).replace("spl::wc_bytes(NC)", "(%s)" % wcb),
                spl_limit=int(plan.group(2)), kc_spe_in=kc.replace("/", "//"))


def spectral_nA(T, B, NC):
    """input-ring depth spectral_logits_plan picks for B bands at class width NC"""
    KC = eval(T["kc_spe_in"], {"B": B})
    for a in range(4, 0, -1):
        if eval(T["spl_bytes"], {"KC": KC, "a": a, "NC": NC}) <= T["spl_limit"]:
            return a
    return 0


cdiv = lambda a, b: -(-a // b)


def tiles_per_cta(T, band_rows, cols, w, n_spectral, sms):
    """Most tiles one CTA of each persistent dense kernel walks (grid = min(SMs, tiles), tiles t = blockIdx.x + k gridDim.x)"""
    PR, PC = band_rows + w - 1, cols + w - 1
    PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
    per = lambda nt: cdiv(nt, min(sms, nt))
    c1 = cdiv(2 * PR2, T["c1p_OH"]) * cdiv(2 * PC2, T["c1p_OW"])
    c2 = 4 * cdiv(PR2, T["c2s_TH"]) * cdiv(PC2, T["c2s_TW"])
    p2 = 4 * cdiv(PR2, T["p2c_TH"]) * cdiv(PC2, T["p2c_TW"])
    mt = cdiv(n_spectral, 128)
    quarters = min(sms // 4 * 4, mt * 4) // 4                         # CTAs per hidden quarter
    return dict(conv0=per(cdiv(PR * PC, 128)), conv1_pool=per(c1), conv2=per(c2), pool2_cls=per(p2),
                spectral=cdiv(mt, quarters))


# Many-tile cases of the stage test: (name, scene rows, cols, band_row0, band_rows, B, K, w).  A band away from the top
# and bottom reads its halo from a slab of the scene; the slab is all the test generates.
CASES = [
    ("c1_paviau", 610, 340, 0, 610, 103, 9, 20),          # whole PaviaU scene: 12-14 tiles per CTA, partial class quad
    ("c5_mid", 8192, 8192, 4096, 64, 224, 16, 11),        # c5 band: w = 11 kernels, 8192-column boxes, spectral nA = 1
    ("c5_last", 8192, 8192, 8128, 64, 224, 16, 11),       # ... the last band: bottom mirror
    ("houston_top", 601, 2384, 0, 96, 48, 20, 20),        # Houston-2018 band: NC = 32, top mirror
    ("w11_nc32", 300, 260, 0, 300, 160, 30, 11),          # NC = 32 at w = 11, spectral nA = 3, partial class quad
]
# spectral branch alone: (B, K) on 60 001 pixels, nA = 4 / 3 / 2 / 1 at both class widths
SPECTRAL_N = 60001
SPECTRAL_CASES = [(B, K) for B in (103, 150, 204, 224) for K in (13, 24)]
