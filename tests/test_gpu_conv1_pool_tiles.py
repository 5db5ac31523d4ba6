"""conv1_pool_kernel at the edges of its tile geometry.  A tile holds 4 conv rows in each of two TMEM frames (frame 1
one scene row below frame 0) and emits 4 pooled rows x 29 pooled columns, so the interesting bands are the ones whose
plane height 2*PR2 leaves a half-used last tile row (2*PR2 mod 4 = 2), whose last tile holds a single pooled cell row,
that are only 1-3 rows high, and whose width leaves a partial last column tile.  Every case is compared with a plain
torch fp32 evaluation of the pooled border-class planes on the kernel's own conv0 map, at w = 20 and w = 11 (which
stores only the top / mid classes of both directions).  Bars: max|d| <= 1e-3 * max|ref|, >= 99.9 % of the stored
entries bit-equal to the fp16-rounded reference, entries without a pooled cell exactly 0, no NaN."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cmlpl_oracle as O

pytestmark = pytest.mark.gpu
S = ((1, 2), (0, 1, 2), (0, 1))     # conv1 taps dy (dx) a top / mid / bottom (left / mid / right) patch border keeps
AB = ((0, 1), (1, 1), (1, 2))       # conv1 border class of the two rows (columns) of a top / mid / bottom pooled cell


def planes_ref(f0, W1, b1, PR, PC):
    """torch fp32: G[a][b] = relu(b1 + F0 + the taps border class (a, b) keeps), PM[A][B] = the 2x2 mean of
    G[a(A,u)][b(B,v)], scattered into the parity planes [9][4][8 chunks][PR2][PC2][8]; plus the mask of plane
    entries that hold a pooled cell (pr < PR-1, pc < PC-1)."""
    PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
    F0 = f0.view(8, PR, PC, 8).permute(0, 3, 1, 2).reshape(64, PR, PC).float()
    Fp = F.pad(F0, (1, 1, 1, 1))
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


# (w, band rows, columns): 2*PR2 mod 4 = 0 and 2 at both windows; 1-, 2- and 3-row bands; bands whose last tile holds a
# single pooled cell row (PR = 2 mod 4); widths from a sliver to a few tiles, none a multiple of the 29-column tile
# (the scene itself is at least 12 rows high and w/2 columns wide: the conv0 map mirrors its halo from inside the scene)
CASES = [(20, 1, 10), (20, 2, 40), (20, 3, 13), (20, 7, 50), (20, 10, 11), (20, 13, 75),
         (11, 1, 7), (11, 2, 30), (11, 3, 29), (11, 4, 41), (11, 8, 5)]


@pytest.mark.parametrize("w,R,C", CASES)
def test_conv1_pool_tile_edges_match_torch(dev, w, R, C):
    from cmlpl_b200 import _lib, ops
    B, K = 103, 9
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(R * 1000 + C)
    SR = max(R, 12)                                   # scene rows; the band is its first R rows
    cube = torch.from_numpy(rng.standard_normal((SR, C, 60)).astype(np.float32)).to(dev)
    torch.manual_seed(R * 1000 + C)
    sd = {k: v.to(dev) for k, v in O.basenet2_init(B, K, conv_feat=1600 if w == 20 else 256).items()}
    packed = ops.pack_basenet2(sd, B, K, w)
    PR, PC = R + w - 1, C + w - 1
    PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
    f0 = torch.empty(8 * PR * PC * 8, dtype=torch.float16, device=dev)
    pmq = torch.full((9, 4, 8, PR2, PC2, 8), float("nan"), dtype=torch.float16, device=dev)
    _lib.call("cmlpl_conv0_map_f16", cube.data_ptr(), SR, C, 0, SR, w, 0, R, packed.data_ptr(), f0.data_ptr(), st)
    _lib.call("cmlpl_conv1_pool_planes_f16", f0.data_ptr(), C, w, R, packed.data_ptr(), pmq.data_ptr(), st)
    torch.cuda.synchronize()
    ref, cell = planes_ref(f0, sd["conv1.weight"].half().float(), sd["conv1.bias"], PR, PC)
    ncls = 3 if w == 20 else 2
    idx = [A * 3 + Bc for A in range(ncls) for Bc in range(ncls)]
    got, want = pmq[idx].float(), ref[idx]
    assert not torch.isnan(got).any(), f"{int(torch.isnan(got).sum())} plane entries never written"
    off = ~cell.view(1, 4, 1, PR2, PC2, 1).expand_as(got)
    assert (got[off] == 0).all(), "plane entries without a pooled cell must be 0"
    rel = float((got - want).abs().max() / want.abs().max())
    bit_equal = float((pmq[idx] == want.half()).float().mean())
    print(f"[w={w} R={R} C={C} 2*PR2%4={2 * PR2 % 4}] max|d|/max|ref| {rel:.2e}, bit-equal {bit_equal:.5f}")
    assert rel <= 1e-3 and bit_equal >= 0.999, (rel, bit_equal)


def test_cases_cover_the_tile_edges():
    """The parameter list above reaches every edge it claims to: both values of 2*PR2 mod 4 at both windows, a last
    tile with a single pooled cell row, 1-3 row bands and partial last column tiles."""
    seen = set()
    for w, R, C in CASES:
        PR, PC = R + w - 1, C + w - 1
        PR2, PC2 = (PR + 1) // 2, (PC + 1) // 2
        seen.add((w, "mod4", 2 * PR2 % 4))
        if (PR - 1) % 4 == 1:                      # cell rows 0..PR-2: the last tile starts at a multiple of 4
            seen.add((w, "single"))
        if R <= 3:
            seen.add(("rows", R))
        if (2 * PC2) % 29:
            seen.add((w, "partial"))
    for w in (20, 11):
        assert {(w, "mod4", 0), (w, "mod4", 2), (w, "single"), (w, "partial")} <= seen, (w, seen)
    assert {("rows", 1), ("rows", 2), ("rows", 3)} <= seen
