"""conv1_pool_kernel at the edges of its tile geometry.  A tile holds 4 conv rows in each of two TMEM frames (frame 1
one scene row below frame 0) and emits 4 pooled rows x 29 pooled columns, so the interesting bands are the ones whose
plane height 2*PR2 leaves a half-used last tile row (2*PR2 mod 4 = 2), whose last tile holds a single pooled cell row,
that are only 1-3 rows high, and whose width leaves a partial last column tile.  Every case is compared with the
float64 pooled border-class planes of tests/dense_refs.py on the kernel's own conv0 map, at w = 20 and w = 11 (which
stores only the top / mid classes of both directions).  Bars: every entry within fp16 rounding plus fp32 accumulation
(dense_refs.bound), max|d| <= 1e-3 * max|ref|, >= 99.9 % of the stored entries bit-equal to the fp16-rounded
reference, entries without a pooled cell exactly 0, no NaN."""
import numpy as np
import pytest
import torch

import dense_refs as D
from oracle import cmlpl_oracle as O

pytestmark = pytest.mark.gpu
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
    q = D.check_conv1_planes(f0, pmq, sd, w, PR, PC)[0]
    print(f"[w={w} R={R} C={C} 2*PR2%4={2 * PR2 % 4}] {q}")
    assert q["nan"] == 0, f"{q['nan']} plane entries never written"
    assert q["noncell_zero"], "plane entries without a pooled cell must be 0"
    assert q["rel"] <= 1e-3 and q["bit_equal"] >= 0.999 and q["ratio"] <= 1.0, q


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
