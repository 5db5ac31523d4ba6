"""CPU tests (-m "not gpu") of the data-layer drop-ins against what the UNMODIFIED reference produced
(tests/golden/loader.npz, written by oracle/make_golden.py::gold_loader from the reference's own
sample_generation.main + hsi_loader.HSIDataSet): split arrays, lengths / order / items of every ``setindex`` mode
including both tiling branches (hsi_loader.py:29-45), for the cube-backed layout (XPCA.npy) and the reference's
materialised XP.npy layout."""
import os

import numpy as np
import pytest

from oracle import cmlpl_oracle as O
from oracle import golden

CASES = {"label_tiled": dict(setindex="label", max_iters=137), "label_plain": dict(setindex="label"),
         "unlabel_head": dict(setindex="unlabel", max_iters=300, num_unlabel=200),
         "unlabel_short": dict(setindex="unlabel", max_iters=96, num_unlabel=200),
         "unlabel_plain": dict(setindex="unlabel", num_unlabel=50),
         "test": dict(setindex="test"), "wholeset": dict(setindex="wholeset")}


@pytest.fixture(scope="module")
def gold(golden_dir):
    return golden.load(os.path.join(golden_dir, "loader.npz")), golden.load(os.path.join(golden_dir, "train_infer.npz"))


def _write_dir(root, z, ti, materialise):
    os.makedirs(root, exist_ok=True)
    for f in ("train_array", "test_array", "unlabel_array", "Y", "X"):
        np.save(os.path.join(root, f + ".npy"), z[f])
    if materialise:
        np.save(os.path.join(root, "XP.npy"), O.extract_patches(ti["cube_pca"], 20))       # the reference's layout
    else:
        np.save(os.path.join(root, "XPCA.npy"), ti["cube_pca"])
        np.save(os.path.join(root, "meta.npy"), np.array([20, 40, 36], dtype=np.int64))
    return root + "/"


def test_split_indices_match_the_reference_files(gold):
    from cmlpl_b200 import sample_generation as SG
    z, ti = gold
    tr, te, un = SG.split_indices(z["Y"], 5)
    assert np.array_equal(tr, z["train_array"]) and np.array_equal(te, z["test_array"])
    assert np.array_equal(un, z["unlabel_array"])            # the sorted set difference (sample_generation.py:65)
    assert tr.dtype == z["train_array"].dtype and un.dtype == z["unlabel_array"].dtype
    # the same arrays the training fixture was produced with
    assert np.array_equal(tr, ti["train_array"]) and np.array_equal(un, ti["unlabel_array"])


@pytest.mark.parametrize("materialise", [False, True])
def test_hsidataset_matches_the_reference(gold, tmp_path, materialise):
    from cmlpl_b200.hsi_loader import HSIDataSet
    z, ti = gold
    root = _write_dir(str(tmp_path / ("xp" if materialise else "cube")), z, ti, materialise)
    for name, kw in CASES.items():
        ds = HSIDataSet(1, root=root, **kw)
        assert ds.scene_ready == (not materialise)
        n = int(z[f"{name}.len"])
        assert len(ds) == n, name
        assert len(ds[0]) == int(z[f"{name}.arity"]), name                    # (XP, X, Y) or (XP, X) for 'wholeset'
        sig = np.array([ds[i][1][:4] for i in range(n)])
        assert np.array_equal(sig, z[f"{name}.spec_sig"]), name               # same pixels in the same (tiled) order
        if kw["setindex"] != "wholeset":
            assert np.array_equal(np.array([int(ds[i][2]) for i in range(n)]), z[f"{name}.labels"]), name
        for j, i in enumerate(z[f"{name}.picks"][:2]):
            item = ds[int(i)]
            assert item[0].dtype == np.float32 and item[0].shape == (60, 20, 20) and item[0].flags["C_CONTIGUOUS"]
            assert np.array_equal(item[0], z[f"{name}.item{j}.xp"]), (name, i)   # bit-exact patch
            assert item[1].dtype == np.float32 and np.array_equal(item[1], z[f"{name}.item{j}.x"])
            if len(item) == 3:
                assert np.issubdtype(np.asarray(item[2]).dtype, np.integer)
    with pytest.raises(ValueError):
        HSIDataSet(1, setindex="bogus", root=root)


def test_synthetic_generator_is_the_oracles(gold):
    """One recipe, two call sites: the product's synthetic scene equals the oracle's (SURVEY 8d)."""
    from cmlpl_b200 import synth
    for shape in ((40, 36, 103, 9), (23, 31, 20, 4)):
        a, ga = synth.synth_scene(*shape, seed=1088)
        b, gb = O.synth_cube(*shape, seed=1088)
        assert np.array_equal(a, b) and np.array_equal(ga, gb) and a.dtype == b.dtype == np.uint16


def test_sample_generation_cli_writes_the_reference_file_contract(gold, tmp_path, monkeypatch):
    """python -m cmlpl_b200.sample_generation on the scene the reference's sample_generation.main was run on
    (oracle/make_golden.py::gold_loader): X.npy / Y.npy / the three index arrays equal the reference's files, XPCA.npy is
    the float32 PCA cube the reference materialises patches from, and no XP.npy is written unless asked for."""
    from cmlpl_b200 import sample_generation as SG, synth
    z, ti = gold
    monkeypatch.setitem(synth.SHAPES, "paviau", (40, 36, 103, 9))
    root = str(tmp_path) + "/"
    d = SG.main(SG.build_parser().parse_args(["--dataID", "1", "--root", root, "--synthetic"]))
    assert sorted(os.listdir(d)) == ["X.npy", "XPCA.npy", "Y.npy", "meta.npy", "test_array.npy", "train_array.npy",
                                     "unlabel_array.npy"]
    X = np.load(d + "X.npy")
    assert X.dtype == np.float64 and X.shape == z["X"].shape                      # hsi_loader.py:21 reads float64
    assert np.abs(X - z["X"]).max() <= 1e-12 * np.abs(z["X"]).max()
    Y = np.load(d + "Y.npy")
    assert Y.dtype == z["Y"].dtype and np.array_equal(Y, z["Y"])
    for f in ("train_array", "test_array", "unlabel_array"):
        a = np.load(d + f + ".npy")
        assert a.dtype == z[f].dtype and np.array_equal(a, z[f]), f
    cube = np.load(d + "XPCA.npy")
    assert cube.dtype == np.float32 and cube.shape == (40, 36, 60)
    assert np.abs(cube - ti["cube_pca"]).max() <= 1e-5 * np.abs(ti["cube_pca"]).max()
    assert np.array_equal(np.load(d + "meta.npy"), np.array([20, 40, 36]))
