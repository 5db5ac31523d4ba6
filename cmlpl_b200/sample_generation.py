"""``python -m cmlpl_b200.sample_generation`` -- the reference's sample_generation.py CLI
(flags --dataID --num_label --w --n_PC, sample_generation.py:75-82) writing the same
./dataset/<Name>/ contract, with two differences that are both opt-outs:

* the PCA cube is stored once as ``XPCA.npy`` f32 [R,C,n_PC] (+ ``meta.npy`` = [w, R, C]) and the
  19.9 GB materialised ``XP.npy`` is only written with ``--materialize-xp`` (then through the device
  patch-gather kernel, chunked, bit-identical to hyper_tools.py:226-243);
* ``--synthetic`` builds a PaviaU/Salinas/Houston/Indian-Pines/WHU-Hi *shaped* scene when the .mat files
  are not available (they are not, offline).

Splits reproduce sample_generation.py:43-65 exactly (numpy legacy seeds 2 and 0, the sorted
``set`` difference for ``unlabel_array``).
"""
from __future__ import annotations

import argparse
import os

import numpy as np

from .tools.hyper_tools import DATASETS, _MAT, PCANorm, _loadmat, featureNormalize


# dataID -> the synth.SHAPES entry --synthetic builds
SYNTHETIC = {1: "paviau", 2: "salinas", 3: "houston", 4: "indian_pines", 5: "whu_longkou", 6: "whu_hanchuan",
             7: "whu_honghu"}


def split_indices(Y, num_label):
    """sample_generation.py:43-65."""
    n_class = int(Y.max())
    np.random.seed(2)
    labelled = np.where(Y > 0)[0]
    np.random.shuffle(labelled)
    train_parts, test_parts = [], []
    for cls in range(1, n_class + 1):
        members = np.where(Y == cls)[0]
        np.random.seed(0)
        order = np.random.permutation(members.shape[0])
        train_parts.append(members[order[:num_label]])
        test_parts.append(members[order[num_label:]])
    train_array = np.concatenate(train_parts)
    test_array = np.concatenate(test_parts)
    unlabel_array = np.array(list(set(labelled) - set(train_array)))
    return train_array, test_array, unlabel_array


def load_scene(dataID, root="./dataset/", synthetic=False, seed=1088):
    name, n_class, bands = DATASETS[dataID]
    if synthetic:
        from . import synth
        shape = synth.SHAPES[SYNTHETIC[dataID]]
        return synth.synth_scene(*shape, seed=seed)
    fx, kx, fy, ky = _MAT[dataID]
    return _loadmat(os.path.join(root, fx))[kx], _loadmat(os.path.join(root, fy))[ky]


def main(args):
    dataID = int(args.dataID)
    name = DATASETS[dataID][0]
    save_pre_dir = os.path.join(args.root, name) + "/"
    os.makedirs(save_pre_dir, exist_ok=True)
    cube, gt = load_scene(dataID, args.root, args.synthetic)
    row, col, n_feature = cube.shape
    X = cube.reshape(row * col, n_feature)
    X_PCA = featureNormalize(PCANorm(X, args.n_PC), 1).reshape(row, col, args.n_PC)   # hyper_tools.py:289-290
    X = featureNormalize(X, 1)                                                        # hyper_tools.py:292
    Y = gt.reshape(row * col, )
    train_array, test_array, unlabel_array = split_indices(Y, args.num_label)
    np.save(save_pre_dir + "XPCA.npy", X_PCA.astype(np.float32))
    np.save(save_pre_dir + "meta.npy", np.array([args.w, row, col], dtype=np.int64))
    np.save(save_pre_dir + "X.npy", X)
    np.save(save_pre_dir + "Y.npy", Y)
    np.save(save_pre_dir + "train_array.npy", train_array)
    np.save(save_pre_dir + "test_array.npy", test_array)
    np.save(save_pre_dir + "unlabel_array.npy", unlabel_array)
    if args.materialize_xp:
        import torch
        from . import ops
        from .tools.hyper_tools import _to_cube
        cube_d = _to_cube(X_PCA)
        out = np.lib.format.open_memmap(save_pre_dir + "XP.npy", mode="w+", dtype=np.float32,
                                        shape=(row * col, args.n_PC, args.w, args.w))
        step = 8192
        for s in range(0, row * col, step):
            n = min(step, row * col - s)
            out[s:s + n] = ops.patch_gather(cube_d, args.w, first=s, n=n, odd_mode=args.w % 2 == 1).cpu().numpy()
        out.flush()
    return save_pre_dir


def build_parser():
    parser = argparse.ArgumentParser()
    parser.add_argument('--dataID', type=int, default=1)
    parser.add_argument('--num_label', type=int, default=5)
    parser.add_argument('--w', type=int, default=20)
    parser.add_argument('--n_PC', type=int, default=60)
    parser.add_argument('--root', type=str, default='./dataset/')
    parser.add_argument('--synthetic', action='store_true')
    parser.add_argument('--materialize-xp', dest='materialize_xp', action='store_true')
    return parser


if __name__ == '__main__':
    main(build_parser().parse_args())
