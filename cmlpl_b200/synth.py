"""Synthetic hyperspectral scenes of the BASELINE.json shapes (the .mat datasets are not
available offline): blocky class map + noisy class prototypes, PaviaU-like dynamic range."""
from __future__ import annotations

import numpy as np

SHAPES = {
    "paviau": (610, 340, 103, 9),
    "indian_pines": (145, 145, 200, 16),
    "salinas": (512, 217, 204, 16),
    "houston": (349, 1905, 144, 15),
    "whu_longkou": (550, 400, 270, 9),
    "whu_hanchuan": (1217, 303, 274, 16),
    "whu_honghu": (940, 475, 270, 22),
}


def synth_scene(R: int, C: int, B: int, K: int, seed: int = 1088, block: int = 8):
    """-> (cube uint16 [R,C,B], gt uint8 [R,C] with 0 = unlabelled)."""
    rng = np.random.default_rng(seed)
    coarse = rng.integers(0, K + 1, size=(-(-R // block), -(-C // block)))
    gt = np.kron(coarse, np.ones((block, block), dtype=np.int64))[:R, :C]
    flat = gt.reshape(-1)
    for k in range(1, K + 1):
        if (flat == k).sum() < 32:
            flat[rng.choice(flat.size, 32, replace=False)] = k
    gt = flat.reshape(R, C)
    proto = rng.uniform(0, 4000, size=(K + 1, B))
    cube = proto[gt] + rng.normal(0, 200, size=(R, C, B))
    return np.clip(cube, 0, 8000).astype(np.uint16), gt.astype(np.uint8)


def preprocessed_scene(R, C, B, K, n_PC=60, seed=1088, return_raw=False):
    """(cubePCA f32 [R,C,n_PC], spectra f32 [R*C,B], gt) through the reference's preprocessing
    (tools/hyper_tools.py:285-292: PCA + per-channel z-score, float64 on the host)."""
    from .tools.hyper_tools import PCANorm, featureNormalize

    cube, gt = synth_scene(R, C, B, K, seed)
    X = cube.reshape(R * C, B)
    cube_pca = featureNormalize(PCANorm(X, n_PC), 1).reshape(R, C, n_PC).astype(np.float32)
    spectra = featureNormalize(X, 1).astype(np.float32)
    if return_raw:
        return cube_pca, spectra, gt, cube
    return cube_pca, spectra, gt
