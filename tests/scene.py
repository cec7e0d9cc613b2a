"""Deterministic scene builder shared by tests, bench.py and __graft_entry__.smoke().

Restates the recipe of the reference's ``load_test_data`` (/root/reference/gsplat/_helper.py:51-102):
the [-2,2]^3 crop of assets/test_garden.npz (committed as tests/golden/garden_{0,1}.npz), optionally
tiled ``scene_grid`` x ``scene_grid`` times, with random scales in [1e-4, 0.02], unit quaternions
and opacities in [0,1).  Unlike the reference, the random attributes come from numpy's
RandomState(seed) so that every machine (CPU container, GPU box) sees identical inputs.
SH coefficients follow SURVEY.md section 8(d): DC from the point colours, higher bands N(0, 0.1).
"""
from __future__ import annotations

import os

import numpy as np

_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SH_C0 = 0.28209479177387814


def load_garden():
    """The crop is stored in two halves (garden_0.npz holds the cameras) to keep every stored file below 1 MB."""
    parts = [np.load(os.path.join(_GOLDEN, f"garden_{i}.npz")) for i in range(2)]
    g = {k: parts[0][k] for k in parts[0].files}
    for k in ("means", "colors"):
        g[k] = np.concatenate([p[k] for p in parts])
    return g


def make_scene(scene_grid: int = 1, n_max: int | None = None, sh_degree: int = 3, seed: int = 42):
    """Returns dict of float32 numpy arrays: means[N,3] quats[N,4] scales[N,3] opacities[N]
    sh[N,K,3] colors[N,3] viewmats[3,4,4] Ks[3,3,3] and ints width,height."""
    assert scene_grid % 2 == 1
    g = load_garden()
    means, colors = g["means"].astype(np.float32), g["colors"].astype(np.float32) / 255.0
    edges = np.array([4.0, 4.0, 4.0], np.float32)
    r = scene_grid // 2
    gx, gy = np.meshgrid(np.arange(-r, r + 1), np.arange(-r, r + 1), indexing="ij")
    grid = np.stack([gx, gy, np.zeros_like(gx)], -1).reshape(-1, 3).astype(np.float32)
    means = (means[None] + grid[:, None] * edges[None, None]).reshape(-1, 3)
    colors = np.tile(colors, (scene_grid**2, 1))
    rng = np.random.RandomState(seed)
    if n_max is not None and n_max < len(means):
        sel = np.sort(rng.choice(len(means), n_max, replace=False))
        means, colors = means[sel], colors[sel]
    N = len(means)
    scales = (rng.random_sample((N, 3)) * (0.02 - 1e-4) + 1e-4).astype(np.float32)
    quats = rng.standard_normal((N, 4)).astype(np.float32)
    quats /= np.linalg.norm(quats, axis=-1, keepdims=True)
    opacities = rng.random_sample((N,)).astype(np.float32)
    K = (sh_degree + 1) ** 2
    sh = (rng.standard_normal((N, K, 3)) * 0.1).astype(np.float32)
    sh[:, 0, :] = (colors - 0.5) / SH_C0
    return dict(
        means=np.ascontiguousarray(means), quats=quats, scales=scales, opacities=opacities, sh=sh,
        colors=np.ascontiguousarray(colors), viewmats=g["viewmats"].astype(np.float32), Ks=g["Ks"].astype(np.float32),
        width=int(g["width"]), height=int(g["height"]),
    )


def rescale_K(Ks: np.ndarray, w0: int, h0: int, w: int, h: int) -> np.ndarray:
    """Intrinsics for a w x h render of the same field of view (profiling/main.py:101-102)."""
    Ks = Ks.copy()
    Ks[..., 0, :] *= w / w0
    Ks[..., 1, :] *= h / h0
    return Ks
