"""Seeded synthetic scenes for the matching + verification hot path.

The reference ships no dataset (``code/pipeline.py:25`` points at an absent
``dataset/Bicycle/images``), so every workload in BASELINE.json is synthetic.
This module follows the recipe of SURVEY.md §8(d): random 3-D points seen by
pinhole cameras on an arc, SIFT-like uint8 descriptors (integer valued in
[0,255], row norm ~512) with integer observation noise, per-image clutter, and
a controllable outlier rate for the RANSAC stress configuration.

Everything is plain numpy on the host; nothing here is on the timed path.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

IMG_W, IMG_H = 1920, 1080
K_INTR = np.array([[1000.0, 0.0, 960.0], [0.0, 1000.0, 540.0], [0.0, 0.0, 1.0]])


@dataclass
class Scene:
    """A synthetic multi-view scene.

    desc   uint8  [n_images, n_feats, 128]   SIFT-like descriptors
    xy     float32[n_images, n_feats, 2]     keypoint pixel coordinates
    point  int32  [n_images, n_feats]        scene-point id of each feature, -1 = clutter
    P      float64[n_images, 3, 4]           camera matrices K[R|t]
    X      float64[n_points, 3]              world coordinates of the scene points (``point`` indexes them)
    """

    desc: np.ndarray
    xy: np.ndarray
    point: np.ndarray
    P: np.ndarray
    X: np.ndarray | None = None

    @property
    def n_images(self) -> int:
        return self.desc.shape[0]

    @property
    def n_feats(self) -> int:
        return self.desc.shape[1]

    def true_fundamental(self, i: int, j: int) -> np.ndarray:
        """Ground-truth F with x_j^T F x_i = 0, scaled so ||F||_F = 1."""
        return fundamental_from_cameras(self.P[i], self.P[j])


def sift_like(rng: np.random.Generator, n: int, dim: int = 128) -> np.ndarray:
    """uint8 [n, dim] rows that mimic OpenCV SIFT post-processing.

    Gamma-distributed bins -> L2 normalise -> clip at 0.2 -> renormalise ->
    scale by 512 -> saturate to uint8.
    """
    g = rng.gamma(0.6, 30.0, size=(n, dim))
    g /= np.maximum(np.linalg.norm(g, axis=1, keepdims=True), 1e-12)
    g = np.minimum(g, 0.2)
    g /= np.maximum(np.linalg.norm(g, axis=1, keepdims=True), 1e-12)
    return np.clip(np.rint(g * 512.0), 0, 255).astype(np.uint8)


def observe(rng: np.random.Generator, base: np.ndarray, sigma: float = 6.0) -> np.ndarray:
    """One noisy integer observation of base descriptors."""
    noise = np.rint(rng.normal(0.0, sigma, size=base.shape))
    return np.clip(base.astype(np.int32) + noise.astype(np.int32), 0, 255).astype(np.uint8)


def _look_at(cam_pos: np.ndarray, target: np.ndarray) -> np.ndarray:
    z = target - cam_pos
    z /= np.linalg.norm(z)
    up = np.array([0.0, 1.0, 0.0])
    x = np.cross(up, z)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    return np.stack([x, y, z])  # world -> camera rotation


def make_cameras(n_images: int, baseline: float = 1.0) -> np.ndarray:
    """Cameras on an arc looking at (0,0,6); neighbouring views overlap."""
    target = np.array([0.0, 0.0, 6.0])
    span = baseline * max(n_images - 1, 1) * 0.08
    span = min(span, 2.2)
    Ps = np.zeros((n_images, 3, 4))
    for k in range(n_images):
        a = (k / max(n_images - 1, 1) - 0.5) * span
        pos = np.array([6.0 * np.sin(a), 0.15 * np.cos(3.0 * a), 6.0 - 6.0 * np.cos(a)])
        R = _look_at(pos, target)
        t = -R @ pos
        Ps[k] = K_INTR @ np.concatenate([R, t[:, None]], axis=1)
    return Ps


def fundamental_from_cameras(P1: np.ndarray, P2: np.ndarray) -> np.ndarray:
    """F = [e2]_x P2 P1^+ (Hartley & Zisserman eq. 9.1)."""
    _, _, vt = np.linalg.svd(P1)
    C = vt[-1]
    e2 = P2 @ C
    ex = np.array([[0, -e2[2], e2[1]], [e2[2], 0, -e2[0]], [-e2[1], e2[0], 0]])
    F = ex @ P2 @ np.linalg.pinv(P1)
    return F / np.linalg.norm(F)


def make_scene(
    n_images: int,
    n_feats: int = 8192,
    *,
    seed: int = 0,
    shared_frac: float = 0.5,
    desc_sigma: float = 6.0,
    pixel_sigma: float = 0.5,
    dim: int = 128,
) -> Scene:
    """Build a scene: ``shared_frac`` of each image's features observe common
    3-D points, the rest are per-image clutter."""
    rng = np.random.default_rng(np.random.PCG64(seed))
    n_shared = int(round(n_feats * shared_frac))
    n_points = max(int(n_shared * 1.5), n_shared)
    X = np.empty((n_points, 4))
    X[:, 0:2] = rng.uniform(-2.0, 2.0, size=(n_points, 2))
    X[:, 2] = rng.uniform(4.0, 8.0, size=n_points)
    X[:, 3] = 1.0
    base = sift_like(rng, n_points, dim)
    Ps = make_cameras(n_images)

    desc = np.empty((n_images, n_feats, dim), np.uint8)
    xy = np.empty((n_images, n_feats, 2), np.float32)
    point = np.full((n_images, n_feats), -1, np.int32)
    for k in range(n_images):
        ids = rng.permutation(n_points)[:n_shared]
        x = (Ps[k] @ X[ids].T).T
        px = x[:, :2] / x[:, 2:3] + rng.normal(0.0, pixel_sigma, size=(n_shared, 2))
        slot = rng.permutation(n_feats)
        s_sh, s_cl = slot[:n_shared], slot[n_shared:]
        desc[k, s_sh] = observe(rng, base[ids], desc_sigma)
        xy[k, s_sh] = px.astype(np.float32)
        point[k, s_sh] = ids
        n_cl = n_feats - n_shared
        desc[k, s_cl] = sift_like(rng, n_cl, dim)
        xy[k, s_cl, 0] = rng.uniform(0, IMG_W, n_cl).astype(np.float32)
        xy[k, s_cl, 1] = rng.uniform(0, IMG_H, n_cl).astype(np.float32)
    return Scene(desc=desc, xy=xy, point=point, P=Ps, X=X[:, :3].copy())


def exhaustive_pairs(n_images: int) -> np.ndarray:
    """Unordered pairs (i<j), sorted by (i,j): N(N-1)/2 rows (BASELINE configs 2,3)."""
    i, j = np.triu_indices(n_images, k=1)
    return np.stack([i, j], axis=1).astype(np.int32)


def ordered_pairs(n_images: int) -> np.ndarray:
    """The reference's literal loop order: all (i,j), i != j (code/pipeline.py:38-40)."""
    ii, jj = np.meshgrid(np.arange(n_images), np.arange(n_images), indexing="ij")
    m = ii != jj
    return np.stack([ii[m], jj[m]], axis=1).astype(np.int32)


def windowed_pairs(n_images: int, window: int = 20) -> np.ndarray:
    """Sequential matching: (i, i+1..i+window) (BASELINE config 4: 19,790 pairs at N=1000)."""
    out = [(i, j) for i in range(n_images) for j in range(i + 1, min(i + window, n_images - 1) + 1)]
    return np.asarray(out, np.int32).reshape(-1, 2)


def two_view_correspondences(
    n: int,
    *,
    outlier_frac: float = 0.5,
    seed: int = 0,
    pixel_sigma: float = 0.5,
):
    """Direct synthetic correspondences for RANSAC tests (config 5 shape).

    Returns (pts1 f32[n,2], pts2 f32[n,2], gt_inlier bool[n], F_true f64[3,3]).
    """
    rng = np.random.default_rng(np.random.PCG64(seed))
    Ps = make_cameras(2, baseline=6.0)
    X = np.empty((n, 4))
    X[:, 0:2] = rng.uniform(-2.0, 2.0, size=(n, 2))
    X[:, 2] = rng.uniform(4.0, 8.0, size=n)
    X[:, 3] = 1.0
    pts = []
    for k in range(2):
        x = (Ps[k] @ X.T).T
        pts.append(x[:, :2] / x[:, 2:3] + rng.normal(0.0, pixel_sigma, size=(n, 2)))
    n_out = int(round(n * outlier_frac))
    out_idx = rng.permutation(n)[:n_out]
    pts[1][out_idx, 0] = rng.uniform(0, IMG_W, n_out)
    pts[1][out_idx, 1] = rng.uniform(0, IMG_H, n_out)
    gt = np.ones(n, bool)
    gt[out_idx] = False
    F = fundamental_from_cameras(Ps[0], Ps[1])
    return pts[0].astype(np.float32), pts[1].astype(np.float32), gt, F


def planar_correspondences(n: int, *, outlier_frac: float = 0.3, seed: int = 0, pixel_sigma: float = 0.5):
    """Correspondences of a PLANAR scene (points on the plane z = 6 + 0.2 x) seen by the two cameras of
    ``two_view_correspondences``: explained by a homography.  Returns (pts1 f32[n,2], pts2 f32[n,2], gt_inlier bool[n],
    H_true f64[3,3] with H[2,2] = 1)."""
    rng = np.random.default_rng(np.random.PCG64(seed))
    Ps = make_cameras(2, baseline=6.0)
    X = np.empty((n, 4))
    X[:, 0:2] = rng.uniform(-2.0, 2.0, size=(n, 2))
    X[:, 2] = 6.0 + 0.2 * X[:, 0]
    X[:, 3] = 1.0
    clean = []
    for k in range(2):
        x = (Ps[k] @ X.T).T
        clean.append(x[:, :2] / x[:, 2:3])
    # plane parametrisation (x, y, 1) -> world (x, y, 6 + 0.2 x, 1): each camera sees the plane through a 3x3 map
    B = np.array([[1.0, 0, 0], [0, 1.0, 0], [0.2, 0, 6.0], [0, 0, 1.0]])
    H = (Ps[1] @ B) @ np.linalg.inv(Ps[0] @ B)
    H = H / H[2, 2]
    pts = [c + rng.normal(0.0, pixel_sigma, size=(n, 2)) for c in clean]
    n_out = int(round(n * outlier_frac))
    out_idx = rng.permutation(n)[:n_out]
    pts[1][out_idx, 0] = rng.uniform(0, IMG_W, n_out)
    pts[1][out_idx, 1] = rng.uniform(0, IMG_H, n_out)
    gt = np.ones(n, bool)
    gt[out_idx] = False
    return pts[0].astype(np.float32), pts[1].astype(np.float32), gt, H


def relative_pose(P1: np.ndarray, P2: np.ndarray, K: np.ndarray = None):
    """(R, t) with x2 ~ R x1 + t, |t| = 1, from two projection matrices K[R|t] sharing the intrinsics ``K``."""
    K = K_INTR if K is None else K
    M1, M2 = np.linalg.inv(K) @ P1, np.linalg.inv(K) @ P2
    R1, t1, R2, t2 = M1[:, :3], M1[:, 3], M2[:, :3], M2[:, 3]
    R = R2 @ R1.T
    t = t2 - R @ t1
    return R, t / np.linalg.norm(t)
