"""CPU restatement of cv2.ORB's descriptor stage.  TEST INFRASTRUCTURE ONLY (nothing under sfm-project_b200/ imports it).

Follows what ``cv2.ORB_create().detectAndCompute`` (code/feature_matching.py:42-45) does AFTER keypoint detection, as far
as it can be observed from outside (OpenCV 4.13.0; sources not on disk, behaviour pinned by tests/test_oracle_pinned.py
against cv2 itself):

* pyramid: level k has size (round(w * (1 / s_k)), round(h * (1 / s_k))) in float32, s_k = float32(1.2f ** k), round half to
  even, and is resized from level k-1 with
  INTER_LINEAR_EXACT (taken from cv2.resize here: the GPU stage receives the pyramid, it does not build it);
* each level is blurred with GaussianBlur(7x7, sigma 2), which for a sub-matrix source is sepFilter2D with the float32
  kernel: rows  s = k[-3] x[-3]; s = fma(k[d], x[d], s), d = -2..3;  columns  s = k[0] x[0]; s = fma(k[d], x[d] + x[-d], s),
  d = 1..3;  result = round-half-even(s) -- the association that reproduces cv2.sepFilter2D bit for bit on a host with FMA;
* descriptor: centre = (round(pt.x / s), round(pt.y / s)) in the level image, float32 a = cos, b = sin of the angle,
  sample i at (round(x a - y b), round(x b + y a)), bit = I(a_i) < I(b_i), 8 bits per byte, LSB first.
"""
from __future__ import annotations

import cv2
import numpy as np

F32, F64 = np.float32, np.float64
SCALE_FACTOR = F64(F32(1.2))
N_LEVELS = 8


def level_scale(level: int) -> np.float32:
    return F32(np.power(SCALE_FACTOR, F64(level)))


def gaussian_kernel() -> np.ndarray:
    return cv2.getGaussianKernel(7, 2, cv2.CV_32F).ravel().astype(F32)


def build_pyramid(img: np.ndarray, n_levels: int = N_LEVELS):
    """Unblurred level images, each resized from the previous one (what ORB keeps in its pyramid buffer)."""
    h, w = img.shape
    levels = [np.ascontiguousarray(img)]
    for k in range(1, n_levels):
        inv = F32(F32(1.0) / level_scale(k))                              # cv2 multiplies by the inverse scale; it does not divide
        sz = (int(np.rint(F32(F32(w) * inv))), int(np.rint(F32(F32(h) * inv))))
        levels.append(cv2.resize(levels[-1], sz, interpolation=cv2.INTER_LINEAR_EXACT))
    return levels


def _fma(a, b, c):
    return (a.astype(F64) * b.astype(F64) + c.astype(F64)).astype(F32)


def blur_level(img: np.ndarray) -> np.ndarray:
    """GaussianBlur(img, (7, 7), 2, 2, BORDER_REFLECT_101) as ORB's sub-matrix call computes it (see module docstring)."""
    k = gaussian_kernel()
    h, w = img.shape
    x = np.pad(img.astype(F32), ((0, 0), (3, 3)), mode="reflect")
    K = lambda d: np.full((h, w), k[3 + d], F32)  # noqa: E731
    s = (K(-3) * x[:, 0:w]).astype(F32)
    for d in range(-2, 4):
        s = _fma(K(d), x[:, 3 + d: 3 + d + w], s)
    y = np.pad(s, ((3, 3), (0, 0)), mode="reflect")
    v = (K(0) * y[3: 3 + h]).astype(F32)
    for d in (1, 2, 3):
        v = _fma(K(d), (y[3 + d: 3 + d + h] + y[3 - d: 3 - d + h]).astype(F32), v)
    return np.clip(np.rint(v), 0, 255).astype(np.uint8)


def keypoint_arrays(kps):
    """float32 [n, 4] = (pt.x, pt.y, angle in degrees, octave)."""
    return np.array([[k.pt[0], k.pt[1], k.angle, k.octave] for k in kps], F32).reshape(-1, 4)


def describe(img: np.ndarray, kps, pattern: np.ndarray, levels=None) -> np.ndarray:
    """uint8 [n, 32] descriptors of cv2 keypoints (list of cv2.KeyPoint or float32 [n, 4] rows) on ``img``."""
    kp = keypoint_arrays(kps) if not isinstance(kps, np.ndarray) else kps.astype(F32)
    levels = build_pyramid(img) if levels is None else levels
    blurred = {}
    pat = pattern.astype(F32)
    out = np.zeros((len(kp), 32), np.uint8)
    for n, (px, py, ang, octave) in enumerate(kp):
        lv = int(octave)
        if lv not in blurred:
            blurred[lv] = blur_level(levels[lv])
        im = blurred[lv]
        inv = F32(1.0) / level_scale(lv)
        cx, cy = int(np.rint(F32(px) * inv)), int(np.rint(F32(py) * inv))
        rad = F32(ang) * F32(np.pi / 180.0)
        a, b = F32(np.cos(F64(rad))), F32(np.sin(F64(rad)))
        xa = (pat[:, 0] * a).astype(F32) - (pat[:, 1] * b).astype(F32)
        ya = (pat[:, 0] * b).astype(F32) + (pat[:, 1] * a).astype(F32)
        xb = (pat[:, 2] * a).astype(F32) - (pat[:, 3] * b).astype(F32)
        yb = (pat[:, 2] * b).astype(F32) + (pat[:, 3] * a).astype(F32)
        va = im[cy + np.rint(ya).astype(int), cx + np.rint(xa).astype(int)]
        vb = im[cy + np.rint(yb).astype(int), cx + np.rint(xb).astype(int)]
        out[n] = np.packbits(va < vb, bitorder="little")
    return out
