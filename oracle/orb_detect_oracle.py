"""CPU restatement of cv2.ORB's DETECTION stage.  TEST INFRASTRUCTURE ONLY (nothing under sfm-project_b200/ imports it).

What ``cv2.ORB_create().detect(gray, None)`` (the keypoint half of ``detectAndCompute``, code/feature_matching.py:42-45) does,
as far as it can be observed from outside (OpenCV 4.13.0; pinned by tests/test_oracle_pinned.py against cv2 itself):

* per pyramid level (orb_oracle.build_pyramid): FAST-9/16, threshold 20, response = the largest threshold at which the pixel is
  still a corner, 3 x 3 non-maximum suppression (strictly greater than all eight neighbours), row-major order;
* keypoints closer than 31 pixels to the level's border are dropped; the best 2 n_level by FAST response are retained
  (``retainBest``: everything that reaches the n-th response, left in the order of libstdc++'s nth_element + partition --
  oracle/stl_select.cpp runs those very algorithms);
* Harris response on the UNBLURRED level (7 x 7 block of Sobel-like integer gradients, float32 expression, k = 0.04), the best
  n_level retained the same way; n_level = the geometric split of nfeatures = 500 over 8 levels;
* orientation from the integer intensity moments of the radius-15 disc, ``fastAtan2`` (7th-order odd polynomial, float32);
* pt = level position x float32(1.2 ** level), size = 31 x that factor, octave = level.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import orb_oracle

F32, F64 = np.float32, np.float64
_HERE = os.path.dirname(os.path.abspath(__file__))
_STL = None
CIRCLE = [(0, -3), (1, -3), (2, -2), (3, -1), (3, 0), (3, 1), (2, 2), (1, 3), (0, 3), (-1, 3), (-2, 2), (-3, 1), (-3, 0), (-3, -1), (-2, -2), (-1, -3)]
EDGE, PATCH, HALF, HARRIS_BLOCK, HARRIS_K, FAST_T = 31, 31, 15, 7, F32(0.04), 20


def _stl():
    global _STL
    if _STL is None:
        _STL = C.CDLL(os.path.join(_HERE, "_build", "libsfm_oracle_stl.so"))
        _STL.sfm_oracle_retain_best.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        _STL.sfm_oracle_retain_best.restype = C.c_int
    return _STL


def retain_best(response: np.ndarray, n_points: int) -> np.ndarray:
    """Indices of the survivors of KeyPointsFilter::retainBest, in the order cv2 leaves them."""
    r = np.ascontiguousarray(response, F32)
    out = np.zeros(max(len(r), 1), np.int32)
    n = _stl().sfm_oracle_retain_best(r.ctypes.data_as(C.c_void_p), len(r), int(n_points), out.ctypes.data_as(C.c_void_p))
    return out[:n].copy()


def features_per_level(nfeatures: int = 500, n_levels: int = 8) -> list:
    factor = F32(1.0 / orb_oracle.SCALE_FACTOR)
    nd = F32(nfeatures) * (F32(1) - factor) / (F32(1) - F32(np.power(F64(factor), F64(n_levels))))
    out, total = [], 0
    for _ in range(n_levels - 1):
        out.append(int(np.rint(nd)))
        total += out[-1]
        nd = F32(nd * factor)
    out.append(max(nfeatures - total, 0))
    return out


def umax_table() -> np.ndarray:
    um = np.zeros(HALF + 2, np.int64)
    vmax = int(np.floor(F32(HALF) * np.sqrt(F32(2.0)) / F32(2) + F32(1)))
    vmin = int(np.ceil(F32(HALF) * np.sqrt(F32(2.0)) / F32(2)))
    for v in range(vmax + 1):
        um[v] = int(np.rint(np.sqrt(F64(HALF * HALF - v * v))))
    v0 = 0
    for v in range(HALF, vmin - 1, -1):
        while um[v0] == um[v0 + 1]:
            v0 += 1
        um[v] = v0
        v0 += 1
    return um


def fast_scores(img: np.ndarray) -> np.ndarray:
    """int32 [h, w]: FAST-9/16 corner score (0 where the pixel is not a corner at threshold 20 or lies in the 3-pixel frame)."""
    h, w = img.shape
    out = np.zeros((h, w), np.int32)
    if h < 7 or w < 7:
        return out
    I = img.astype(np.int32)
    c = I[3: h - 3, 3: w - 3]
    d = np.stack([c - I[3 + dy: h - 3 + dy, 3 + dx: w - 3 + dx] for dx, dy in CIRCLE], 0)

    def arcmax(d):
        best = np.full(d.shape[1:], -(10 ** 9))
        for s in range(16):
            best = np.maximum(best, np.minimum.reduce([d[(s + k) % 16] for k in range(9)]))
        return best

    score = np.maximum(arcmax(d), arcmax(-d)) - 1
    out[3: h - 3, 3: w - 3] = np.where(score >= FAST_T, score, 0)
    return out


def fast_keypoints(img: np.ndarray):
    """(x, y, response) of cv2.FastFeatureDetector_create(20, True).detect(img), row-major."""
    S = fast_scores(img)
    P = np.pad(S, 1)
    nb = np.maximum.reduce([P[1 + dy: 1 + dy + S.shape[0], 1 + dx: 1 + dx + S.shape[1]] for dy in (-1, 0, 1) for dx in (-1, 0, 1) if (dx, dy) != (0, 0)])
    ys, xs = np.nonzero((S > 0) & (S > nb))
    return xs.astype(np.int32), ys.astype(np.int32), S[ys, xs].astype(F32)


def harris_responses(img: np.ndarray, xs, ys) -> np.ndarray:
    I = img.astype(np.int64)
    xs, ys = np.asarray(xs, np.int64), np.asarray(ys, np.int64)
    r = HARRIS_BLOCK // 2
    scale = F32(1.0) / (F32(4 * HARRIS_BLOCK) * F32(255.0))
    s4 = F32(F32(F32(scale * scale) * scale) * scale)
    o = np.arange(-r - 1, r + 2)
    P = I[ys[:, None, None] + o[None, :, None], xs[:, None, None] + o[None, None, :]]     # [n, 9, 9] around the 7 x 7 block
    Ix = (P[:, 1:-1, 2:] - P[:, 1:-1, :-2]) * 2 + (P[:, :-2, 2:] - P[:, :-2, :-2]) + (P[:, 2:, 2:] - P[:, 2:, :-2])
    Iy = (P[:, 2:, 1:-1] - P[:, :-2, 1:-1]) * 2 + (P[:, 2:, :-2] - P[:, :-2, :-2]) + (P[:, 2:, 2:] - P[:, :-2, 2:])
    a, b, c = (Ix * Ix).sum((1, 2)), (Iy * Iy).sum((1, 2)), (Ix * Iy).sum((1, 2))
    fa, fb, fc = a.astype(F32), b.astype(F32), c.astype(F32)
    t = fa + fb                                                         # float32 arrays: every operation rounds on its own
    return (((fa * fb) - (fc * fc)) - ((HARRIS_K * t) * t)) * s4


def harris_sums(img: np.ndarray, xs, ys) -> np.ndarray:
    """int64 [n] = a + b of the Harris block (the largest value converted to float32 by the response)."""
    I = img.astype(np.int64)
    xs, ys = np.asarray(xs, np.int64), np.asarray(ys, np.int64)
    o = np.arange(-HARRIS_BLOCK // 2, HARRIS_BLOCK // 2 + 2)
    P = I[ys[:, None, None] + o[None, :, None], xs[:, None, None] + o[None, None, :]]
    Ix = (P[:, 1:-1, 2:] - P[:, 1:-1, :-2]) * 2 + (P[:, :-2, 2:] - P[:, :-2, :-2]) + (P[:, 2:, 2:] - P[:, 2:, :-2])
    Iy = (P[:, 2:, 1:-1] - P[:, :-2, 1:-1]) * 2 + (P[:, 2:, :-2] - P[:, :-2, :-2]) + (P[:, 2:, 2:] - P[:, :-2, 2:])
    return (Ix * Ix).sum((1, 2)) + (Iy * Iy).sum((1, 2))


_P1, _P3, _P5, _P7 = (F32(v) * F32(180.0 / np.pi) for v in (0.9997878412794807, -0.3258083974640975, 0.1555786518463281, -0.04432655554792128))


def fast_atan2(y: np.ndarray, x: np.ndarray) -> np.ndarray:
    y, x = np.asarray(y, F32), np.asarray(x, F32)
    ax, ay = np.abs(x), np.abs(y)
    eps = F32(np.finfo(F64).eps)

    def poly(c):
        c2 = (c * c).astype(F32)
        a = (((_P7 * c2).astype(F32) + _P5).astype(F32) * c2).astype(F32)
        a = (((a + _P3).astype(F32) * c2).astype(F32) + _P1).astype(F32)
        return (a * c).astype(F32)

    with np.errstate(all="ignore"):
        lo = poly((ay / (ax + eps)).astype(F32))
        hi = (F32(90.0) - poly((ax / (ay + eps)).astype(F32))).astype(F32)
    a = np.where(ax >= ay, lo, hi)
    a = np.where(x < 0, (F32(180.0) - a).astype(F32), a)
    a = np.where(y < 0, (F32(360.0) - a).astype(F32), a)
    return a.astype(F32)


def ic_moments(img: np.ndarray, xs, ys):
    """int64 (m01, m10): intensity moments of the radius-15 disc (rows v = -15..15 of half-width umax[|v|])."""
    I = img.astype(np.int64)
    xs, ys = np.asarray(xs, np.int64), np.asarray(ys, np.int64)
    um = umax_table()
    du = np.concatenate([np.arange(-um[abs(v)], um[abs(v)] + 1) for v in range(-HALF, HALF + 1)])
    dv = np.concatenate([np.full(2 * um[abs(v)] + 1, v) for v in range(-HALF, HALF + 1)])
    vals = I[ys[:, None] + dv[None], xs[:, None] + du[None]]
    return (vals * dv).sum(1), (vals * du).sum(1)


def ic_angles(img: np.ndarray, xs, ys) -> np.ndarray:
    m01, m10 = ic_moments(img, xs, ys)
    return fast_atan2(m01.astype(F32), m10.astype(F32))


def level_candidates(levels):
    """Per level, (x, y, FAST response) of the FAST keypoints at least 31 pixels from the border, row-major: what does not
    depend on nfeatures, so that several budgets can share it."""
    out = []
    for im in levels:
        h, w = im.shape
        if h <= 2 * EDGE or w <= 2 * EDGE:
            out.append((np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, F32)))
            continue
        xs, ys, resp = fast_keypoints(im)
        inside = (xs >= EDGE) & (xs < w - EDGE) & (ys >= EDGE) & (ys < h - EDGE)
        out.append((xs[inside], ys[inside], resp[inside]))
    return out


def detect(img: np.ndarray, nfeatures: int = 500, n_levels: int = 8, levels=None, candidates=None) -> np.ndarray:
    """float32 [n, 6] = (pt.x, pt.y, size, angle, response, octave) in cv2's order."""
    levels = orb_oracle.build_pyramid(img, n_levels) if levels is None else levels
    candidates = level_candidates(levels) if candidates is None else candidates
    per = features_per_level(nfeatures, n_levels)
    rows = []
    for lv, im in enumerate(levels):
        xs, ys, resp = candidates[lv]
        keep = retain_best(resp, 2 * per[lv])
        xs, ys = xs[keep], ys[keep]
        hr = harris_responses(im, xs, ys)
        keep = retain_best(hr, per[lv])
        xs, ys, hr = xs[keep], ys[keep], hr[keep]
        ang = ic_angles(im, xs, ys)
        sf = orb_oracle.level_scale(lv)
        px, py = (xs.astype(F32) * sf, ys.astype(F32) * sf) if lv > 0 else (xs.astype(F32), ys.astype(F32))
        rows.append(np.stack([px, py, np.full(len(xs), F32(PATCH) * sf, F32), ang, hr, np.full(len(xs), lv, F32)], 1).astype(F32))
    return np.concatenate(rows).reshape(-1, 6)
