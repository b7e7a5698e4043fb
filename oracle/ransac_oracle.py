"""ctypes front end of oracle/ransac_f.c.  TEST INFRASTRUCTURE ONLY (see ransac_f.c header).

Also holds a float64 numpy restatement of cv2's FM_RANSAC inlier metric
(SURVEY.md A.4: ``max(d1^2, d2^2) <= thr^2``) used to pin the metric against
cv2.findFundamentalMat's own returned mask.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libsfm_oracle.so")


class RansacParams(C.Structure):
    """Mirror of sfm_ransac_params (include/sfm_b200.h)."""

    _fields_ = [
        ("solver", C.c_int32),
        ("score", C.c_int32),
        ("threshold", C.c_float),
        ("max_iters", C.c_int32),
        ("confidence", C.c_double),
        ("seed", C.c_uint64),
        ("lo_refit", C.c_int32),
        ("min_inliers", C.c_int32),
        ("reserved", C.c_int32 * 4),
    ]


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, n) for n in ("ransac_f.c", "ransac_h.c", "pose.c", "ransac_common.h")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.run(["make", "-C", _HERE], check=True, capture_output=True)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        for name in ("ransac_f", "ransac_h", "solve_minimal", "solve_h4", "count_inliers", "count_inliers_h",
                     "smallest_eigvec9", "two_view_pose", "triangulate"):
            getattr(_lib, "sfm_oracle_" + name).restype = C.c_int
        _lib.sfm_oracle_draw_sample.restype = None
    return _lib


def make_params(*, solver=7, score=0, thr=3.0, max_iters=2000, confidence=0.99, seed=0, lo=False, min_inliers=0):
    p = RansacParams()
    p.solver, p.score, p.threshold, p.max_iters = int(solver), int(score), float(thr), int(max_iters)
    p.confidence, p.seed, p.lo_refit, p.min_inliers = float(confidence), int(seed), int(bool(lo)), int(min_inliers)
    return p


def _corr(pts1, pts2):
    c = np.concatenate([np.asarray(pts1, np.float32).reshape(-1, 2), np.asarray(pts2, np.float32).reshape(-1, 2)], axis=1)
    return np.ascontiguousarray(c, np.float32)


def _ransac(entry, pts1, pts2, prm, pair_id, samples, *stop_target):
    """Runs sfm_oracle_ransac_f or sfm_oracle_ransac_h (which also takes stop_target)."""
    corr = _corr(pts1, pts2)
    M = corr.shape[0]
    model = np.zeros(9, np.float64)
    mask = np.zeros(max(M, 1), np.uint8)
    ninl, iters = C.c_int32(0), C.c_int32(0)
    sp = None
    if samples is not None:
        samples = np.ascontiguousarray(samples, np.uint32)
        assert samples.shape == (prm.max_iters, 8)
        sp = samples.ctypes.data_as(C.c_void_p)
    entry(corr.ctypes.data_as(C.c_void_p), C.c_int(M), C.byref(prm), C.c_uint32(pair_id), sp, *stop_target,
          model.ctypes.data_as(C.c_void_p), C.byref(ninl), mask.ctypes.data_as(C.c_void_p), C.byref(iters))
    return (model.reshape(3, 3) if ninl.value > 0 else None), mask[:M], int(ninl.value), int(iters.value)


def ransac_f(pts1, pts2, *, pair_id=0, samples=None, **kw):
    """Returns (F float64[3,3] or None, mask uint8[M], n_inliers, iters)."""
    return _ransac(lib().sfm_oracle_ransac_f, pts1, pts2, make_params(**kw), pair_id, samples)


def solve_minimal(pts1, pts2, idx):
    corr = _corr(pts1, pts2)
    idx = np.ascontiguousarray(idx, np.int32)
    out = np.zeros(27, np.float64)
    n = lib().sfm_oracle_solve_minimal(corr.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p), C.c_int(len(idx)), out.ctypes.data_as(C.c_void_p))
    return out[: 9 * n].reshape(n, 3, 3)


def count_inliers(F, pts1, pts2, thr=3.0, score=0):
    corr = _corr(pts1, pts2)
    F = np.ascontiguousarray(F, np.float64).reshape(9)
    mask = np.zeros(max(corr.shape[0], 1), np.uint8)
    n = lib().sfm_oracle_count_inliers(F.ctypes.data_as(C.c_void_p), corr.ctypes.data_as(C.c_void_p), C.c_int(corr.shape[0]), C.c_float(thr), C.c_int(score), mask.ctypes.data_as(C.c_void_p))
    return int(n), mask[: corr.shape[0]]


def draw_sample(seed, pair, hyp, m, M):
    idx = np.zeros(8, np.int32)
    lib().sfm_oracle_draw_sample(C.c_uint64(seed), C.c_uint32(pair), C.c_uint32(hyp), C.c_int(m), C.c_int(M), idx.ctypes.data_as(C.c_void_p))
    return idx[:m]


# --------------------------------------------------------- float64 restatements

def sym_epipolar_err(F, pts1, pts2):
    """cv2 FM_RANSAC's per-point error, float64: max of the two squared
    point-to-epipolar-line distances (SURVEY.md A.4)."""
    F = np.asarray(F, np.float64).reshape(3, 3)
    p1 = np.concatenate([np.asarray(pts1, np.float64).reshape(-1, 2), np.ones((len(pts1), 1))], 1)
    p2 = np.concatenate([np.asarray(pts2, np.float64).reshape(-1, 2), np.ones((len(pts2), 1))], 1)
    l2 = p1 @ F.T          # F x1: line in image 2
    l1 = p2 @ F            # F^T x2: line in image 1
    num = (p2 * l2).sum(1) ** 2
    d2 = num / (l2[:, 0] ** 2 + l2[:, 1] ** 2)
    d1 = num / (l1[:, 0] ** 2 + l1[:, 1] ** 2)
    return np.maximum(d1, d2)


def sampson_err(F, pts1, pts2):
    F = np.asarray(F, np.float64).reshape(3, 3)
    p1 = np.concatenate([np.asarray(pts1, np.float64).reshape(-1, 2), np.ones((len(pts1), 1))], 1)
    p2 = np.concatenate([np.asarray(pts2, np.float64).reshape(-1, 2), np.ones((len(pts2), 1))], 1)
    l2 = p1 @ F.T
    l1 = p2 @ F
    num = (p2 * l2).sum(1) ** 2
    return num / (l2[:, 0] ** 2 + l2[:, 1] ** 2 + l1[:, 0] ** 2 + l1[:, 1] ** 2)


def iou(a, b) -> float:
    a = np.asarray(a).astype(bool).ravel()
    b = np.asarray(b).astype(bool).ravel()
    u = (a | b).sum()
    return float((a & b).sum() / u) if u else 1.0


# ------------------------------------------------------------------ homography (oracle/ransac_h.c)

def ransac_h(pts1, pts2, *, pair_id=0, samples=None, thr=3.0, max_iters=2000, confidence=0.995, seed=0, lo=False, min_inliers=0,
             stop_target=0):
    """Returns (H float64[3,3] or None, mask uint8[M], n_inliers, iters)."""
    prm = make_params(solver=8, thr=thr, max_iters=max_iters, confidence=confidence, seed=seed, lo=lo, min_inliers=min_inliers)
    return _ransac(lib().sfm_oracle_ransac_h, pts1, pts2, prm, pair_id, samples, C.c_int(int(stop_target)))


def solve_h4(pts1, pts2, idx):
    corr = _corr(pts1, pts2)
    idx = np.ascontiguousarray(idx, np.int32)
    out = np.zeros(9, np.float64)
    ok = lib().sfm_oracle_solve_h4(corr.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out.reshape(3, 3) if ok else None


def transfer_err(H, pts1, pts2):
    """cv2 findHomography's per-point error, float64: squared forward reprojection distance."""
    H = np.asarray(H, np.float64).reshape(3, 3)
    p1 = np.concatenate([np.asarray(pts1, np.float64).reshape(-1, 2), np.ones((len(pts1), 1))], 1)
    q = p1 @ H.T
    return ((q[:, :2] / q[:, 2:3] - np.asarray(pts2, np.float64).reshape(-1, 2)) ** 2).sum(1)


# ------------------------------------------------------------------ two-view pose (oracle/pose.c)

def two_view_pose(pts1, pts2, F, cam, *, mask=None, distance_thresh=50.0):
    """Returns (n_good, R [3,3], t [3], E [3,3], mask uint8 [M], X float32 [M,3])."""
    corr = _corr(pts1, pts2)
    M = corr.shape[0]
    F = np.ascontiguousarray(F, np.float64).reshape(9)
    cam = np.ascontiguousarray(cam, np.float64).reshape(8)
    R, t, E = np.zeros(9), np.zeros(3), np.zeros(9)
    omask = np.zeros(max(M, 1), np.uint8)
    X = np.zeros((max(M, 1), 3), np.float32)
    mp = None
    if mask is not None:
        mask = np.ascontiguousarray(np.asarray(mask).ravel(), np.uint8)
        assert mask.shape[0] == M
        mp = mask.ctypes.data_as(C.c_void_p)
    n = lib().sfm_oracle_two_view_pose(corr.ctypes.data_as(C.c_void_p), C.c_int(M), mp, F.ctypes.data_as(C.c_void_p),
                                       cam.ctypes.data_as(C.c_void_p), C.c_double(distance_thresh), R.ctypes.data_as(C.c_void_p),
                                       t.ctypes.data_as(C.c_void_p), E.ctypes.data_as(C.c_void_p), omask.ctypes.data_as(C.c_void_p),
                                       X.ctypes.data_as(C.c_void_p))
    return int(n), R.reshape(3, 3), t, E.reshape(3, 3), omask[:M], X[:M]
