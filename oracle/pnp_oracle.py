"""Oracles of registration.  TEST INFRASTRUCTURE ONLY (see pnp.c header).

``pnp_ransac`` is the ctypes front end of oracle/pnp.c: host arrays in the layout of ``sfm_pnp_ransac`` (include/sfm_b200.h,
"absolute pose / registration"), the same outputs, computed serially on the CPU.  ``p3p`` exposes its minimal solver.
``gather`` restates ``sfm_pnp_gather`` in numpy.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libsfm_oracle_pnp.so")
# the flags of the other C oracles (oracle/Makefile): no implicit contraction, so results compare bit for bit with the kernel
CFLAGS = ["-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-Wall", "-Wextra", "-Wno-unused-parameter"]
STATUS_NAMES = ("registered", "too_few_points", "no_model", "too_few_inliers", "invalid")


class PnpParams(C.Structure):
    """Mirror of sfm_pnp_params (include/sfm_b200.h)."""

    _fields_ = [("max_error", C.c_double), ("confidence", C.c_double), ("seed", C.c_uint64), ("max_iters", C.c_int32),
                ("min_inliers", C.c_int32), ("min_inlier_ratio", C.c_double), ("refine_iters", C.c_int32), ("reserved", C.c_int32 * 5)]


def build(force: bool = False) -> str:
    """Compile pnp.c into its own library under _build/ when it is missing or older than its sources."""
    srcs = [os.path.join(_HERE, n) for n in ("pnp.c", "ransac_common.h")] + [os.path.join(_HERE, "..", "include", "sfm_b200.h")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        tmp = f"{_SO}.{os.getpid()}.tmp"
        cc = os.environ.get("CC") or shutil.which("gcc") or "cc"
        subprocess.run([cc, *CFLAGS, "-o", tmp, os.path.join(_HERE, "pnp.c"), "-lm"], check=True, capture_output=True)
        os.replace(tmp, _SO)                        # atomic: concurrent builders never load a half-written library
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.sfm_oracle_pnp_ransac.restype = C.c_int
        _lib.sfm_oracle_p3p.restype = C.c_int
    return _lib


def make_params(*, max_error=12.0, confidence=0.9999, seed=0, max_iters=10000, min_inliers=30, min_inlier_ratio=0.25, refine_iters=10):
    return PnpParams(float(max_error), float(confidence), int(seed), int(max_iters), int(min_inliers), float(min_inlier_ratio),
                     int(refine_iters))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def p3p(nxy, X):
    """nxy float64 [3, 2] normalised coordinates, X float64 [3, 3] world points.  Returns a list of (R [3,3], t [3])."""
    nxy = np.ascontiguousarray(nxy, np.float64).reshape(3, 2)
    nx, ny = np.ascontiguousarray(nxy[:, 0]), np.ascontiguousarray(nxy[:, 1])
    X = np.ascontiguousarray(X, np.float64).reshape(9)
    out = np.zeros(48, np.float64)
    n = lib().sfm_oracle_p3p(_p(nx), _p(ny), _p(X), _p(out))
    return [(out[12 * r: 12 * r + 9].reshape(3, 3).copy(), out[12 * r + 9: 12 * r + 12].copy()) for r in range(n)]


def pnp_ransac(xy, X, count, cams, image, **kw):
    """xy float32 [Q, stride, 2], X float64 [Q, stride, 3], count int32 [Q], cams float64 [n_images, 16], image int32 [Q].
    Returns a dict of pose [Q, 12], n_inliers [Q], status [Q], mask [Q, stride], iters [Q] and counts [5]."""
    xy = np.ascontiguousarray(xy, np.float32)
    X = np.ascontiguousarray(X, np.float64)
    Q, stride = xy.shape[0], xy.shape[1]
    count = np.ascontiguousarray(count, np.int32).reshape(Q)
    image = np.ascontiguousarray(image, np.int32).reshape(Q)
    cams = np.ascontiguousarray(cams, np.float64).reshape(-1, 16)
    prm = make_params(**kw)
    out = {"pose": np.zeros((Q, 12), np.float64), "n_inliers": np.zeros(Q, np.int32), "status": np.zeros(Q, np.uint8),
           "mask": np.zeros((Q, stride), np.uint8), "iters": np.zeros(Q, np.int32), "counts": np.zeros(5, np.int64)}
    rc = lib().sfm_oracle_pnp_ransac(C.c_int(cams.shape[0]), _p(cams), _p(image), C.c_int(Q), _p(xy), _p(X), C.c_int(stride), _p(count),
                                     C.byref(prm), _p(out["pose"]), _p(out["n_inliers"]), _p(out["status"]), _p(out["mask"]),
                                     _p(out["iters"]), _p(out["counts"]))
    if rc != 0:
        raise MemoryError("sfm_oracle_pnp_ransac could not allocate its scratch")
    return out


def gather(track_of, n_tracks, point_status, X, xy, image):
    """numpy restatement of sfm_pnp_gather: track_of int32 [n_images, S], point_status uint8 / X float64 [>= n_tracks(, 3)],
    xy float32 [n_images, >= S, 2], image int [Q].  Returns xy [Q, S, 2], X [Q, S, 3], feature [Q, S] (zeros past count) and
    count [Q]."""
    track_of = np.asarray(track_of)
    n_images, S = track_of.shape
    image = np.asarray(image, np.int64).reshape(-1)
    Q = len(image)
    out = {"xy": np.zeros((Q, S, 2), np.float32), "X": np.zeros((Q, S, 3), np.float64), "feature": np.zeros((Q, S), np.int32),
           "count": np.zeros(Q, np.int32)}
    ok_track = np.zeros(n_tracks + 1, bool)                 # slot n_tracks: "no track"
    ok_track[:n_tracks] = np.asarray(point_status)[:n_tracks] == 0
    for q, img in enumerate(image):
        if not 0 <= img < n_images:
            continue
        k = track_of[img].astype(np.int64)
        k = np.where((k >= 0) & (k < n_tracks), k, n_tracks)
        f = np.nonzero(ok_track[k])[0]
        n = len(f)
        out["count"][q] = n
        out["feature"][q, :n] = f
        out["xy"][q, :n] = np.asarray(xy)[img, f]
        out["X"][q, :n] = np.asarray(X)[k[f]]
    return out
