"""ctypes front end of oracle/triangulate.c.  TEST INFRASTRUCTURE ONLY (see triangulate.c header).

``triangulate_tracks`` takes host arrays in the layout of ``sfm_triangulate_tracks`` (include/sfm_b200.h, "track
triangulation") and returns the same six outputs, computed serially on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libsfm_oracle_triangulate.so")
# the flags of the other C oracles (oracle/Makefile): no implicit contraction, so results compare bit for bit with the kernel
CFLAGS = ["-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-Wall", "-Wextra", "-Wno-unused-parameter"]
STATUS_NAMES = ("triangulated", "too_few_views", "no_model", "too_few_inliers", "invalid")


class TriangulateParams(C.Structure):
    """Mirror of sfm_triangulate_params (include/sfm_b200.h)."""

    _fields_ = [("max_error", C.c_double), ("min_angle", C.c_double), ("confidence", C.c_double), ("seed", C.c_uint64),
                ("max_iters", C.c_int32), ("min_inliers", C.c_int32), ("reserved", C.c_int32 * 6)]


def build(force: bool = False) -> str:
    """Compile triangulate.c into its own library under _build/ when it is missing or older than its sources."""
    srcs = [os.path.join(_HERE, n) for n in ("triangulate.c", "ransac_common.h")] + [os.path.join(_HERE, "..", "include", "sfm_b200.h")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        tmp = f"{_SO}.{os.getpid()}.tmp"
        cc = os.environ.get("CC") or shutil.which("gcc") or "cc"
        subprocess.run([cc, *CFLAGS, "-o", tmp, os.path.join(_HERE, "triangulate.c"), "-lm"], check=True, capture_output=True)
        os.replace(tmp, _SO)                        # atomic: concurrent builders never load a half-written library
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.sfm_oracle_triangulate_tracks.restype = C.c_int
    return _lib


def make_params(*, max_error=4.0, min_angle=1.5, confidence=0.999, seed=0, max_iters=500, min_inliers=2):
    return TriangulateParams(float(max_error), float(min_angle), float(confidence), int(seed), int(max_iters), int(min_inliers))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def triangulate_tracks(offsets, obs, xy, cams, registered=None, **kw):
    """offsets int64 [T+1], obs int32 [n_obs, 2], xy float32 [n_images, S, 2], cams float64 [n_images, 16], registered uint8
    [n_images] or None.  Returns a dict of X [T,3], n_inliers [T], status [T], obs_inlier [n_obs], obs_error [n_obs] and
    counts [5]."""
    offsets = np.ascontiguousarray(offsets, np.int64)
    obs = np.ascontiguousarray(obs, np.int32).reshape(-1, 2)
    xy = np.ascontiguousarray(xy, np.float32)
    cams = np.ascontiguousarray(cams, np.float64).reshape(-1, 16)
    reg = None if registered is None else np.ascontiguousarray(registered, np.uint8)
    n_images, S = xy.shape[0], xy.shape[1]
    T, n_obs = len(offsets) - 1, int(offsets[-1]) if len(offsets) else 0
    prm = make_params(**kw)
    out = {"X": np.zeros((T, 3), np.float64), "n_inliers": np.zeros(T, np.int32), "status": np.zeros(T, np.uint8),
           "obs_inlier": np.zeros(n_obs, np.uint8), "obs_error": np.zeros(n_obs, np.float32), "counts": np.zeros(5, np.int64)}
    rc = lib().sfm_oracle_triangulate_tracks(
        C.c_int(n_images), C.c_int(S), _p(offsets), _p(obs), C.c_int64(T), _p(xy), C.c_int(S), _p(cams), _p(reg), C.byref(prm),
        _p(out["X"]), _p(out["n_inliers"]), _p(out["status"]), _p(out["obs_inlier"]), _p(out["obs_error"]), _p(out["counts"]))
    if rc != 0:
        raise MemoryError("sfm_oracle_triangulate_tracks could not allocate its scratch")
    return out

