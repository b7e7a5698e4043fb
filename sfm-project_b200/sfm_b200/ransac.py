"""Batched RANSAC fundamental-matrix verification (C ABI: sfm_ransac_f_batch).

Fills the reference's empty ``code/geometric_verification.py``; conventions follow
``cv2.findFundamentalMat(FM_RANSAC)`` (SURVEY.md A.4).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib


@dataclass
class VerifyBatch:
    """F float64 [P,3,3] (zeros when no model), n_inliers int32 [P], mask uint8 [P, cap], iters int32 [P]."""

    F: torch.Tensor
    n_inliers: torch.Tensor
    mask: torch.Tensor
    iters: torch.Tensor


def ransac_params(*, thr=3.0, confidence=0.99, max_iters=2000, solver="7pt", score="sym_epipolar", lo=False, seed=0,
                  min_inliers=0) -> _lib.RansacParams:
    if solver not in _lib.SOLVERS:
        raise ValueError(f"solver must be '7pt' or '8pt', got {solver!r}")
    if score not in _lib.SCORES:
        raise ValueError(f"score must be one of {list(_lib.SCORES)}, got {score!r}")
    if not (thr > 0) or max_iters <= 0:
        raise ValueError("thr and max_iters must be positive")
    p = _lib.RansacParams()
    p.solver, p.score = _lib.SOLVERS[solver], _lib.SCORES[score]
    p.threshold, p.max_iters, p.confidence = float(thr), int(max_iters), float(confidence)
    p.seed, p.lo_refit, p.min_inliers = int(seed), int(bool(lo)), int(min_inliers)
    return p


def _run(entry: str, corr: torch.Tensor, counts: torch.Tensor, prm, pair_id, samples, *stop_target) -> VerifyBatch:
    """One call of ``sfm_ransac_f_batch`` or, with a ``stop_target`` argument (None or [P]), ``sfm_ransac_h_batch``."""
    if corr.dtype != torch.float32 or corr.dim() != 3 or corr.shape[2] != 4 or not corr.is_cuda:
        raise ValueError("corr must be a CUDA float32 tensor [P, cap, 4]")
    corr = corr.contiguous()
    counts = counts.to(device=corr.device, dtype=torch.int32).contiguous()
    P, cap, dev = corr.shape[0], corr.shape[1], corr.device
    model = torch.zeros((P, 3, 3), dtype=torch.float64, device=dev)
    ninl = torch.zeros(P, dtype=torch.int32, device=dev)
    mask = torch.zeros((P, cap), dtype=torch.uint8, device=dev)
    iters = torch.zeros(P, dtype=torch.int32, device=dev)
    pid = None if pair_id is None else torch.as_tensor(np.asarray(pair_id, np.int64).astype(np.uint32).view(np.int32)).to(dev)
    smp = None
    if samples is not None:
        s = np.ascontiguousarray(samples, np.uint32)
        if s.shape != (prm.max_iters, 8):
            raise ValueError(f"samples must be [max_iters, 8], got {s.shape}")
        smp = torch.from_numpy(s.view(np.int32)).to(dev)
    tgt = [None if t is None else torch.as_tensor(t).to(device=dev, dtype=torch.int32).contiguous() for t in stop_target]
    if any(t is not None and tuple(t.shape) != (P,) for t in tgt):
        raise ValueError("stop_target must be [P]")
    if P:
        _lib.check(
            getattr(_lib.lib(), entry)(_lib.ptr(corr), cap, _lib.ptr(counts), P, _lib.ptr(pid), _lib.ptr(smp), *map(_lib.ptr, tgt),
                                       C.byref(prm), _lib.ptr(model), _lib.ptr(ninl), _lib.ptr(mask), _lib.ptr(iters),
                                       _lib.current_stream_ptr(dev)),
            entry,
        )
    return VerifyBatch(model, ninl, mask, iters)


def verify_corr(corr: torch.Tensor, counts: torch.Tensor, *, pair_id=None, samples=None, **kw) -> VerifyBatch:
    """corr float32 [P, cap, 4] (x1,y1,x2,y2) on the GPU, counts int32 [P]."""
    return _run("sfm_ransac_f_batch", corr, counts, ransac_params(**kw), pair_id, samples)


def h_stop_target(n_inliers_f, ratio: float):
    """The homography stop target of the scene-graph test "does H explain more than ``ratio`` of what F explains":
    floor(ratio * n) in INTEGER arithmetic (ratio rounded up to a multiple of 2^-16), so that python ints, numpy arrays and
    device tensors give the same number and every public API hands the same target to sfm_ransac_h_*."""
    num = int(np.ceil(float(ratio) * 65536.0 - 1e-9))
    if isinstance(n_inliers_f, torch.Tensor):
        return ((n_inliers_f.to(torch.int64) * num) >> 16).to(torch.int32)
    if isinstance(n_inliers_f, np.ndarray):
        return ((n_inliers_f.astype(np.int64) * num) >> 16).astype(np.int32)
    return (int(n_inliers_f) * num) >> 16


def verify_h_corr(corr: torch.Tensor, counts: torch.Tensor, *, pair_id=None, samples=None, thr=3.0, confidence=0.995,
                  max_iters=2000, lo=False, seed=0, min_inliers=0, stop_target=None) -> VerifyBatch:
    """Batched RANSAC homography on the same buffers as ``verify_corr`` (C ABI: sfm_ransac_h_batch); conventions of
    ``cv2.findHomography(RANSAC)``.  ``VerifyBatch.F`` holds H (x2 ~ H x1, H[2,2] == 1).  ``stop_target`` (int32 [P], e.g.
    0.8 * the pair's F inliers) ends sampling once a model with that support would have been found (see include/sfm_b200.h)."""
    prm = ransac_params(thr=thr, confidence=confidence, max_iters=max_iters, solver="8pt", lo=lo, seed=seed, min_inliers=min_inliers)
    return _run("sfm_ransac_h_batch", corr, counts, prm, pair_id, samples, stop_target)


@dataclass
class PoseBatch:
    """R float64 [P,3,3], t float64 [P,3] (x2 ~ R x1 + t, |t| = 1; zeros when no pose), E float64 [P,3,3] (unit Frobenius
    norm), n_good int32 [P], mask uint8 [P, cap] (inlier AND in front of both cameras), points float32 [P, cap, 3]."""

    R: torch.Tensor
    t: torch.Tensor
    E: torch.Tensor
    n_good: torch.Tensor
    mask: torch.Tensor
    points: torch.Tensor


def camera_rows(K1, K2=None, P: int = 1) -> np.ndarray:
    """float64 [P, 8] rows (fx1 fy1 cx1 cy1 fx2 fy2 cx2 cy2) from 3x3 pinhole matrices (one shared, or one per pair)."""
    def four(K):
        K = np.asarray(K, np.float64)
        if K.shape[-2:] != (3, 3):
            raise ValueError(f"camera matrix must be [3,3] or [P,3,3], got {K.shape}")
        if np.any(np.abs(K[..., 0, 1]) > 1e-12):
            raise ValueError("camera matrices with skew are not supported")
        K = np.broadcast_to(K, (P, 3, 3))
        return np.stack([K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2]], axis=1)
    a = four(K1)
    b = a if K2 is None else four(K2)
    return np.ascontiguousarray(np.concatenate([a, b], axis=1))


def recover_pose_corr(corr: torch.Tensor, counts: torch.Tensor, F: torch.Tensor, cam, *, mask: torch.Tensor | None = None,
                      distance_thresh: float = 50.0) -> PoseBatch:
    """Batched E = K2^T F K1 -> (R, t) by cheirality vote + DLT triangulation (C ABI: sfm_two_view_pose_batch);
    conventions of ``cv2.recoverPose`` / ``cv2.triangulatePoints``.  ``cam`` float64 [P,8] (see ``camera_rows``)."""
    if corr.dtype != torch.float32 or corr.dim() != 3 or corr.shape[2] != 4 or not corr.is_cuda:
        raise ValueError("corr must be a CUDA float32 tensor [P, cap, 4]")
    corr = corr.contiguous()
    P, cap, dev = corr.shape[0], corr.shape[1], corr.device
    counts = counts.to(device=dev, dtype=torch.int32).contiguous()
    F = F.to(device=dev, dtype=torch.float64).reshape(P, 9).contiguous()
    cam_d = torch.as_tensor(np.ascontiguousarray(cam, np.float64).reshape(P, 8)).to(dev)
    if mask is not None:
        mask = mask.to(device=dev, dtype=torch.uint8).contiguous()
        if tuple(mask.shape) != (P, cap):
            raise ValueError("mask must be [P, cap]")
    if not (distance_thresh > 0):
        raise ValueError("distance_thresh must be positive")
    R = torch.zeros((P, 3, 3), dtype=torch.float64, device=dev)
    t = torch.zeros((P, 3), dtype=torch.float64, device=dev)
    E = torch.zeros((P, 3, 3), dtype=torch.float64, device=dev)
    ngood = torch.zeros(P, dtype=torch.int32, device=dev)
    omask = torch.zeros((P, cap), dtype=torch.uint8, device=dev)
    X = torch.zeros((P, cap, 3), dtype=torch.float32, device=dev)
    if P:
        _lib.check(
            _lib.lib().sfm_two_view_pose_batch(_lib.ptr(corr), cap, _lib.ptr(counts), P, _lib.ptr(mask), _lib.ptr(F), _lib.ptr(cam_d),
                                               float(distance_thresh), _lib.ptr(R), _lib.ptr(t), _lib.ptr(E), _lib.ptr(ngood),
                                               _lib.ptr(omask), _lib.ptr(X), _lib.current_stream_ptr(dev)),
            "sfm_two_view_pose_batch",
        )
    return PoseBatch(R, t, E, ngood, omask, X)
