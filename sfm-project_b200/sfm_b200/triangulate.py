"""Robust multi-view triangulation of feature tracks from known cameras: host plumbing of csrc/triangulate.cu
(include/sfm_b200.h, "track triangulation").

Every track becomes one 3-D point in world coordinates: two-view DLT hypotheses sampled RANSAC-style, scored by pixel
reprojection error in every registered view, the best refit by an N-view DLT over its inliers.  Cameras follow
x ~ K (R X + t).  Nothing here computes or waits for the device: the track count is read by the kernel, the outputs are
sized for the worst case, and ``TrackPoints`` reads its counts back on first look.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from .tracks import Tracks

STATUS_NAMES = ("triangulated", "too_few_views", "no_model", "too_few_inliers", "invalid")
TRIANGULATE_LAUNCHES = 1        # kernels sfm_triangulate_tracks launches


@dataclass
class TrackPoints:
    """Points of a ``Tracks`` on the device.  ``X`` float64 [T,3] (zeros unless triangulated), ``n_inliers`` int32 [T],
    ``status`` uint8 [T] (``STATUS_NAMES`` order); per observation of ``tracks.obs``: ``obs_inlier`` uint8 and ``obs_error``
    float32 (pixel reprojection error of the track's point, +inf behind the camera, NaN in unregistered images and for tracks
    without a point).  The first look at a count or a view reads the tracks' and the statuses' counts back and trims the
    worst-case buffers."""

    tracks: Tracks
    X_buf: torch.Tensor
    n_inliers_buf: torch.Tensor
    status_buf: torch.Tensor
    obs_inlier_buf: torch.Tensor
    obs_error_buf: torch.Tensor
    counts_dev: torch.Tensor                       # int64 [5], STATUS_NAMES order
    _counts: dict | None = field(default=None, repr=False)

    @property
    def counts(self) -> dict:
        """Tracks per status."""
        if self._counts is None:
            self._counts = dict(zip(STATUS_NAMES, (int(v) for v in self.counts_dev.cpu().tolist())))
        return self._counts

    @property
    def n_tracks(self) -> int:
        return self.tracks.n_tracks

    @property
    def X(self) -> torch.Tensor:
        return self.X_buf[: self.n_tracks]

    @property
    def n_inliers(self) -> torch.Tensor:
        return self.n_inliers_buf[: self.n_tracks]

    @property
    def status(self) -> torch.Tensor:
        return self.status_buf[: self.n_tracks]

    @property
    def obs_inlier(self) -> torch.Tensor:
        return self.obs_inlier_buf[: self.tracks.n_obs]

    @property
    def obs_error(self) -> torch.Tensor:
        return self.obs_error_buf[: self.tracks.n_obs]

    def to_host(self) -> dict:
        """numpy ``X``, ``n_inliers``, ``status``, ``obs_inlier``, ``obs_error`` and the per-status counts."""
        out = {k: getattr(self, k).cpu().numpy() for k in ("X", "n_inliers", "status", "obs_inlier", "obs_error")}
        out.update(self.counts)
        return out


def triangulate_params(*, max_error=4.0, min_angle=1.5, max_iters=500, confidence=0.999, seed=0, min_inliers=2):
    if not float(max_error) > 0:
        raise ValueError(f"max_error must be positive, got {max_error}")
    if not 0 <= float(min_angle) < 90:
        raise ValueError(f"min_angle must lie in [0, 90) degrees, got {min_angle}")
    if int(max_iters) <= 0:
        raise ValueError(f"max_iters must be positive, got {max_iters}")
    if int(min_inliers) < 2:
        raise ValueError(f"min_inliers must be at least 2, got {min_inliers}")
    return _lib.TriangulateParams(float(max_error), float(min_angle), float(confidence), int(seed), int(max_iters), int(min_inliers))


def triangulate_tracks_device(tracks: Tracks, xy: torch.Tensor, cams: torch.Tensor, registered=None, *, S: int | None = None,
                              **params) -> TrackPoints:
    """Triangulate every track of ``tracks`` on its device, enqueued on the current stream without a host wait.

    ``xy`` float32 [n_images, xy_stride, 2] (a bank's ``DescriptorBank.xy``, used in place), ``cams`` float64 [n_images, 16] =
    fx fy cx cy, R (row-major), t (x ~ K (R X + t)), ``registered`` uint8 [n_images] or None (all registered) -- device tensors of
    these dtypes are used in place.  ``S`` is the feature numbering of the tracks (default ``xy_stride``): an observation with a
    feature outside [0, S) or an image outside [0, n_images) marks its track invalid.  ``params``: see ``triangulate_params``."""
    dev = tracks.obs_buf.device
    prm = triangulate_params(**params)
    if xy.dtype != torch.float32 or xy.dim() != 3 or xy.shape[2] != 2 or xy.device != dev or not xy.is_contiguous():
        raise ValueError("xy must be a contiguous float32 tensor [n_images, stride, 2] on the tracks' device")
    n_images, stride = int(xy.shape[0]), int(xy.shape[1])
    cams = torch.as_tensor(cams).to(device=dev, dtype=torch.float64).contiguous()
    if tuple(cams.shape) != (n_images, 16):
        raise ValueError(f"cams must be [{n_images}, 16], got {tuple(cams.shape)}")
    if registered is not None:
        registered = torch.as_tensor(registered).to(device=dev, dtype=torch.uint8).contiguous().reshape(-1)
        if registered.numel() != n_images:
            raise ValueError(f"registered must have {n_images} entries, got {registered.numel()}")
    max_tracks, max_obs = int(tracks.offsets_buf.numel()) - 1, int(tracks.obs_buf.shape[0])
    p = TrackPoints(tracks=tracks,
                    X_buf=torch.empty((max_tracks, 3), dtype=torch.float64, device=dev),
                    n_inliers_buf=torch.empty(max_tracks, dtype=torch.int32, device=dev),
                    status_buf=torch.empty(max_tracks, dtype=torch.uint8, device=dev),
                    obs_inlier_buf=torch.empty(max_obs, dtype=torch.uint8, device=dev),
                    obs_error_buf=torch.empty(max_obs, dtype=torch.float32, device=dev),
                    counts_dev=torch.empty(len(STATUS_NAMES), dtype=torch.int64, device=dev))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sfm_triangulate_tracks(
            n_images, stride if S is None else int(S), _lib.ptr(tracks.offsets_buf), _lib.ptr(tracks.obs_buf), _lib.ptr(tracks.counts_dev),
            max_tracks, _lib.ptr(xy), stride, _lib.ptr(cams), _lib.ptr(registered), C.byref(prm), _lib.ptr(p.X_buf),
            _lib.ptr(p.n_inliers_buf), _lib.ptr(p.status_buf), _lib.ptr(p.obs_inlier_buf), _lib.ptr(p.obs_error_buf),
            _lib.ptr(p.counts_dev), _lib.current_stream_ptr(dev)), "sfm_triangulate_tracks")
    return p


def camera_table(K, R, t) -> np.ndarray:
    """float64 [n, 16] rows (fx fy cx cy, R row-major, t) from pinhole ``K`` (one [3,3] or [n,3,3]), ``R`` [n,3,3], ``t`` [n,3]."""
    from .ransac import camera_rows

    R = np.asarray(R, np.float64)
    t = np.asarray(t, np.float64)
    if R.ndim != 3 or R.shape[1:] != (3, 3):
        raise ValueError(f"R must be [n,3,3], got {R.shape}")
    n = R.shape[0]
    t = t.reshape(n, 3) if t.size == 3 * n else t
    if t.shape != (n, 3):
        raise ValueError(f"t must be [{n},3], got {t.shape}")
    Kf = np.asarray(K, np.float64)
    if Kf.shape[-2:] != (3, 3) or Kf.ndim not in (2, 3) or (Kf.ndim == 3 and Kf.shape[0] != n):
        raise ValueError(f"K must be [3,3] or [{n},3,3], got {Kf.shape}")
    if np.any(Kf[..., 1, 0] != 0) or np.any(Kf[..., 2, :] != np.array([0.0, 0.0, 1.0])):
        raise ValueError("camera matrices must be pinhole: K[1,0] == 0 and last row (0, 0, 1)")
    four = camera_rows(Kf, None, n)[:, :4]              # (rejects skew)
    if np.any(four[:, :2] == 0) or not np.all(np.isfinite(four)):
        raise ValueError("focal lengths must be non-zero and finite")
    return np.ascontiguousarray(np.concatenate([four, R.reshape(n, 9), t], axis=1))
