"""Registration: camera poses from 2-D / 3-D correspondences, host plumbing of csrc/pnp.cu (include/sfm_b200.h, "absolute
pose / registration").

Each query is one image: RANSAC over Lambda Twist P3P samples, scored by pixel reprojection error (track triangulation's inlier
predicate), the best pose refined by Gauss-Newton on its inliers.  Cameras follow x ~ K (R X + t), so a pose drops into
``cams[image, 4:]`` of the table ``triangulate_tracks_device`` reads.  Nothing here computes or waits for the device:
``AbsolutePoses`` reads its counts back on first look.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from .tracks import Tracks
from .triangulate import TrackPoints

STATUS_NAMES = ("registered", "too_few_points", "no_model", "too_few_inliers", "invalid")
PNP_LAUNCHES = 2                # kernels register_images_device launches: the gather and the RANSAC


@dataclass
class AbsolutePoses:
    """Poses of a batch of queries on the device.  ``pose`` float64 [Q, 12] = R (row-major), t (zeros unless registered),
    ``n_inliers`` int32 [Q], ``status`` uint8 [Q] (``STATUS_NAMES`` order), ``iters`` int32 [Q] hypotheses drawn; per
    correspondence ``mask`` uint8 [Q, stride] (inliers of the final pose) and, when the correspondences were gathered from
    tracks, ``feature`` int32 [Q, stride] (the image's feature index); ``count`` int32 [Q] correspondences per query (entries
    past it are not meaningful).  The first look at ``counts`` reads the per-status counts back."""

    images: torch.Tensor
    pose: torch.Tensor
    n_inliers: torch.Tensor
    status: torch.Tensor
    iters: torch.Tensor
    mask: torch.Tensor
    count: torch.Tensor
    counts_dev: torch.Tensor                       # int64 [5], STATUS_NAMES order
    feature: torch.Tensor | None = None
    _counts: dict | None = field(default=None, repr=False)

    @property
    def counts(self) -> dict:
        """Queries per status."""
        if self._counts is None:
            self._counts = dict(zip(STATUS_NAMES, (int(v) for v in self.counts_dev.cpu().tolist())))
        return self._counts

    @property
    def R(self) -> torch.Tensor:
        return self.pose[:, :9].reshape(-1, 3, 3)

    @property
    def t(self) -> torch.Tensor:
        return self.pose[:, 9:]

    def to_host(self) -> dict:
        """numpy ``images``, ``pose``, ``R``, ``t``, ``n_inliers``, ``status``, ``iters``, ``mask``, ``count`` (and ``feature``) and
        the per-status counts."""
        keys = ("images", "pose", "R", "t", "n_inliers", "status", "iters", "mask", "count") + (("feature",) if self.feature is not None else ())
        out = {k: getattr(self, k).cpu().numpy() for k in keys}
        out.update(self.counts)
        return out


def pnp_params(*, max_error=12.0, confidence=0.9999, seed=0, max_iters=10000, min_inliers=30, min_inlier_ratio=0.25, refine_iters=10):
    """The defaults of ``max_error``, ``min_inliers`` and ``min_inlier_ratio`` are COLMAP's incremental-mapper options
    ``abs_pose_max_error``, ``abs_pose_min_num_inliers`` and ``abs_pose_min_inlier_ratio``."""
    if not 0 < float(max_error) < 1e150:
        raise ValueError(f"max_error must be positive and finite, got {max_error}")
    if int(max_iters) <= 0:
        raise ValueError(f"max_iters must be positive, got {max_iters}")
    if int(min_inliers) < 3:
        raise ValueError(f"min_inliers must be at least 3, got {min_inliers}")
    if not 0 <= float(min_inlier_ratio) <= 1:
        raise ValueError(f"min_inlier_ratio must lie in [0, 1], got {min_inlier_ratio}")
    if not 0 <= int(refine_iters) <= 1000:
        raise ValueError(f"refine_iters must lie in [0, 1000], got {refine_iters}")
    return _lib.PnpParams(float(max_error), float(confidence), int(seed), int(max_iters), int(min_inliers), float(min_inlier_ratio),
                          int(refine_iters))


def _images(images, dev) -> torch.Tensor:
    return torch.as_tensor(np.asarray(images, np.int32).reshape(-1) if not isinstance(images, torch.Tensor) else images).to(
        device=dev, dtype=torch.int32).contiguous().reshape(-1)


def _cams(cams, dev) -> torch.Tensor:
    cams = torch.as_tensor(cams).to(device=dev, dtype=torch.float64).contiguous()
    if cams.dim() != 2 or cams.shape[1] != 16 or cams.shape[0] == 0:
        raise ValueError(f"cams must be [n_images, 16] with n_images > 0, got {tuple(cams.shape)}")
    return cams


def pnp_ransac_device(xy: torch.Tensor, X: torch.Tensor, count: torch.Tensor, cams, images, *, feature=None, **params) -> AbsolutePoses:
    """One pose per query, enqueued on the current stream without a host wait.

    ``xy`` float32 [Q, stride, 2] pixel coordinates, ``X`` float64 [Q, stride, 3] world points, ``count`` int32 [Q]: query q uses its
    first ``count[q]`` rows (device tensors, used in place); ``cams`` float64 [n_images, 16] (fx fy cx cy ...; row ``images[q]`` gives
    the intrinsics of query q and its image id seeds the sampler); ``images`` int [Q].  ``params``: see ``pnp_params``."""
    prm = pnp_params(**params)
    dev = xy.device
    if xy.dtype != torch.float32 or xy.dim() != 3 or xy.shape[2] != 2 or not xy.is_cuda or not xy.is_contiguous():
        raise ValueError("xy must be a contiguous float32 CUDA tensor [Q, stride, 2]")
    Q, stride = int(xy.shape[0]), int(xy.shape[1])
    if X.dtype != torch.float64 or tuple(X.shape) != (Q, stride, 3) or X.device != dev or not X.is_contiguous():
        raise ValueError(f"X must be a contiguous float64 tensor [{Q}, {stride}, 3] on {dev}")
    if count.dtype != torch.int32 or count.numel() != Q or count.device != dev or not count.is_contiguous():
        raise ValueError(f"count must be a contiguous int32 tensor of {Q} entries on {dev}")
    if stride <= 0:
        raise ValueError("stride must be positive")
    cams = _cams(cams, dev)
    images = _images(images, dev)
    if images.numel() != Q:
        raise ValueError(f"images must have {Q} entries, got {images.numel()}")
    out = AbsolutePoses(images=images, pose=torch.empty((Q, 12), dtype=torch.float64, device=dev),
                        n_inliers=torch.empty(Q, dtype=torch.int32, device=dev), status=torch.empty(Q, dtype=torch.uint8, device=dev),
                        iters=torch.empty(Q, dtype=torch.int32, device=dev), mask=torch.empty((Q, stride), dtype=torch.uint8, device=dev),
                        count=count, counts_dev=torch.empty(len(STATUS_NAMES), dtype=torch.int64, device=dev), feature=feature)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sfm_pnp_ransac(
            int(cams.shape[0]), _lib.ptr(cams), _lib.ptr(images), Q, _lib.ptr(xy), _lib.ptr(X), stride, _lib.ptr(count), C.byref(prm),
            _lib.ptr(out.pose), _lib.ptr(out.n_inliers), _lib.ptr(out.status), _lib.ptr(out.mask), _lib.ptr(out.iters),
            _lib.ptr(out.counts_dev), _lib.current_stream_ptr(dev)), "sfm_pnp_ransac")
    return out


def _check_xy(tracks: Tracks, xy: torch.Tensor) -> int:
    n_tr, S = int(tracks.track_of_buf.shape[0]), int(tracks.track_of_buf.shape[1])
    if xy.dtype != torch.float32 or xy.dim() != 3 or xy.shape[2] != 2 or xy.device != tracks.obs_buf.device or not xy.is_contiguous():
        raise ValueError("xy must be a contiguous float32 tensor [n_images, stride, 2] on the tracks' device")
    if n_tr > xy.shape[0] or S > xy.shape[1]:
        raise ValueError(f"the tracks number {n_tr} images x {S} features; xy holds {xy.shape[0]} x {xy.shape[1]}")
    return int(xy.shape[0])


def gather_device(tracks: Tracks, points: TrackPoints, xy: torch.Tensor, images):
    """The correspondences of ``images`` (sfm_pnp_gather): per image, its features whose track has a point (``points.status ==
    0``), in feature order.  Returns ``xy`` float32 [Q, S, 2], ``X`` float64 [Q, S, 3], ``feature`` int32 [Q, S] and ``count`` int32
    [Q] on the tracks' device (S: the tracks' feature numbering), enqueued on the current stream without a host wait."""
    dev = tracks.obs_buf.device
    _check_xy(tracks, xy)
    n_tr, S = int(tracks.track_of_buf.shape[0]), int(tracks.track_of_buf.shape[1])
    images = _images(images, dev)
    Q = int(images.numel())
    g_xy = torch.empty((Q, S, 2), dtype=torch.float32, device=dev)
    g_X = torch.empty((Q, S, 3), dtype=torch.float64, device=dev)
    feature = torch.empty((Q, S), dtype=torch.int32, device=dev)
    count = torch.empty(Q, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sfm_pnp_gather(
            n_tr, S, _lib.ptr(tracks.track_of_buf), _lib.ptr(tracks.counts_dev), int(points.status_buf.numel()), _lib.ptr(points.status_buf),
            _lib.ptr(points.X_buf), _lib.ptr(xy), int(xy.shape[1]), _lib.ptr(images), Q, _lib.ptr(g_xy), _lib.ptr(g_X), _lib.ptr(feature),
            _lib.ptr(count), _lib.current_stream_ptr(dev)), "sfm_pnp_gather")
    return g_xy, g_X, feature, count


def register_images_device(tracks: Tracks, points: TrackPoints, xy: torch.Tensor, cams: torch.Tensor, images, *, update: bool = False,
                           registered: torch.Tensor | None = None, **params) -> AbsolutePoses:
    """Register ``images`` against the triangulated points of their tracks, enqueued on the current stream without a host wait.

    The correspondences of image i are its features whose track has a point (``points.status == 0``), in feature order.  ``xy``
    float32 [n_images, xy_stride, 2] (a bank's ``DescriptorBank.xy``), ``cams`` float64 [n_images, 16] (the table
    ``triangulate_tracks_device`` reads; only the intrinsics of ``images`` are read here).  With ``update=True`` the pose of every
    registered query is written into ``cams[image, 4:]`` and ``registered[image]`` (uint8 [n_images] or None) is set to 1, by
    torch index copies on the same stream, so the next ``triangulate_tracks_device`` call reads them; ``cams`` must then be a
    contiguous float64 tensor on the tracks' device.  ``params``: see ``pnp_params``."""
    dev = tracks.obs_buf.device
    n_images = _check_xy(tracks, xy)
    if update:
        if not (isinstance(cams, torch.Tensor) and cams.dtype == torch.float64 and cams.device == dev and cams.is_contiguous()):
            raise ValueError("update=True writes the poses into cams: it must be a contiguous float64 tensor on the tracks' device")
        if registered is not None and not (isinstance(registered, torch.Tensor) and registered.dtype == torch.uint8 and registered.device == dev):
            raise ValueError("update=True sets registered: it must be a uint8 tensor on the tracks' device")
        if not isinstance(images, torch.Tensor) and len(np.unique(np.asarray(images).reshape(-1))) != np.asarray(images).size:
            raise ValueError("update=True needs distinct images")
    cams_t = _cams(cams, dev)
    if int(cams_t.shape[0]) != n_images:
        raise ValueError(f"cams must be [{n_images}, 16], got {tuple(cams_t.shape)}")
    images = _images(images, dev)
    Q = int(images.numel())
    g_xy, g_X, feature, count = gather_device(tracks, points, xy, images)
    with torch.cuda.device(dev):
        out = pnp_ransac_device(g_xy, g_X, count, cams_t, images, feature=feature, **params)
        if update and Q:
            ok = out.status == 0
            # queries that did not register write into a spare row n_images, so repeated or invalid images never collide
            tgt = torch.where(ok, images.long().clamp(0, n_images - 1), torch.full_like(images, n_images, dtype=torch.int64))
            rows = torch.cat([cams_t[:, 4:], cams_t.new_zeros((1, 12))])
            rows.index_copy_(0, tgt, out.pose)
            cams_t[:, 4:] = rows[:n_images]
            if registered is not None:
                flags = torch.cat([registered.reshape(-1), registered.new_zeros(1)])
                flags.index_fill_(0, tgt, 1)
                registered.reshape(-1).copy_(flags[:n_images])
    return out
