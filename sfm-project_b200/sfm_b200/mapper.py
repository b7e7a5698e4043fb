"""Incremental reconstruction on the device: host plumbing of csrc/mapper.cu (include/sfm_b200.h, "incremental
reconstruction") and the loop that joins it to registration, triangulation and bundle adjustment.

``next_images_device`` picks the next images to register (COLMAP's visibility-pyramid next-best-view score),
``filter_points_device`` drops the observations and points a bundle adjustment leaves bad, and ``reconstruct_device``
runs COLMAP's incremental mapper from the verified pairs: an initial pair, then rounds of selection, registration,
triangulation, bundle adjustment and filtering until no image can be added.  Every stage's data stays on the device; the
host reads two numbers per round to decide whether to go on.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from .bundle import MAX_IMAGES, BundleResult, bundle_adjust_device, bundle_launches, workspace_bytes
from .pnp import PNP_LAUNCHES, register_images_device
from .tracks import Tracks
from .triangulate import TRIANGULATE_LAUNCHES, TrackPoints, camera_table, triangulate_tracks_device

NEXT_IMAGES_LAUNCHES = 2        # kernels sfm_next_images launches: the score, then the selection
FILTER_LAUNCHES = 1             # kernels sfm_filter_points launches


def round_launches(bundle_max_iters: int = 50) -> int:
    """Kernels of one ``reconstruct_device`` round that registers an image: selection, registration, triangulation, bundle
    adjustment and the filter.  A round that registers nothing stops after registration (NEXT_IMAGES_LAUNCHES + PNP_LAUNCHES)."""
    return NEXT_IMAGES_LAUNCHES + PNP_LAUNCHES + TRIANGULATE_LAUNCHES + bundle_launches(bundle_max_iters) + FILTER_LAUNCHES


@dataclass
class NextImages:
    """``images`` int32 [max_select] (the selection, best first, -1 padded), ``n_selected`` int32 [1], ``visible`` int32
    [n_images], ``score`` int64 [n_images] -- device tensors."""

    images: torch.Tensor
    n_selected: torch.Tensor
    visible: torch.Tensor
    score: torch.Tensor

    def to_host(self) -> dict:
        out = {k: getattr(self, k).cpu().numpy() for k in ("images", "visible", "score")}
        out["n_selected"] = int(self.n_selected.cpu()[0])
        return out


def next_images_params(*, max_select=16, min_visible=30, max_trials=3, levels=6):
    if int(max_select) < 1:
        raise ValueError(f"max_select must be positive, got {max_select}")
    if int(min_visible) < 0:
        raise ValueError(f"min_visible must be non-negative, got {min_visible}")
    if int(max_trials) < 1:
        raise ValueError(f"max_trials must be positive, got {max_trials}")
    if not 1 <= int(levels) <= 8:
        raise ValueError(f"levels must lie in [1, 8], got {levels}")
    return _lib.NextImagesParams(int(min_visible), int(max_trials), int(max_select), int(levels))


def filter_params(*, max_error=4.0, min_angle=1.5, min_inliers=2):
    """The defaults are COLMAP's incremental-mapper options ``filter_max_reproj_error`` and ``filter_min_tri_angle``."""
    if not 0 <= float(max_error) < 1e150:
        raise ValueError(f"max_error must be non-negative and finite, got {max_error}")
    if not 0 <= float(min_angle) < 90:
        raise ValueError(f"min_angle must lie in [0, 90) degrees, got {min_angle}")
    if int(min_inliers) < 2:
        raise ValueError(f"min_inliers must be at least 2, got {min_inliers}")
    return _lib.FilterPointsParams(float(max_error), float(min_angle), int(min_inliers))


def image_sizes(cams) -> torch.Tensor:
    """int32 [n, 2] = (round(2 cx), round(2 cy)) of a camera table: the image size when the principal point is its centre."""
    cams = torch.as_tensor(cams)
    return torch.round(2.0 * cams[:, 2:4].to(torch.float64)).to(torch.int32).contiguous()


def _u8(t, n, dev, name):
    if not (isinstance(t, torch.Tensor) and t.dtype == torch.uint8 and t.device == dev and t.is_contiguous() and t.numel() == n):
        raise ValueError(f"{name} must be a contiguous uint8 tensor of {n} entries on {dev}")
    return t


def next_images_device(tracks: Tracks, points: TrackPoints, xy: torch.Tensor, registered: torch.Tensor, trials: torch.Tensor, *,
                       image_size=None, cams=None, **params) -> NextImages:
    """Score every image of the tracks by the visibility pyramid of its visible points (features whose track has a point) and
    select the next ones to register, enqueued on the current stream without a host wait.

    n_images is the tracks' image count (``track_of`` rows, at most 1024); ``xy`` float32 [>= n_images, xy_stride, 2];
    ``registered`` uint8 [n_images] and ``trials`` int32 [n_images] are device tensors, ``trials`` is incremented in place for
    every selected image.  ``image_size`` int [n_images, 2] = (w, h), default ``image_sizes(cams)``.  ``params``: see
    ``next_images_params``."""
    dev = tracks.obs_buf.device
    prm = next_images_params(**params)
    n_images, S = int(tracks.track_of_buf.shape[0]), int(tracks.track_of_buf.shape[1])
    if not 0 < n_images <= MAX_IMAGES:
        raise ValueError(f"next-image selection takes 1 to {MAX_IMAGES} images, got {n_images}")
    if xy.dtype != torch.float32 or xy.dim() != 3 or xy.shape[2] != 2 or xy.device != dev or not xy.is_contiguous():
        raise ValueError("xy must be a contiguous float32 tensor [n_images, stride, 2] on the tracks' device")
    if xy.shape[0] < n_images or xy.shape[1] < S:
        raise ValueError(f"the tracks number {n_images} images x {S} features; xy holds {xy.shape[0]} x {xy.shape[1]}")
    _u8(registered, n_images, dev, "registered")
    if not (isinstance(trials, torch.Tensor) and trials.dtype == torch.int32 and trials.device == dev and trials.is_contiguous()
            and trials.numel() == n_images):
        raise ValueError(f"trials must be a contiguous int32 tensor of {n_images} entries on {dev}")
    if image_size is None:
        if cams is None:
            raise ValueError("pass image_size or cams")
        image_size = image_sizes(cams)[:n_images]
    size = torch.as_tensor(image_size).to(device=dev, dtype=torch.int32).reshape(-1, 2).contiguous()
    if size.shape[0] != n_images:
        raise ValueError(f"image_size must be [{n_images}, 2], got {tuple(size.shape)}")
    out = NextImages(images=torch.empty(prm.max_select, dtype=torch.int32, device=dev), n_selected=torch.empty(1, dtype=torch.int32, device=dev),
                     visible=torch.empty(n_images, dtype=torch.int32, device=dev), score=torch.empty(n_images, dtype=torch.int64, device=dev))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sfm_next_images(
            n_images, S, _lib.ptr(tracks.track_of_buf), _lib.ptr(tracks.counts_dev), int(points.status_buf.numel()), _lib.ptr(points.status_buf),
            _lib.ptr(xy), int(xy.shape[1]), _lib.ptr(size), _lib.ptr(registered), _lib.ptr(trials), C.byref(prm), _lib.ptr(out.images),
            _lib.ptr(out.n_selected), _lib.ptr(out.visible), _lib.ptr(out.score), _lib.current_stream_ptr(dev)), "sfm_next_images")
    return out


def filter_points_device(points: TrackPoints, cams: torch.Tensor, registered: torch.Tensor, **params) -> TrackPoints:
    """Filter ``points`` in place after a bundle adjustment (COLMAP's FilterPoints), enqueued on the current stream without a
    host wait: an observation of a triangulated track stays an inlier iff its image is registered and its ``obs_error`` is at
    most ``max_error``; a track left with fewer than ``min_inliers`` gets status 3, one whose remaining views meet at no angle
    of ``min_angle`` or more status 2 (X zeroed, flags cleared).  ``cams`` float64 [n_images, 16] and ``registered`` uint8
    [n_images] are device tensors.  The per-status counts are replaced by the filtered ones.  Returns ``points``."""
    tracks = points.tracks
    dev = tracks.obs_buf.device
    prm = filter_params(**params)
    if not (isinstance(cams, torch.Tensor) and cams.dtype == torch.float64 and cams.device == dev and cams.is_contiguous()
            and cams.dim() == 2 and cams.shape[1] == 16):
        raise ValueError("cams must be a contiguous float64 tensor [n_images, 16] on the tracks' device")
    n_images = int(cams.shape[0])
    _u8(registered, n_images, dev, "registered")
    counts = torch.empty(5, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sfm_filter_points(
            n_images, _lib.ptr(tracks.offsets_buf), _lib.ptr(tracks.obs_buf), _lib.ptr(tracks.counts_dev), int(points.status_buf.numel()),
            _lib.ptr(cams), _lib.ptr(registered), _lib.ptr(points.obs_error_buf), C.byref(prm), _lib.ptr(points.X_buf),
            _lib.ptr(points.n_inliers_buf), _lib.ptr(points.status_buf), _lib.ptr(points.obs_inlier_buf), _lib.ptr(counts),
            _lib.current_stream_ptr(dev)), "sfm_filter_points")
    points.counts_dev = counts
    points._counts = None
    return points


def initial_pair_order(n_pose, n_inliers, n_inliers_h=None, *, min_inliers=100, max_h_ratio=0.8) -> np.ndarray:
    """Indices of the pairs that may start a reconstruction, best first: ``n_pose >= min_inliers`` and, when the homography
    stage ran, ``n_inliers_h <= max_h_ratio * n_inliers`` (not planar or a pure rotation); ordered by ``n_pose`` descending, then
    pair index ascending."""
    n_pose = np.asarray(n_pose, np.int64).reshape(-1)
    ok = n_pose >= int(min_inliers)
    if n_inliers_h is not None:
        ok &= np.asarray(n_inliers_h, np.float64).reshape(-1) <= float(max_h_ratio) * np.asarray(n_inliers, np.float64).reshape(-1)
    idx = np.nonzero(ok)[0]
    return idx[np.lexsort((idx, -n_pose[idx]))]


def _median_angle(X, R, t) -> float:
    """Median triangulation angle (degrees) of points X seen by [I|0] and [R|t]."""
    if len(X) == 0:
        return 0.0
    Cb = -R.T @ t
    da, db = X, X - Cb
    c = np.sum(da * db, 1) / np.sqrt(np.sum(da * da, 1) * np.sum(db * db, 1))
    return float(np.median(np.degrees(np.arccos(np.clip(c, -1.0, 1.0)))))


@dataclass
class Reconstruction:
    """The result of ``reconstruct_device``.  ``cams`` float64 [n_images, 16] and ``registered`` uint8 [n_images] on the device;
    ``round`` int32 [n_images] (numpy): the round that registered each image (0 for the initial pair, -1 if never);
    ``init_pair`` (i, j) or None; ``points`` the filtered ``TrackPoints``; ``bundle`` the last ``BundleResult``; ``rounds`` one
    dict per round (``round``, ``selected``, ``registered``, ``ba_status``, ``ba_iterations``, ``initial_cost``,
    ``final_cost``, ``filtered_obs``, ``points``); ``status`` "ok" or "no_initial_pair"."""

    cams: torch.Tensor
    registered: torch.Tensor
    round: np.ndarray
    init_pair: tuple | None
    points: TrackPoints | None
    bundle: BundleResult | None
    rounds: list = field(default_factory=list)
    status: str = "ok"

    def to_host(self) -> dict:
        """numpy ``R`` [n,3,3], ``t`` [n,3], ``registered``, ``round``, ``X`` [T,3], ``point_status`` [T], ``obs_inlier``,
        ``obs_error`` [n_obs], and ``init_pair``, ``status``, ``rounds``."""
        cams = self.cams.cpu().numpy()
        out = {"R": cams[:, 4:13].reshape(-1, 3, 3).copy(), "t": cams[:, 13:].copy(), "registered": self.registered.cpu().numpy(),
               "round": self.round.copy(), "init_pair": self.init_pair, "status": self.status, "rounds": list(self.rounds)}
        if self.points is not None:
            h = self.points.to_host()
            out.update(X=h["X"], point_status=h["status"], obs_inlier=h["obs_inlier"], obs_error=h["obs_error"])
        return out


def reconstruct_device(result, xy: torch.Tensor, K, *, init_pair=None, max_per_round=16, max_trials=3, min_visible=30,
                       init_min_inliers=100, init_min_angle=16.0, init_max_h_ratio=0.8, init_max_trials=10, triangulate=None, pnp=None,
                       bundle=None, filter=None, seed=0) -> Reconstruction:
    """Incremental reconstruction (COLMAP's incremental mapper) of a ``VerifiedPairs`` that has the two-view pose stage
    (``match_and_verify(..., intrinsics=K)``) and ``tracks`` (``tracks=True``); ``homography=True`` adds the initial pair's
    planarity test.  ``xy`` float32 [n_images, stride, 2] (the bank's ``DescriptorBank.xy``), ``K`` one pinhole [3,3] or
    [n_images,3,3].  At most 1024 images.

    1. Initial pair: the candidates of ``initial_pair_order`` are tried in turn (at most ``init_max_trials``): camera i at
       [I|0], camera j at the pair's (R, t), only i and j registered, the tracks triangulated; the first with at least
       ``init_min_inliers`` points whose median triangulation angle is at least ``init_min_angle`` degrees is taken (an explicit
       ``init_pair`` skips the search).  Then bundle adjustment with camera i fixed, then the point filter.
    2. Rounds: ``next_images_device`` (``max_select = max_per_round``), registration of its selection straight from the device,
       one host read of (selected, registered); stop when nothing was selected, go on when nothing registered, else triangulate
       every track from the registered cameras, bundle-adjust with camera i fixed and filter.  A round that registers launches
       ``round_launches(bundle max_iters)`` kernels.  Every selection increments its images' trials, so there are at most
       n_images * max_trials rounds.
    ``triangulate``, ``pnp``, ``bundle`` and ``filter`` are the keyword parameters of each stage; ``seed`` seeds triangulation and
    registration unless they name their own."""
    triangulate, pnp, bundle, filter = dict(triangulate or {}), dict(pnp or {}), dict(bundle or {}), dict(filter or {})
    triangulate.setdefault("seed", seed)
    pnp.setdefault("seed", seed)
    tracks = getattr(result, "tracks", None)
    if tracks is None:
        raise ValueError("reconstruct_device needs the result's tracks: match_and_verify(..., tracks=True)")
    if getattr(result, "n_pose", None) is None or result.R is None or result.t is None:
        raise ValueError("reconstruct_device needs the two-view pose stage: match_and_verify(..., intrinsics=K)")
    dev = tracks.obs_buf.device
    if xy.dtype != torch.float32 or xy.dim() != 3 or xy.shape[2] != 2 or xy.device != dev or not xy.is_contiguous():
        raise ValueError("xy must be a contiguous float32 tensor [n_images, stride, 2] on the tracks' device")
    n_images = int(xy.shape[0])
    n_tr, S = int(tracks.track_of_buf.shape[0]), int(tracks.track_of_buf.shape[1])
    if not 0 < n_images <= MAX_IMAGES or n_tr > n_images:
        raise ValueError(f"reconstruction takes 1 to {MAX_IMAGES} images and xy rows for every tracked image, got {n_images} rows "
                         f"for {n_tr} tracked images")
    base = camera_table(K, np.tile(np.eye(3), (n_images, 1, 1)), np.zeros((n_images, 3)))
    size = image_sizes(torch.from_numpy(base[:n_tr])).to(dev)
    pairs = result.pairs.cpu().numpy()
    Rp, tp = result.R.cpu().numpy(), result.t.cpu().numpy()
    n_pose = result.n_pose.cpu().numpy()
    n_inl = result.n_inliers.cpu().numpy()
    n_h = None if getattr(result, "n_inliers_h", None) is None else result.n_inliers_h.cpu().numpy()
    n_tracks = tracks.n_tracks                                     # (the tracks' one host read)

    def start(p):
        i, j = int(pairs[p, 0]), int(pairs[p, 1])
        cams = torch.from_numpy(base.copy()).to(dev)
        cams[j, 4:13] = torch.from_numpy(Rp[p].reshape(9)).to(dev)
        cams[j, 13:] = torch.from_numpy(tp[p]).to(dev)
        reg = torch.zeros(n_images, dtype=torch.uint8, device=dev)
        reg[[i, j]] = 1
        return i, j, cams, reg, triangulate_tracks_device(tracks, xy, cams, reg, S=S, **triangulate)

    chosen = None
    if init_pair is not None:
        a, b = (int(v) for v in init_pair)
        hit = np.nonzero((pairs[:, 0] == a) & (pairs[:, 1] == b))[0]
        if len(hit) == 0:
            hit = np.nonzero((pairs[:, 0] == b) & (pairs[:, 1] == a))[0]
        if len(hit) == 0 or a == b:
            raise ValueError(f"init_pair {tuple(init_pair)} is not a pair of the result")
        chosen = start(int(hit[0]))
    else:
        for p in initial_pair_order(n_pose, n_inl, n_h, min_inliers=init_min_inliers, max_h_ratio=init_max_h_ratio)[: int(init_max_trials)]:
            if pairs[p, 0] == pairs[p, 1]:
                continue
            cand = start(int(p))
            st = cand[4].status.cpu().numpy()
            X = cand[4].X.cpu().numpy()[st == 0]
            if len(X) >= init_min_inliers and _median_angle(X, Rp[p], tp[p]) >= init_min_angle:
                chosen = cand
                break
    if chosen is None:
        return Reconstruction(cams=torch.from_numpy(base).to(dev), registered=torch.zeros(n_images, dtype=torch.uint8, device=dev),
                              round=np.full(n_images, -1, np.int32), init_pair=None, points=None, bundle=None, status="no_initial_pair")
    i, j, cams, reg, pts = chosen
    fixed = torch.zeros(n_images, dtype=torch.uint8, device=dev)
    fixed[i] = 1
    max_tracks, max_obs = int(tracks.offsets_buf.numel()) - 1, int(tracks.obs_buf.shape[0])
    ws = torch.empty(workspace_bytes(n_images, max_tracks, max_obs), dtype=torch.uint8, device=dev)
    trials = torch.zeros(n_tr, dtype=torch.int32, device=dev)
    pending = []                                                   # per round: device tensors read once at the end

    def adjust(pts):
        ba = bundle_adjust_device(tracks, pts, xy, cams, reg, fixed=fixed, update=True, S=S, workspace=ws, **bundle)
        before = pts.obs_inlier.sum(dtype=torch.int64)
        filter_points_device(pts, cams, reg, **filter)
        return ba, before - pts.obs_inlier.sum(dtype=torch.int64)

    ba, filtered = adjust(pts)
    pending.append((0, torch.tensor([i, j], dtype=torch.int32, device=dev), torch.zeros(2, dtype=torch.uint8, device=dev), ba, filtered,
                    pts.counts_dev))
    r = 0
    while True:
        r += 1
        nxt = next_images_device(tracks, pts, xy, reg[:n_tr], trials, image_size=size, max_select=max_per_round, min_visible=min_visible,
                                 max_trials=max_trials)
        out = register_images_device(tracks, pts, xy, cams, nxt.images, update=True, registered=reg, **pnp)
        n_sel, n_reg = torch.stack([nxt.n_selected[0].to(torch.int64), out.counts_dev[0]]).cpu().tolist()
        if n_sel == 0:
            break
        if n_reg == 0:
            pending.append((r, nxt.images[:n_sel], out.status[:n_sel], None, None, None))
            continue
        pts = triangulate_tracks_device(tracks, xy, cams, reg, S=S, **triangulate)
        ba, filtered = adjust(pts)
        pending.append((r, nxt.images[:n_sel], out.status[:n_sel], ba, filtered, pts.counts_dev))

    rnd = np.full(n_images, -1, np.int32)
    rounds = []
    for k, images, status, ba_k, filt, counts in pending:
        images, status = images.cpu().numpy(), status.cpu().numpy()
        got = images if k == 0 else images[status == 0]
        rnd[got] = k
        e = {"round": k, "selected": images.tolist(), "registered": got.tolist()}
        if ba_k is not None:
            s = ba_k.summary
            e.update(ba_status=s["status"], ba_iterations=int(s["iterations"]), initial_cost=float(s["initial_cost"]),
                     final_cost=float(s["final_cost"]), filtered_obs=int(filt.cpu()), points=int(counts[0].cpu()))
        rounds.append(e)
    return Reconstruction(cams=cams, registered=reg, round=rnd, init_pair=(i, j), points=pts, bundle=ba, rounds=rounds)
