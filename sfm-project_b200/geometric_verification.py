"""Geometric verification: the module the reference left empty.

``code/geometric_verification.py`` is a 0-byte file that ``code/pipeline.py:3`` star-imports, and the
"Geometric Verification" section of ``main()`` is a bare comment (code/pipeline.py:60-65).  This module
defines the API (SURVEY.md §8b) with the conventions of ``cv2.findFundamentalMat(pts1, pts2,
cv2.FM_RANSAC, thr, confidence, maxIters)`` so that cv2 is a one-line oracle: F is float64 [3,3] with
``x2^T F x1 = 0`` and ``F[2,2] == 1``, the mask is uint8 [M,1], and ``(None, zeros)`` is returned when no
model is found.  All computation is the batched CUDA kernel csrc/ransac_f.cu; there is no CPU fallback.
"""
import numpy as np
import torch

import sfm_b200 as _sfm
from sfm_b200.ransac import h_stop_target


def _as_points(pts, name):
    a = np.asarray(pts)
    if a.size == 0:
        return np.zeros((0, 2), np.float32)
    if a.ndim == 3 and a.shape[1] == 1:
        a = a[:, 0, :]
    if a.ndim != 2 or a.shape[1] != 2:
        raise ValueError(f"{name} must be [M,2] or [M,1,2], got {a.shape}")
    if a.dtype not in (np.float32, np.float64):
        raise ValueError(f"{name} must be float32 or float64")
    return np.ascontiguousarray(a, np.float32)


def verify_pairs(points1, points2, *, thr=3.0, confidence=0.99, max_iters=2000, solver="7pt", score="sym_epipolar",
                 lo=False, seed=0, min_inliers=0):
    """Batched verification.  ``points1[k]``, ``points2[k]`` are the [M_k,2] matched pixel coordinates of pair k.
    Returns a list of ``(F or None, mask uint8 [M_k,1])``."""
    if len(points1) == len(points2) == 0:
        return []
    corr, counts_t, counts = _corr_batch(points1, points2)
    vb = _sfm.verify_corr(corr, counts_t, thr=thr, confidence=confidence, max_iters=max_iters, solver=solver, score=score, lo=lo,
                          seed=seed, min_inliers=min_inliers)
    F, ninl, mask = vb.F.cpu().numpy(), vb.n_inliers.cpu().numpy(), vb.mask.cpu().numpy()
    return [(F[k].copy() if ninl[k] > 0 else None, mask[k, : counts[k]].reshape(-1, 1).copy()) for k in range(len(counts))]


def verify_pair(pts1, pts2, *, thr=3.0, confidence=0.99, max_iters=2000, solver="7pt", score="sym_epipolar", lo=False,
                seed=0):
    """Single-pair form of cv2.findFundamentalMat(FM_RANSAC): returns ``(F float64[3,3] | None, mask uint8[M,1])``."""
    return verify_pairs([pts1], [pts2], thr=thr, confidence=confidence, max_iters=max_iters, solver=solver, score=score,
                        lo=lo, seed=seed)[0]


def verify_matches(kp1, kp2, matches, **kw):
    """Verify a ``list[cv2.DMatch]`` (as returned by ``extract_and_match``) between two keypoint lists.
    Returns ``(F or None, inlier_matches)``."""
    if not matches:
        return None, []
    pts1 = np.array([kp1[m.queryIdx].pt for m in matches], np.float32)
    pts2 = np.array([kp2[m.trainIdx].pt for m in matches], np.float32)
    F, mask = verify_pair(pts1, pts2, **kw)
    if F is None:
        return None, []
    return F, [m for m, keep in zip(matches, mask.ravel()) if keep]


# ------------------------------------------------------------------ homography model (SURVEY.md §8f rank 2)
def _corr_batch(points1, points2):
    if len(points1) != len(points2):
        raise ValueError("points1 and points2 must have the same number of pairs")
    p1 = [_as_points(p, "pts1") for p in points1]
    p2 = [_as_points(p, "pts2") for p in points2]
    for a, b in zip(p1, p2):
        if len(a) != len(b):
            raise ValueError("pts1 and pts2 must have the same number of points")
    cap = max(16, max(len(a) for a in p1))
    corr = np.zeros((len(p1), cap, 4), np.float32)
    counts = np.zeros(len(p1), np.int32)
    for k, (a, b) in enumerate(zip(p1, p2)):
        corr[k, : len(a), :2], corr[k, : len(a), 2:] = a, b
        counts[k] = len(a)
    return torch.from_numpy(corr).cuda(), torch.from_numpy(counts), counts


def find_homographies(points1, points2, *, thr=3.0, confidence=0.995, max_iters=2000, lo=False, seed=0, min_inliers=0,
                      stop_targets=None):
    """Batched ``cv2.findHomography(pts1, pts2, cv2.RANSAC, thr)``: a list of ``(H float64[3,3] | None, mask uint8[M_k,1])``
    with ``x2 ~ H x1`` and ``H[2,2] == 1`` (csrc/ransac_h.cu, one CTA per pair).  ``stop_targets[k]`` (optional) is the
    inlier count the caller cares about for pair k: sampling stops once a homography with that support would have been
    found, so a pair that no homography explains costs 32 hypotheses instead of ``max_iters``."""
    if len(points1) == 0:
        return []
    corr, counts_t, counts = _corr_batch(points1, points2)
    vb = _sfm.ransac.verify_h_corr(corr, counts_t, thr=thr, confidence=confidence, max_iters=max_iters, lo=lo, seed=seed,
                                   min_inliers=min_inliers,
                                   stop_target=None if stop_targets is None else np.asarray(stop_targets, np.int32).reshape(len(counts)))
    H, ninl, mask = vb.F.cpu().numpy(), vb.n_inliers.cpu().numpy(), vb.mask.cpu().numpy()
    return [(H[k].copy() if ninl[k] > 0 else None, mask[k, : counts[k]].reshape(-1, 1).copy()) for k in range(len(counts))]


def find_homography(pts1, pts2, *, stop_target=None, **kw):
    """Single-pair form: ``(H | None, mask uint8[M,1])``."""
    return find_homographies([pts1], [pts2], stop_targets=None if stop_target is None else [stop_target], **kw)[0]


# ------------------------------------------------------------------ two-view initialisation (SURVEY.md §8f rank 4)
def recover_poses(Fs, points1, points2, K1, K2=None, *, masks=None, distance_thresh=50.0):
    """Batched ``cv2.recoverPose`` starting from F: ``E = K2^T F K1``, the (R, t) among the four decompositions with
    the most correspondences in front of both cameras, and their DLT triangulation (csrc/pose.cu).  ``K1`` / ``K2``
    are 3x3 pinhole matrices (shared) or ``[P,3,3]`` stacks (``K2=None``: same camera).  Returns a list of
    ``(n_good, R float64[3,3], t float64[3], mask uint8[M_k,1], points3d float32[M_k,3])``; points are expressed in
    the first camera's frame and are zero where the mask is 0; ``n_good == 0`` means no pose."""
    P = len(points1)
    if P == 0:
        return []
    corr, counts_t, counts = _corr_batch(points1, points2)
    F = np.zeros((P, 3, 3), np.float64)
    for k, f in enumerate(Fs):
        if f is not None:
            f = np.asarray(f, np.float64)
            if f.shape != (3, 3):
                raise ValueError(f"F must be [3,3], got {f.shape}")
            F[k] = f
    m = None
    if masks is not None:
        m = torch.zeros((P, corr.shape[1]), dtype=torch.uint8)
        for k, mk in enumerate(masks):
            mk = np.asarray(mk).reshape(-1)
            if len(mk) != counts[k]:
                raise ValueError("mask length must equal the number of points of its pair")
            m[k, : counts[k]] = torch.from_numpy((mk != 0).astype(np.uint8))
    cam = _sfm.ransac.camera_rows(K1, K2, P)
    pb = _sfm.ransac.recover_pose_corr(corr, counts_t, torch.from_numpy(F), cam, mask=m, distance_thresh=distance_thresh)
    R, t, ng = pb.R.cpu().numpy(), pb.t.cpu().numpy(), pb.n_good.cpu().numpy()
    pm, X = pb.mask.cpu().numpy(), pb.points.cpu().numpy()
    return [(int(ng[k]), R[k].copy(), t[k].copy(), pm[k, : counts[k]].reshape(-1, 1).copy(), X[k, : counts[k]].copy()) for k in range(P)]


def recover_pose(F, pts1, pts2, K1, K2=None, *, mask=None, distance_thresh=50.0):
    """Single-pair form: ``(n_good, R, t, mask, points3d)``."""
    return recover_poses([F], [pts1], [pts2], K1, K2, masks=None if mask is None else [mask], distance_thresh=distance_thresh)[0]


# ------------------------------------------------------------------ scene-graph classification (SURVEY.md §8f rank 2)
DEGENERATE, PLANAR_OR_PANORAMIC, UNCALIBRATED, CALIBRATED = "degenerate", "planar_or_panoramic", "uncalibrated", "calibrated"


def classify_pairs(n_inliers_f, n_inliers_h, *, min_inliers=15, max_h_inlier_ratio=0.8, calibrated=False):
    """Scene-graph edge type per pair from the two inlier counts (the two-view geometry test of Schoenberger & Frahm
    2016 §4.1, ``papers/schoenberger2016sfm.pdf`` in the reference): a pair is kept iff F explains at least
    ``min_inliers`` matches; it is planar / panoramic (not usable to seed triangulation) when H explains more than
    ``max_h_inlier_ratio`` of what F explains."""
    nf = np.asarray(n_inliers_f, np.int64)
    nh = np.asarray(n_inliers_h, np.int64)
    out = np.full(nf.shape, CALIBRATED if calibrated else UNCALIBRATED, dtype=object)
    out[nh > max_h_inlier_ratio * nf] = PLANAR_OR_PANORAMIC
    out[nf < min_inliers] = DEGENERATE
    return out


def two_view_geometry(pts1, pts2, K1=None, K2=None, *, thr=3.0, confidence=0.99, max_iters=2000, solver="7pt", lo=True, seed=0,
                      min_inliers=15, max_h_inlier_ratio=0.8, distance_thresh=50.0):
    """Everything the scene graph stores for one pair: F and its inliers, H and its inliers, the edge type, and with
    intrinsics the relative pose and the triangulated inliers.  All three estimators run on the GPU."""
    F, fmask = verify_pair(pts1, pts2, thr=thr, confidence=confidence, max_iters=max_iters, solver=solver, lo=lo, seed=seed)
    H, hmask = find_homography(pts1, pts2, thr=thr, confidence=confidence, max_iters=max_iters, lo=lo, seed=seed,
                               stop_target=h_stop_target(int(fmask.sum()), max_h_inlier_ratio))
    out = {"F": F, "inlier_mask": fmask, "n_inliers": int(fmask.sum()), "H": H, "inlier_mask_h": hmask, "n_inliers_h": int(hmask.sum())}
    out["config"] = classify_pairs([out["n_inliers"]], [out["n_inliers_h"]], min_inliers=min_inliers,
                                   max_h_inlier_ratio=max_h_inlier_ratio, calibrated=K1 is not None)[0]
    if K1 is not None and F is not None:
        n, R, t, pm, X = recover_pose(F, pts1, pts2, K1, K2, mask=fmask, distance_thresh=distance_thresh)
        out.update(n_pose=n, R=R if n else None, t=t if n else None, in_front=pm, points3d=X)
    return out


# ------------------------------------------------------------------ feature tracks (correspondence search output)
def build_tracks(result, n_images, n_features, *, flags="inlier", min_pair_inliers=15, min_length=2, keep_conflicts=False):
    """Feature tracks of a matched image set (csrc/tracks.cu): the connected components of the graph whose nodes are
    ``image * n_features + feature`` and whose edges are the used match rows -- what ``code/3d_reconstruction.py`` (empty;
    imported at ``code/pipeline.py:4``) would build from ``pair_matches`` for registration and triangulation.

    ``result`` is one of
      * ``VerifiedPairs.to_host()`` (numpy; uploaded once),
      * the dict ``sfm_b200.dist.match_and_verify_sharded(gather="full")`` returns on its destination rank (device tensors,
        used in place),
      * the reference's ``pair_matches`` list (``Pair`` records whose ``matches`` are ``cv2.DMatch`` lists or int rows, as
        ``code/pipeline.py:36-47`` or ``sfm_b200.to_reference_pairs`` build it): every match is used, ``flags`` and
        ``min_pair_inliers`` do not apply.
    A row is used when its ``flags`` array (``"inlier"``, ``"inlier_h"``, ``"in_front"`` or None = every row) is set and its pair
    has ``n_inliers >= min_pair_inliers``.  Candidates holding two features of one image are dropped unless ``keep_conflicts``,
    then those with fewer than ``min_length`` observations.  Returns ``sfm_b200.Tracks`` (device; ``.to_host()`` for numpy)."""
    from sfm_b200 import tracks as tr

    opts = dict(min_length=min_length, keep_conflicts=keep_conflicts)
    if isinstance(result, dict) and "row_start" in result:
        return tr.build_tracks_from_rows(result, n_images, n_features, flags=flags, min_pair_inliers=min_pair_inliers, **opts)
    if isinstance(result, dict):
        off = np.asarray(result["offsets"], np.int64)
        return tr.build_tracks_device(result["pairs"], off[:-1], np.diff(off), result["matches"], tr.flag_rows(result, flags),
                                      result["n_inliers"], n_images, n_features, min_pair_inliers=min_pair_inliers, **opts)
    pairs, counts, rows = [], [], []
    for p in result:
        m = p.matches
        r = (np.asarray(m, np.int32).reshape(-1, 3)[:, :2] if isinstance(m, np.ndarray)
             else np.array([(d.queryIdx, d.trainIdx) for d in m], np.int32).reshape(-1, 2))
        pairs.append((p.img_inx_1, p.img_inx_2))
        counts.append(len(r))
        rows.append(np.concatenate([r, np.zeros((len(r), 1), np.int32)], axis=1))
    counts = np.asarray(counts, np.int64)
    start = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64) if len(counts) else np.zeros(0, np.int64)
    return tr.build_tracks_device(np.asarray(pairs, np.int32).reshape(-1, 2), start, counts,
                                  np.concatenate(rows) if rows else np.zeros((0, 3), np.int32), None, None, n_images, n_features, **opts)


# ------------------------------------------------------------------ track triangulation (tracks + cameras -> points)
def _device_tracks(tracks):
    """``sfm_b200.Tracks`` as given, or uploaded from its ``to_host()`` dict."""
    from sfm_b200 import tracks as tr

    if isinstance(tracks, dict):
        dev = torch.device("cuda", torch.cuda.current_device())
        counts = torch.tensor([tracks[k] for k in tr.COUNT_NAMES], dtype=torch.int64)
        return tr.Tracks(offsets_buf=torch.as_tensor(np.asarray(tracks["offsets"], np.int64)).to(dev),
                         obs_buf=torch.as_tensor(np.asarray(tracks["obs"], np.int32).reshape(-1, 2)).to(dev),
                         track_of_buf=torch.as_tensor(np.asarray(tracks["track_of"], np.int32)).to(dev), counts_dev=counts.to(dev))
    if not isinstance(tracks, tr.Tracks):
        raise TypeError(f"tracks must be sfm_b200.Tracks or its to_host() dict, got {type(tracks).__name__}")
    return tracks


def _keypoints(keypoints, n, dev):
    """(xy float32 [n, S, 2] on dev, S) of a ``DescriptorBank`` (its xy, in place) or an [n, S, 2] array."""
    if isinstance(keypoints, _sfm.DescriptorBank):
        if keypoints.device != dev:
            raise ValueError(f"the bank lives on {keypoints.device}, the tracks on {dev}")
        if n > keypoints.max_images:
            raise ValueError(f"{n} cameras for a bank of {keypoints.max_images} images")
        return keypoints.xy[:n], keypoints.max_feats
    a = np.asarray(keypoints)
    if a.ndim != 3 or a.shape[2] != 2 or a.shape[0] != n:
        raise ValueError(f"keypoints must be [{n}, S, 2], got {a.shape}")
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(dev), a.shape[1]


def triangulate_tracks(tracks, keypoints, K, R, t, *, registered=None, max_error=4.0, min_angle=1.5, max_iters=500, confidence=0.999,
                       seed=0, min_inliers=2):
    """One world point per feature track from known cameras ``x ~ K (R X + t)`` (csrc/triangulate.cu): two-view DLT
    hypotheses sampled RANSAC-style, kept when both depths are positive and the rays meet at ``min_angle`` degrees or more,
    scored by pixel reprojection error (an observation is an inlier within ``max_error`` pixels, in front of its camera), the
    best refit by an N-view DLT over its inliers.  The defaults of ``max_error`` and ``min_angle`` are COLMAP's mapper filter
    defaults.

    ``tracks``     ``sfm_b200.Tracks`` (device, e.g. ``match_and_verify(..., tracks=True).tracks``; nothing waits for the host) or
                   its ``to_host()`` dict
    ``keypoints``  the ``DescriptorBank`` the tracks were built from (its ``xy`` is read in place) or an [n_images, S, 2] array
    ``K``          one 3x3 pinhole matrix or [n,3,3]; ``R`` [n,3,3]; ``t`` [n,3] -- camera i observes image i
    ``registered`` bool / uint8 [n] or None: observations in images whose entry is 0 are not used
    Returns ``sfm_b200.TrackPoints`` (device; ``.to_host()`` for numpy): ``X``, ``n_inliers``, ``status`` per track (0 triangulated,
    1 too few views, 2 no model, 3 too few inliers, 4 invalid observation), ``obs_inlier`` and ``obs_error`` per observation."""
    from sfm_b200 import triangulate as tri

    cams = tri.camera_table(K, R, t)
    n = cams.shape[0]
    tracks = _device_tracks(tracks)
    dev = tracks.obs_buf.device
    xy, S = _keypoints(keypoints, n, dev)
    reg = None if registered is None else (np.asarray(registered).reshape(-1) != 0).astype(np.uint8)
    return tri.triangulate_tracks_device(tracks, xy, torch.from_numpy(cams).to(dev), reg, S=S, max_error=max_error, min_angle=min_angle,
                                         max_iters=max_iters, confidence=confidence, seed=seed, min_inliers=min_inliers)


# ------------------------------------------------------------------ registration (2-D / 3-D correspondences -> camera pose)
def estimate_absolute_poses(points2d, points3d, K, *, max_error=12.0, confidence=0.9999, max_iters=10000, min_inliers=30,
                            min_inlier_ratio=0.25, refine_iters=10, seed=0):
    """Batched ``cv2.solvePnPRansac`` + ``cv2.solvePnPRefineLM`` for calibrated pinhole cameras (csrc/pnp.cu): RANSAC over Lambda
    Twist P3P samples, an observation an inlier within ``max_error`` pixels in front of the camera, the best pose refined by
    Gauss-Newton on its inliers.  ``points2d`` / ``points3d`` are lists of [M_k, 2] pixel and [M_k, 3] world arrays, ``K`` one 3x3
    or [P,3,3].  The defaults of ``max_error``, ``min_inliers`` and ``min_inlier_ratio`` are COLMAP's incremental-mapper ones.
    Returns a list of ``(n_inliers, R float64[3,3], t float64[3], mask uint8[M_k,1])`` with x ~ K (R X + t); ``n_inliers == 0``
    means no pose (R and t are then zero)."""
    from sfm_b200 import pnp
    from sfm_b200 import triangulate as tri

    P = len(points2d)
    if len(points3d) != P:
        raise ValueError(f"{P} point sets of 2-D points, {len(points3d)} of 3-D points")
    if P == 0:
        return []
    p2 = [np.asarray(p, np.float64).reshape(-1, 2) for p in points2d]
    p3 = [np.asarray(p, np.float64).reshape(-1, 3) for p in points3d]
    counts = np.array([len(p) for p in p2], np.int32)
    if any(len(a) != len(b) for a, b in zip(p2, p3)):
        raise ValueError("every 2-D point set must have as many points as its 3-D set")
    cams = tri.camera_table(K, np.tile(np.eye(3), (P, 1, 1)), np.zeros((P, 3)))
    stride = max(int(counts.max()), 1)
    xy = np.zeros((P, stride, 2), np.float32)
    X = np.zeros((P, stride, 3), np.float64)
    for k in range(P):
        xy[k, : counts[k]] = p2[k]
        X[k, : counts[k]] = p3[k]
    dev = torch.device("cuda", torch.cuda.current_device())
    res = pnp.pnp_ransac_device(torch.from_numpy(xy).to(dev), torch.from_numpy(X).to(dev), torch.from_numpy(counts).to(dev),
                                torch.from_numpy(cams).to(dev), np.arange(P, dtype=np.int32), max_error=max_error, confidence=confidence,
                                max_iters=max_iters, min_inliers=min_inliers, min_inlier_ratio=min_inlier_ratio, refine_iters=refine_iters,
                                seed=seed).to_host()
    ok = res["status"] == 0
    return [(int(res["n_inliers"][k]) if ok[k] else 0, res["R"][k].copy(), res["t"][k].copy(), res["mask"][k, : counts[k]].reshape(-1, 1).copy())
            for k in range(P)]


def estimate_absolute_pose(pts2d, pts3d, K, **kw):
    """Single-set form: ``(n_inliers, R, t, mask)``."""
    return estimate_absolute_poses([pts2d], [pts3d], K, **kw)[0]


def register_images(tracks, points, keypoints, K, R, t, images, *, registered=None, max_error=12.0, confidence=0.9999, max_iters=10000,
                    min_inliers=30, min_inlier_ratio=0.25, refine_iters=10, seed=0):
    """Register ``images`` against triangulated tracks (csrc/pnp.cu): the correspondences of image i are its features whose track
    has a point (``points``, from ``triangulate_tracks``), in feature order; the pose as ``estimate_absolute_poses``.

    ``tracks``, ``keypoints``, ``K``, ``R``, ``t`` as ``triangulate_tracks`` (only the intrinsics of ``images`` are read);
    ``registered`` None or a bool / uint8 [n] array or tensor, set to 1 in place for every image registered here.  Returns
    ``sfm_b200.AbsolutePoses`` (device; ``.to_host()`` for numpy): ``R``, ``t``, ``n_inliers``, ``status`` per image (0 registered,
    1 fewer than 3 points, 2 no model, 3 too few inliers, 4 invalid image), ``mask`` and ``feature`` per correspondence."""
    from sfm_b200 import pnp
    from sfm_b200 import triangulate as tri

    cams = tri.camera_table(K, R, t)
    n = cams.shape[0]
    tracks = _device_tracks(tracks)
    dev = tracks.obs_buf.device
    xy, _ = _keypoints(keypoints, n, dev)
    res = pnp.register_images_device(tracks, points, xy, torch.from_numpy(cams).to(dev), images, max_error=max_error, confidence=confidence,
                                     max_iters=max_iters, min_inliers=min_inliers, min_inlier_ratio=min_inlier_ratio,
                                     refine_iters=refine_iters, seed=seed)
    if registered is not None:
        ok = res.status == 0
        img = res.images.long()[ok]
        if isinstance(registered, torch.Tensor):
            registered[img.to(registered.device)] = 1
        else:
            registered[img.cpu().numpy()] = 1
    return res


# ------------------------------------------------------------------ bundle adjustment (cameras + points, jointly)
def bundle_adjust(tracks, points, keypoints, K, R, t, *, registered=None, fixed=None, max_iters=50, function_tolerance=1e-6,
                  parameter_tolerance=1e-8):
    """Refine the registered cameras ``x ~ K (R X + t)`` and the triangulated points together (csrc/bundle.cu):
    Levenberg-Marquardt on the squared pixel errors of every observation whose track has a point (``points``, from
    ``triangulate_tracks``), that is an inlier of it and lies in a registered image; intrinsics fixed, no robust loss.

    ``tracks``, ``keypoints``, ``K``, ``R``, ``t``, ``registered`` as ``triangulate_tracks``; ``fixed`` bool / uint8 [n] or None
    (None: the lowest-index registered camera is held fixed).  At most 1024 cameras.  Returns a dict of numpy ``R`` [n,3,3],
    ``t`` [n,3], ``X`` [T,3], ``obs_error`` [n_obs] (pixel error after the adjustment; NaN where triangulation writes NaN) and
    ``status`` (one of ``sfm_b200.bundle.STATUS_NAMES``), ``iterations``, ``accepted``, ``initial_cost``, ``final_cost``,
    ``used_obs``, ``variable_cameras``, ``adjusted_points``."""
    from sfm_b200 import bundle
    from sfm_b200 import triangulate as tri

    cams = tri.camera_table(K, R, t)
    n = cams.shape[0]
    tracks = _device_tracks(tracks)
    dev = tracks.obs_buf.device
    xy, S = _keypoints(keypoints, n, dev)
    reg = None if registered is None else (np.asarray(registered).reshape(-1) != 0).astype(np.uint8)
    fix = None if fixed is None else (np.asarray(fixed).reshape(-1) != 0).astype(np.uint8)
    res = bundle.bundle_adjust_device(tracks, points, xy, torch.from_numpy(cams).to(dev), reg, fixed=fix, S=S, max_iters=max_iters,
                                      function_tolerance=function_tolerance, parameter_tolerance=parameter_tolerance).to_host()
    res.pop("pose")
    return res
