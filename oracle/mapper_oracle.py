"""numpy restatement of the incremental-reconstruction kernels (csrc/mapper.cu; include/sfm_b200.h, "incremental
reconstruction").  TEST INFRASTRUCTURE ONLY.

``next_images`` restates sfm_next_images: the visible points of every image (sfm_pnp_gather's predicate), the visibility-
pyramid score (integers), the candidate order and the trials update.  ``filter_points`` restates sfm_filter_points: the
observations that stay inliers, the recount and the triangulation-angle test, with the operations of the shared device
helpers ``camera_center`` and ``ray_cos`` (csrc/ransac_common.cuh) in the same order, so both equal the kernels bit for bit.
"""
from __future__ import annotations

import math

import numpy as np


def visible_mask(track_of, n_tracks, point_status):
    """bool [n_images, S]: features whose track has a point (sfm_pnp_gather's predicate)."""
    k = np.asarray(track_of).astype(np.int64)
    ok = np.zeros(n_tracks + 1, bool)                       # slot n_tracks: "no track"
    ok[:n_tracks] = np.asarray(point_status)[:n_tracks] == 0
    return ok[np.where((k >= 0) & (k < n_tracks), k, n_tracks)]


def pyramid_score(x, y, w, h, levels=6):
    """int score of the visible points (x, y) (float32) of one image of size (w, h)."""
    x = np.asarray(x, np.float32).astype(np.float64)
    y = np.asarray(y, np.float32).astype(np.float64)
    s = 0
    for lv in range(levels):
        d = 2 << lv
        cells = []
        for v, size in ((x, float(w)), (y, float(h))):
            with np.errstate(divide="ignore", invalid="ignore"):
                c = np.floor(v * float(d) / size)
            cells.append(np.where(c > 0.0, np.where(c < float(d - 1), c, float(d - 1)), 0.0).astype(np.int64))
        s += d * d * len(np.unique(cells[1] * d + cells[0]))
    return s


def next_images(track_of, n_tracks, point_status, xy, image_size, registered, trials, *, max_select, min_visible=30, max_trials=3,
                levels=6):
    """track_of int32 [n_images, S], point_status uint8 [>= n_tracks], xy float32 [n_images, >= S, 2], image_size int [n_images, 2]
    (w, h), registered uint8 [n_images], trials int32 [n_images].  Returns ``images`` int32 [max_select] (-1 padded),
    ``n_selected``, ``visible`` int32 [n_images], ``score`` int64 [n_images] and the updated ``trials``."""
    track_of = np.asarray(track_of)
    n_images, S = track_of.shape
    vis = visible_mask(track_of, n_tracks, point_status)
    xy = np.asarray(xy, np.float32)
    size = np.asarray(image_size, np.int64).reshape(n_images, 2)
    visible = vis.sum(1).astype(np.int32)
    score = np.zeros(n_images, np.int64)
    for i in range(n_images):
        f = np.nonzero(vis[i])[0]
        score[i] = pyramid_score(xy[i, f, 0], xy[i, f, 1], size[i, 0], size[i, 1], levels)
    reg = np.asarray(registered).reshape(n_images)
    trials = np.asarray(trials, np.int32).reshape(n_images).copy()
    cand = np.nonzero((reg == 0) & (trials < max_trials) & (visible >= min_visible))[0]
    order = sorted(cand.tolist(), key=lambda i: (-int(score[i]), -int(visible[i]), i))
    sel = order[:max_select]
    images = np.full(max_select, -1, np.int32)
    images[: len(sel)] = sel
    trials[sel] += 1
    return {"images": images, "n_selected": len(sel), "visible": visible, "score": score, "trials": trials}


def camera_center(cam):
    """C = -R^T t of one camera-table row, as camera_center (csrc/ransac_common.cuh)."""
    r, t = [float(v) for v in cam[4:13]], [float(v) for v in cam[13:16]]
    return [-(r[i] * t[0] + r[3 + i] * t[1] + r[6 + i] * t[2]) for i in range(3)]


def ray_cos(X, Ca, Cb):
    """ray_cos (csrc/ransac_common.cuh) in Python floats (IEEE fp64, the same operation order)."""
    da = [X[0] - Ca[0], X[1] - Ca[1], X[2] - Ca[2]]
    db = [X[0] - Cb[0], X[1] - Cb[1], X[2] - Cb[2]]
    dot = da[0] * db[0] + da[1] * db[1] + da[2] * db[2]
    na = da[0] * da[0] + da[1] * da[1] + da[2] * da[2]
    nb = db[0] * db[0] + db[1] * db[1] + db[2] * db[2]
    with np.errstate(divide="ignore", invalid="ignore"):         # a point on a centre divides by zero, as the kernel does
        return float(np.float64(dot) / np.sqrt(np.float64(na * nb)))


def cos_min_of(min_angle):
    return math.cos(float(min_angle) * 0.017453292519943295)


def filter_points(offsets, obs, cams, registered, X, n_inliers, status, obs_inlier, obs_error, *, max_error=4.0, min_angle=1.5,
                  min_inliers=2):
    """offsets int64 [T+1], obs int32 [n_obs, 2], cams float64 [n_images, 16], registered uint8 [n_images], and the
    triangulation outputs X [T,3], n_inliers [T], status [T], obs_inlier [n_obs], obs_error float32 [n_obs].  Returns the
    filtered X, n_inliers, status, obs_inlier and counts int64 [5] (copies; the inputs are not changed)."""
    offsets = np.asarray(offsets, np.int64)
    obs = np.asarray(obs).reshape(-1, 2)
    cams = np.asarray(cams, np.float64)
    reg = np.asarray(registered).reshape(-1)
    n_images = len(reg)
    T = len(offsets) - 1
    X = np.array(X, np.float64).reshape(-1, 3)[:T].copy()
    n_inl = np.array(n_inliers, np.int32)[:T].copy()
    st = np.array(status, np.uint8)[:T].copy()
    n_obs = int(offsets[-1]) if T >= 0 and len(offsets) else 0
    inl = np.array(obs_inlier, np.uint8)[:n_obs].copy()
    err = np.asarray(obs_error, np.float32)[:n_obs].astype(np.float64)
    cos_min = cos_min_of(min_angle)
    centres = {}
    for k in np.nonzero(st == 0)[0]:
        a0, a1 = int(offsets[k]), int(offsets[k + 1])
        img = obs[a0:a1, 0].astype(np.int64)
        ok = (inl[a0:a1] != 0) & (img >= 0) & (img < n_images)
        ok[ok] &= reg[img[ok]] != 0
        with np.errstate(invalid="ignore"):
            ok &= err[a0:a1] <= float(max_error)
        inl[a0:a1] = ok
        n = int(ok.sum())
        s = 0
        if n < min_inliers:
            s = 3
        else:
            Xk = [float(v) for v in X[k]]
            cs = []
            for i in img[ok]:
                if i not in centres:
                    centres[i] = camera_center(cams[i])
                cs.append(centres[i])
            found = any(ray_cos(Xk, cs[a], cs[b]) <= cos_min for a in range(n) for b in range(a + 1, n))
            if not found:
                s = 2
        if s:
            inl[a0:a1] = 0
            X[k] = 0.0
        n_inl[k] = 0 if s == 2 else n
        st[k] = s
    counts = np.bincount(st, minlength=5)[:5].astype(np.int64)
    return {"X": X, "n_inliers": n_inl, "status": st, "obs_inlier": inl, "counts": counts}
