"""A float64 bundle-adjustment reference written from the textbook, sharing no code with csrc/bundle.cu.

It differs from the kernel on purpose: rotations are perturbed in the world frame by angle-axis vectors through
``scipy.spatial.transform.Rotation`` (R' = R exp([d]x), where the kernel perturbs in the camera frame), and each step solves
the full sparse damped normal equations with ``scipy.sparse.linalg.spsolve`` (no Schur complement).  Levenberg-Marquardt
with Marquardt's diagonal scaling and Nielsen's damping update, run until the cost stops falling; a trial that puts a point
behind a camera is rejected.  The world is first translated to the centroid of the points (an exact change of gauge, undone
at the end): world-frame rotations couple to the translations through |X|, and far from the origin LM would crawl.

A problem is the set of used observations: ``cams`` float64 [n, 16] (fx fy cx cy, R row-major, t), ``X`` [T, 3], ``cam``
int [M], ``pt`` int [M], ``xy`` float64 [M, 2] pixels, ``var_cams`` bool [n] (cameras that move), ``adj_pts`` bool [T] (points
that move).  Residuals are pixels: fx p0 / p2 + cx - x, fy p1 / p2 + cy - y with p = R X + t.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
from scipy.sparse.linalg import spsolve
from scipy.spatial.transform import Rotation


def residuals(cams, X, cam, pt, xy):
    R = cams[cam, 4:13].reshape(-1, 3, 3)
    p = np.einsum("mij,mj->mi", R, X[pt]) + cams[cam, 13:16]
    u = cams[cam, 0] * p[:, 0] / p[:, 2] + cams[cam, 2] - xy[:, 0]
    v = cams[cam, 1] * p[:, 1] / p[:, 2] + cams[cam, 3] - xy[:, 1]
    return np.column_stack([u, v]).ravel()


def _layout(var_cams, adj_pts):
    ci = -np.ones(len(var_cams), np.int64)
    ci[var_cams] = np.arange(var_cams.sum())
    pi = -np.ones(len(adj_pts), np.int64)
    pi[adj_pts] = np.arange(adj_pts.sum())
    return ci, pi, 6 * int(var_cams.sum()), 3 * int(adj_pts.sum())


def jacobian(cams, X, cam, pt, var_cams, adj_pts):
    """Sparse d(residuals) / d(d, t of the variable cameras, X of the adjusted points), d the world-frame rotation."""
    ci, pi, nc, npt = _layout(var_cams, adj_pts)
    M = len(cam)
    R = cams[cam, 4:13].reshape(-1, 3, 3)
    Xm = X[pt]
    p = np.einsum("mij,mj->mi", R, Xm) + cams[cam, 13:16]
    fx, fy = cams[cam, 0], cams[cam, 1]
    du = np.column_stack([fx / p[:, 2], np.zeros(M), -fx * p[:, 0] / p[:, 2] ** 2])
    dv = np.column_stack([np.zeros(M), fy / p[:, 2], -fy * p[:, 1] / p[:, 2] ** 2])
    skew = np.zeros((M, 3, 3))
    skew[:, 0, 1], skew[:, 0, 2], skew[:, 1, 2] = -Xm[:, 2], Xm[:, 1], -Xm[:, 0]
    skew[:, 1, 0], skew[:, 2, 0], skew[:, 2, 1] = Xm[:, 2], -Xm[:, 1], Xm[:, 0]
    dp_dd = -np.einsum("mij,mjk->mik", R, skew)                  # p = R (X + d x X) + t
    rows, cols, vals = [], [], []
    for k, d in ((0, du), (1, dv)):
        r = 2 * np.arange(M) + k
        vc = ci[cam] >= 0
        blocks = np.concatenate([np.einsum("mi,mij->mj", d, dp_dd), d], axis=1)
        for c in range(6):
            rows.append(r[vc]); cols.append(6 * ci[cam][vc] + c); vals.append(blocks[vc, c])
        vp = pi[pt] >= 0
        bx = np.einsum("mi,mij->mj", d, R)
        for c in range(3):
            rows.append(r[vp]); cols.append(nc + 3 * pi[pt][vp] + c); vals.append(bx[vp, c])
    return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(2 * M, nc + npt))


def apply_step(cams, X, h, var_cams, adj_pts):
    ci, pi, nc, _ = _layout(var_cams, adj_pts)
    cams, X = cams.copy(), X.copy()
    for i in np.nonzero(var_cams)[0]:
        d = h[6 * ci[i]: 6 * ci[i] + 6]
        R = cams[i, 4:13].reshape(3, 3) @ Rotation.from_rotvec(d[:3]).as_matrix()
        cams[i, 4:13] = R.ravel()
        cams[i, 13:16] += d[3:]
    X[adj_pts] += h[nc:].reshape(-1, 3)
    return cams, X


def gradient(cams, X, cam, pt, xy, var_cams, adj_pts):
    """J^T r in the reference's parameters."""
    return jacobian(cams, X, cam, pt, var_cams, adj_pts).T @ residuals(cams, X, cam, pt, xy)


def bundle_adjust(cams, X, cam, pt, xy, var_cams, adj_pts, *, max_iters=500, ftol=1e-15):
    """Returns dict(cams, X, cost, residuals, iterations, initial_cost)."""
    cams, X = np.asarray(cams, np.float64).copy(), np.asarray(X, np.float64).copy()
    cam, pt, xy = np.asarray(cam), np.asarray(pt), np.asarray(xy, np.float64)
    var_cams, adj_pts = np.asarray(var_cams, bool), np.asarray(adj_pts, bool)
    o = X[np.unique(pt)].mean(0) if len(pt) else np.zeros(3)
    X = X - o
    cams[:, 13:16] += np.einsum("nij,j->ni", cams[:, 4:13].reshape(-1, 3, 3), o)
    out = _lm(cams, X, cam, pt, xy, var_cams, adj_pts, max_iters, ftol)
    out["X"] = out["X"] + o
    out["cams"][:, 13:16] -= np.einsum("nij,j->ni", out["cams"][:, 4:13].reshape(-1, 3, 3), o)
    return out


def _in_front(cams, X, cam, pt):
    return bool(np.all(np.einsum("mj,mj->m", cams[cam, 10:13], X[pt]) + cams[cam, 15] > 0))


def _lm(cams, X, cam, pt, xy, var_cams, adj_pts, max_iters, ftol):
    r = residuals(cams, X, cam, pt, xy)
    cost = float(r @ r)
    init = cost
    lam, nu, it = 1e-4, 2.0, 0
    for it in range(1, max_iters + 1):
        J = jacobian(cams, X, cam, pt, var_cams, adj_pts)
        if J.shape[1] == 0:
            break
        A = (J.T @ J).tocsc()
        g = J.T @ r
        D = A.diagonal()
        while True:
            h = spsolve(A + sp.diags(lam * D), -g)
            c2, X2 = apply_step(cams, X, h, var_cams, adj_pts)
            r2 = residuals(c2, X2, cam, pt, xy)
            new = float(r2 @ r2)
            pred = float(h @ (lam * D * h - g))
            if np.isfinite(new) and new < cost and pred > 0 and _in_front(c2, X2, cam, pt):
                rho = (cost - new) / pred
                lam *= max(1.0 / 3.0, 1.0 - (2.0 * rho - 1.0) ** 3)
                nu = 2.0
                break
            lam *= nu
            nu *= 2.0
            if lam > 1e32:
                return dict(cams=cams, X=X, cost=cost, residuals=r, iterations=it, initial_cost=init)
        done = cost - new < ftol * cost
        cams, X, r, cost = c2, X2, r2, new
        if done:
            break
    return dict(cams=cams, X=X, cost=cost, residuals=r, iterations=it, initial_cost=init)


def problem(offsets, obs, point_status, obs_inlier, n_images, registered=None, fixed=None):
    """The used observations of tracks as sfm_tracks_finalize / sfm_triangulate_tracks write them, and the variable cameras
    and adjusted points, by the definitions of include/sfm_b200.h: returns (cam, pt, obs index, var_cams, adj_pts)."""
    offsets, obs = np.asarray(offsets, np.int64), np.asarray(obs).reshape(-1, 2)
    T = len(offsets) - 1
    reg = np.ones(n_images, bool) if registered is None else np.asarray(registered).reshape(-1) != 0
    if fixed is None:
        fix = np.zeros(n_images, bool)
        if reg.any():
            fix[np.argmax(reg)] = True
    else:
        fix = np.asarray(fixed).reshape(-1) != 0
    track = np.repeat(np.arange(T), np.diff(offsets))
    img = obs[: offsets[-1], 0]
    used = (np.asarray(point_status)[track] == 0) & (np.asarray(obs_inlier)[: offsets[-1]] == 1) & reg[img]
    o = np.nonzero(used)[0]
    adj = np.bincount(track[o], minlength=T) >= 2
    var = reg & ~fix & (np.bincount(img[o], minlength=n_images) > 0)
    return img[o], track[o], o, var, adj
