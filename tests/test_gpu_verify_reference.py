"""RANSAC-F, RANSAC-H and two-view pose against an independent float64 reference, at real camera sizes and with a
different camera for each image of a pair.

The C oracles under ``oracle/`` restate the kernels operation for operation, so bit-exact agreement with them cannot catch
a flaw the two copies share.  The reference here is written from the textbook definitions instead (Hartley & Zisserman,
2nd ed.: normalised 8-point §11.2, 7-point §11.1.2, DLT §4.1, essential-matrix decomposition §9.6), uses SVD where the
kernels use Gauss-Jordan, Jacobi or inverse iteration, and finds cubic roots with ``np.roots``.  Its CPU tests (no
``gpu`` mark, no GPU needed) pin it against cv2.  The GPU tests then hold the kernels to it:

* minimal solvers through explicit samples: 8-point and DLT models to 1e-9, the 7-point model is the best-scoring root;
* degenerate samples give no model;
* full runs: every inlier decision outside a narrow band around thr^2 is the float64 decision on the returned model;
* pose with K1 != K2, and the per-pair camera rows of ``match_and_verify(intrinsics=...)``.

The scenes are built here, each camera with its own intrinsics and image size (640x480 up to 7680x4320, off-centre
principal points, one camera whose pixel origin is the image centre so that coordinates are negative).
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

try:
    import torch

    HAS_CUDA = torch.cuda.is_available()
except ImportError:                                    # pragma: no cover - torch is a dependency of the package
    HAS_CUDA = False


def gpu_test(fn):
    """GPU tests are marked and skipped one by one: the reference's own CPU tests in this file must still run without one."""
    return pytest.mark.gpu(pytest.mark.skipif(not HAS_CUDA, reason="needs a GPU")(fn))


# ====================================================================================================== float64 reference

def to_h(p):
    p = np.asarray(p, np.float64).reshape(-1, 2)
    return np.column_stack([p, np.ones(len(p))])


def hartley(p):
    """Hartley's normalisation: centroid to the origin, mean distance from it sqrt(2).  Returns (T, normalised points)."""
    p = np.asarray(p, np.float64).reshape(-1, 2)
    c = p.mean(axis=0)
    s = np.sqrt(2.0) / np.linalg.norm(p - c, axis=1).mean()
    T = np.array([[s, 0.0, -s * c[0]], [0.0, s, -s * c[1]], [0.0, 0.0, 1.0]])
    return T, (p - c) * s


def epipolar_rows(u1, u2):
    """One row per correspondence of x2^T F x1 = 0 with F row-major."""
    x, y, xp, yp = u1[:, 0], u1[:, 1], u2[:, 0], u2[:, 1]
    return np.column_stack([xp * x, xp * y, xp, yp * x, yp * y, yp, x, y, np.ones(len(x))])


def unit(M):
    M = np.asarray(M, np.float64).reshape(3, 3)
    return M / np.linalg.norm(M)


def model_dist(A, B):
    """Distance between two projective 3x3 models: both scaled to unit Frobenius norm, sign chosen to match."""
    a, b = unit(A), unit(B)
    return min(np.abs(a - b).max(), np.abs(a + b).max())


def fundamental_8pt(p1, p2):
    """Normalised 8-point (least squares for more than 8 points): SVD null vector, rank 2 by zeroing the smallest
    singular value, denormalised.  Returns (F with unit Frobenius norm, singular values of the design matrix)."""
    T1, u1 = hartley(p1)
    T2, u2 = hartley(p2)
    A = epipolar_rows(u1, u2)
    _, sv, vt = np.linalg.svd(A)
    U, S, Vt = np.linalg.svd(vt[-1].reshape(3, 3))
    Fn = U @ np.diag([S[0], S[1], 0.0]) @ Vt
    return unit(T2.T @ Fn @ T1), sv


def fundamental_7pt(p1, p2):
    """7-point: the 2-D null space {G1, G2}, every real root of the cubic det(l G1 + (1 - l) G2) = 0.  The cubic is
    recovered exactly from four evaluations of the determinant.  Returns (list of F, singular values of the design matrix)."""
    T1, u1 = hartley(p1)
    T2, u2 = hartley(p2)
    _, sv, vt = np.linalg.svd(epipolar_rows(u1, u2), full_matrices=True)
    G1, G2 = vt[-2].reshape(3, 3), vt[-1].reshape(3, 3)
    ls = np.array([-1.0, 0.0, 1.0, 2.0])
    coef = np.polyfit(ls, [np.linalg.det(l * G1 + (1.0 - l) * G2) for l in ls], 3)
    models = []
    for r in np.roots(coef):
        if abs(r.imag) <= 1e-9 * (1.0 + abs(r)):
            l = r.real
            models.append(unit(T2.T @ (l * G1 + (1.0 - l) * G2) @ T1))
    return models, sv


def homography_dlt(p1, p2):
    """Normalised DLT, x2 ~ H x1.  Returns (H with H[2,2] = 1, singular values of the design matrix)."""
    T1, u1 = hartley(p1)
    T2, u2 = hartley(p2)
    x, y, xp, yp = u1[:, 0], u1[:, 1], u2[:, 0], u2[:, 1]
    z, o = np.zeros(len(x)), np.ones(len(x))
    A = np.concatenate([np.column_stack([x, y, o, z, z, z, -xp * x, -xp * y, -xp]),
                        np.column_stack([z, z, z, x, y, o, -yp * x, -yp * y, -yp])])
    _, sv, vt = np.linalg.svd(A)
    H = np.linalg.inv(T2) @ vt[-1].reshape(3, 3) @ T1
    return H / H[2, 2], sv


def f_errors(F, p1, p2):
    """(cv2's symmetric epipolar error max(d1^2, d2^2), Sampson error), px^2."""
    x1, x2 = to_h(p1), to_h(p2)
    F = np.asarray(F, np.float64).reshape(3, 3)
    l2, l1 = x1 @ F.T, x2 @ F                     # epipolar lines in image 2 and in image 1
    r2 = ((x2 * l2).sum(1)) ** 2
    n2, n1 = l2[:, 0] ** 2 + l2[:, 1] ** 2, l1[:, 0] ** 2 + l1[:, 1] ** 2
    return r2 / np.minimum(n1, n2), r2 / (n1 + n2)


def h_error(H, p1, p2):
    """Forward transfer error |proj(H x1) - x2|^2, px^2."""
    q = to_h(p1) @ np.asarray(H, np.float64).reshape(3, 3).T
    return ((q[:, :2] / q[:, 2:] - np.asarray(p2, np.float64).reshape(-1, 2)) ** 2).sum(1)


def algebraic_residual(F, p1, p2):
    """Sum of squared algebraic residuals in the Hartley frame of these points, F scaled to unit norm in that frame."""
    T1, u1 = hartley(p1)
    T2, u2 = hartley(p2)
    Fn = unit(np.linalg.inv(T2).T @ np.asarray(F, np.float64).reshape(3, 3) @ np.linalg.inv(T1))
    return float(((epipolar_rows(u1, u2) @ Fn.ravel()) ** 2).sum())


def triangulate(R, t, n1, n2):
    """DLT triangulation with P1 = [I|0], P2 = [R|t] on normalised coordinates; X in camera 1's frame."""
    P1 = np.hstack([np.eye(3), np.zeros((3, 1))])
    P2 = np.hstack([R, t.reshape(3, 1)])
    A = np.stack([n1[:, :1] * P1[2] - P1[0], n1[:, 1:] * P1[2] - P1[1], n2[:, :1] * P2[2] - P2[0], n2[:, 1:] * P2[2] - P2[1]], axis=1)
    v = np.linalg.svd(A)[2][:, -1]
    with np.errstate(divide="ignore", invalid="ignore"):
        return v[:, :3] / v[:, 3:]


def normalise_pixels(p, K):
    K = np.asarray(K, np.float64)
    p = np.asarray(p, np.float64).reshape(-1, 2)
    return np.column_stack([(p[:, 0] - K[0, 2]) / K[0, 0], (p[:, 1] - K[1, 2]) / K[1, 1]])


def relative_pose(F, K1, K2, p1, p2, mask=None, dist=50.0):
    """E = K2^T F K1, its four (R, t), cheirality vote over the masked correspondences (depth in (0, dist) in both
    cameras), in cv2.recoverPose's candidate order.  Returns (R, t, good mask, X [M,3] zero where not good, votes)."""
    E = np.asarray(K2, np.float64).T @ np.asarray(F, np.float64).reshape(3, 3) @ np.asarray(K1, np.float64)
    U, _, Vt = np.linalg.svd(E / np.linalg.norm(E))
    U, Vt = U * np.sign(np.linalg.det(U)), Vt * np.sign(np.linalg.det(Vt))
    W = np.array([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    Ra, Rb, t = U @ W @ Vt, U @ W.T @ Vt, U[:, 2]
    n1, n2 = normalise_pixels(p1, K1), normalise_pixels(p2, K2)
    use = np.ones(len(n1), bool) if mask is None else np.asarray(mask).ravel().astype(bool)
    best = None
    votes = []
    for R, tt in ((Ra, t), (Rb, t), (Ra, -t), (Rb, -t)):
        X = np.zeros((len(n1), 3))
        X[use] = triangulate(R, tt, n1[use], n2[use])
        z2 = X @ R[2] + tt[2]
        with np.errstate(invalid="ignore"):
            good = use & (X[:, 2] > 0) & (X[:, 2] < dist) & (z2 > 0) & (z2 < dist)
        votes.append(int(good.sum()))
        if best is None or votes[-1] > votes[best[0]]:
            best = (len(votes) - 1, R, tt, good, np.where(good[:, None], X, 0.0))
    _, R, tt, good, X = best
    return R, tt, good, X, votes


# ====================================================================================================== two-camera scenes

Camera = namedtuple("Camera", "w h fx fy cx cy x0 y0", defaults=(0.0, 0.0))   # pixel domain [x0, x0 + w) x [y0, y0 + h)


def K_of(c: Camera):
    return np.array([[c.fx, 0.0, c.cx], [0.0, c.fy, c.cy], [0.0, 0.0, 1.0]])


# one rig per image size, the two cameras of a rig always differ (focal length, aspect, principal point)
RIGS = {
    "640x480": (Camera(640, 480, 560.0, 560.0, 320.0, 240.0), Camera(640, 480, 610.0, 612.0, 301.5, 255.25)),
    "1920x1080": (Camera(1920, 1080, 1500.0, 1500.0, 960.0, 540.0), Camera(1920, 1080, 1320.0, 1318.0, 1003.0, 517.5)),
    "4000x3000": (Camera(4000, 3000, 3100.0, 3100.0, 2000.0, 1500.0), Camera(4000, 3000, 3500.0, 3496.0, 1890.0, 1575.0)),
    "7680x4320": (Camera(7680, 4320, 5800.0, 5800.0, 3840.0, 2160.0), Camera(7680, 4320, 6400.0, 6390.0, 3702.0, 2251.0)),
    "640x480+7680x4320": (Camera(640, 480, 560.0, 560.0, 331.0, 236.0), Camera(7680, 4320, 6400.0, 6400.0, 3840.0, 2160.0)),
    # pixel origin at the image centre: coordinates from -2000 to 2000 (and a principal point off that centre)
    "4000x3000-centred": (Camera(4000, 3000, 3100.0, 3100.0, 0.0, 0.0, -2000.0, -1500.0),
                          Camera(4000, 3000, 3300.0, 3300.0, 35.0, -20.0, -2000.0, -1500.0)),
}
RIG_NAMES = list(RIGS)


def _look_at(pos, target):
    z = target - pos
    z = z / np.linalg.norm(z)
    x = np.cross([0.0, 1.0, 0.0], z)
    x = x / np.linalg.norm(x)
    return np.stack([x, np.cross(z, x), z])


def rig_scene(name, n, *, planar=False, outlier_frac=0.3, sigma=0.5, seed=0):
    """Correspondences seen by the two cameras of RIGS[name].  Camera 1 sits at the origin looking down +z; camera 2 is
    1.2 units to the side and looks at (0, 0, 8).  General scenes have depths 4..12, planar ones lie on one tilted plane.
    Returns dict(p1, p2 float32 [n,2], gt bool [n], K1, K2, R, t (x2 ~ R x1 + t, |t| = 1), F (unit norm), H or None)."""
    c1, c2 = RIGS[name]
    K1, K2 = K_of(c1), K_of(c2)
    rng = np.random.default_rng(seed)
    C2 = np.array([1.2, 0.15, 0.3])
    R = _look_at(C2, np.array([0.0, 0.0, 8.0]))
    t = -R @ C2
    nrm, d0 = np.array([-0.3, 0.2, 1.0]), 8.0                 # plane nrm . X = d0 (camera 1 frame)
    x1s, x2s = [], []
    while sum(len(a) for a in x1s) < n:
        m = 4 * n
        px = np.column_stack([rng.uniform(c1.x0, c1.x0 + c1.w, m), rng.uniform(c1.y0, c1.y0 + c1.h, m)])
        ray = np.linalg.solve(K1, to_h(px).T).T
        z = d0 / (ray @ nrm) if planar else rng.uniform(4.0, 12.0, m)
        X = ray * z[:, None]
        q = (K2 @ (X @ R.T + t).T).T
        x2 = q[:, :2] / q[:, 2:]
        ok = (q[:, 2] > 0) & (x2[:, 0] >= c2.x0) & (x2[:, 0] < c2.x0 + c2.w) & (x2[:, 1] >= c2.y0) & (x2[:, 1] < c2.y0 + c2.h)
        x1s.append(px[ok])
        x2s.append(x2[ok])
    p1 = np.concatenate(x1s)[:n] + rng.normal(0.0, sigma, (n, 2))
    p2 = np.concatenate(x2s)[:n] + rng.normal(0.0, sigma, (n, 2))
    out = rng.permutation(n)[: int(round(outlier_frac * n))]
    p2[out] = np.column_stack([rng.uniform(c2.x0, c2.x0 + c2.w, len(out)), rng.uniform(c2.y0, c2.y0 + c2.h, len(out))])
    gt = np.ones(n, bool)
    gt[out] = False
    tx = np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]])
    F = unit(np.linalg.inv(K2).T @ tx @ R @ np.linalg.inv(K1))
    H = None
    if planar:
        H = K2 @ (R + np.outer(t, nrm) / d0) @ np.linalg.inv(K1)
        H = H / H[2, 2]
    return dict(p1=p1.astype(np.float32), p2=p2.astype(np.float32), gt=gt, K1=K1, K2=K2, R=R, t=t / np.linalg.norm(t), F=F, H=H)


def exact_affine_pairs(name, n, seed=0):
    """n correspondences related EXACTLY, in float32, by one affine map (a homography induced by a plane): integer pixels
    in image 1, dyadic coefficients.  Every 8 of them are coplanar for F, every 4 are consistent with one H."""
    c1, _ = RIGS[name]
    rng = np.random.default_rng(seed)
    p1 = np.column_stack([rng.integers(int(c1.x0), int(c1.x0 + c1.w), n), rng.integers(int(c1.y0), int(c1.y0 + c1.h), n)]).astype(np.float64)
    A = np.array([[0.75, 0.125], [-0.25, 1.5]])
    p2 = p1 @ A.T + np.array([37.5, -12.25])
    assert np.array_equal(p2.astype(np.float32).astype(np.float64), p2)
    return p1.astype(np.float32), p2.astype(np.float32)


# ====================================================================================================== the reference vs cv2 (CPU)

def _pin_cases():
    return [(name, seed) for name in RIG_NAMES for seed in (1, 2)]


@pytest.mark.parametrize("name,seed", _pin_cases())
def test_reference_minimal_solvers_equal_cv2(name, seed):
    """8-point == cv2 FM_8POINT (8 points and least squares over all inliers), the 7-point root set == cv2 FM_7POINT's
    models, 4-point DLT == cv2.findHomography(method=0)."""
    s = rig_scene(name, 300, seed=seed, outlier_frac=0.2, sigma=0.5)
    p1, p2, gt = s["p1"], s["p2"], s["gt"]
    rng = np.random.default_rng(seed)
    inl = np.flatnonzero(gt)
    for _ in range(10):
        i8 = rng.choice(len(p1), 8, replace=False)
        F, _ = fundamental_8pt(p1[i8], p2[i8])
        Fc, _ = cv2.findFundamentalMat(p1[i8].astype(np.float64), p2[i8].astype(np.float64), cv2.FM_8POINT)
        assert model_dist(F, Fc) < 1e-8
        i7 = rng.choice(len(p1), 7, replace=False)
        models, _ = fundamental_7pt(p1[i7], p2[i7])
        Fc, _ = cv2.findFundamentalMat(p1[i7].astype(np.float64), p2[i7].astype(np.float64), cv2.FM_7POINT)
        cv_models = [] if Fc is None else [Fc[3 * k: 3 * k + 3] for k in range(len(Fc) // 3)]
        assert len(models) == len(cv_models) >= 1
        for M in cv_models:
            assert min(model_dist(M, F) for F in models) < 1e-7
    F, _ = fundamental_8pt(p1[inl], p2[inl])
    Fc, _ = cv2.findFundamentalMat(p1[inl].astype(np.float64), p2[inl].astype(np.float64), cv2.FM_8POINT)
    assert model_dist(F, Fc) < 1e-8
    assert model_dist(F, s["F"]) < 1e-2                          # and the scene's own F is what the data say
    q = rig_scene(name, 300, planar=True, seed=seed, outlier_frac=0.0, sigma=0.5)
    for _ in range(10):
        i4 = rng.choice(300, 4, replace=False)
        H, _ = homography_dlt(q["p1"][i4], q["p2"][i4])
        Hc, _ = cv2.findHomography(q["p1"][i4].astype(np.float64), q["p2"][i4].astype(np.float64), 0)
        assert np.abs(H - Hc).max() / np.abs(Hc).max() < 1e-7      # cv2 solves the normal equations: half the digits
    H, _ = homography_dlt(q["p1"], q["p2"])
    assert np.median(h_error(H, q["p1"], q["p2"])) <= 1.1 * np.median(h_error(q["H"], q["p1"], q["p2"])) and model_dist(H, q["H"]) < 1e-2


@pytest.mark.parametrize("name", RIG_NAMES)
def test_reference_scores_equal_cv2(name):
    """Sampson error == cv2.sampsonDistance, the symmetric epipolar error == distances to cv2.computeCorrespondEpilines'
    lines, the transfer error == cv2.perspectiveTransform's residual, all to 1e-9 relative."""
    s = rig_scene(name, 200, seed=5, outlier_frac=0.3, sigma=1.0)
    p1, p2 = s["p1"].astype(np.float64), s["p2"].astype(np.float64)
    F = s["F"] * 3.7
    sym, samp = f_errors(F, p1, p2)
    cs = np.array([cv2.sampsonDistance(to_h(p1[i:i + 1]).T, to_h(p2[i:i + 1]).T, F) for i in range(len(p1))])
    assert np.abs(samp - cs).max() / cs.max() < 1e-9 and np.all(np.abs(samp - cs) <= 1e-9 * cs + 1e-12)
    l2 = cv2.computeCorrespondEpilines(p1.reshape(-1, 1, 2), 1, F).reshape(-1, 3)      # unit-normal lines
    l1 = cv2.computeCorrespondEpilines(p2.reshape(-1, 1, 2), 2, F).reshape(-1, 3)
    d2 = ((to_h(p2) * l2).sum(1)) ** 2
    d1 = ((to_h(p1) * l1).sum(1)) ** 2
    ref = np.maximum(d1, d2)
    assert np.all(np.abs(sym - ref) <= 1e-9 * ref + 1e-9)
    q = rig_scene(name, 200, planar=True, seed=6, sigma=1.0)
    e = h_error(q["H"], q["p1"], q["p2"])
    pc = cv2.perspectiveTransform(q["p1"].astype(np.float64).reshape(-1, 1, 2), q["H"]).reshape(-1, 2)
    ec = ((pc - q["p2"].astype(np.float64)) ** 2).sum(1)
    assert np.all(np.abs(e - ec) <= 1e-9 * ec + 1e-9)


@pytest.mark.parametrize("name", RIG_NAMES)
def test_reference_pose_equals_cv2_and_ground_truth(name):
    """E = K2^T F K1 + decomposition + cheirality vote == cv2.recoverPose on coordinates normalised by each image's own K
    (R, t to 1e-9, same mask, points to 1e-7 relative); on noise-free data it recovers the scene's motion, and swapping
    the two cameras does not."""
    s = rig_scene(name, 400, seed=7, outlier_frac=0.0, sigma=0.0)
    R, t, good, X, votes = relative_pose(s["F"], s["K1"], s["K2"], s["p1"], s["p2"])
    assert np.abs(R - s["R"]).max() < 1e-6 and np.abs(t - s["t"]).max() < 1e-6 and good.all()
    Rs = relative_pose(s["F"], s["K2"], s["K1"], s["p1"], s["p2"])[0]
    assert np.abs(Rs - s["R"]).max() > 1e-3
    n = rig_scene(name, 800, seed=8, outlier_frac=0.3, sigma=0.5)
    F, _ = fundamental_8pt(n["p1"][n["gt"]], n["p2"][n["gt"]])
    R, t, good, X, votes = relative_pose(F, n["K1"], n["K2"], n["p1"], n["p2"], mask=n["gt"])
    E = n["K2"].T @ F @ n["K1"]
    q1, q2 = normalise_pixels(n["p1"][n["gt"]], n["K1"]), normalise_pixels(n["p2"][n["gt"]], n["K2"])
    nc, Rc, tc, mc, Xc = cv2.recoverPose(E, q1, q2, np.eye(3), distanceThresh=50.0)
    assert sorted(votes)[-1] > sorted(votes)[-2] and int(good.sum()) == nc
    assert np.abs(R - Rc).max() < 1e-9 and np.abs(t - tc.ravel()).max() < 1e-9
    assert np.array_equal(good[n["gt"]], mc.ravel() > 0)
    Xc = (Xc[:3] / Xc[3]).T[mc.ravel() > 0]
    Xr = X[n["gt"]][mc.ravel() > 0]
    assert (np.abs(Xr - Xc).max(1) / np.abs(Xc).max(1)).max() < 1e-7
    assert np.abs(R - n["R"]).max() < 2e-2


@pytest.mark.parametrize("name", RIG_NAMES)
def test_reference_degenerate_samples_are_rank_deficient(name):
    """The degenerate samples the GPU test feeds the solvers really are rank-deficient: the design matrix of the
    reference loses one (repeated index, 3 collinear of 4) or two (8 coplanar) singular values, down to rounding."""
    for a, b, m, k, kind in _degenerate_cases(name):
        if k is None:                                       # identical points: no Hartley frame exists at all
            assert np.ptp(a[:m], axis=0).max() == 0 and np.ptp(b[:m], axis=0).max() == 0
            assert np.linalg.matrix_rank(epipolar_rows(a[:m].astype(np.float64), b[:m].astype(np.float64))) == 1
            continue
        sv = (fundamental_8pt if kind == "8pt" else fundamental_7pt if kind == "7pt" else homography_dlt)(a[:m], b[:m])[1]
        assert (sv[len(sv) - k:] <= 1e-12 * sv[0]).all() and sv[len(sv) - k - 1] > 1e-6 * sv[0], (kind, sv)


def _degenerate_cases(name):
    """(pts1, pts2, sample size, rank deficiency of the design matrix or None for identical points, solver): the sample is
    rows 0..m-1."""
    s = rig_scene(name, 64, seed=11, outlier_frac=0.0)
    p1, p2 = s["p1"], s["p2"]
    rep = np.r_[[0, 0], np.arange(1, 63)]                   # row 0 twice: m - 1 distinct points in an m-point sample
    a1, a2 = exact_affine_pairs(name, 64, seed=4)           # coplanar: x2 = A x1 + b exactly
    c1, _ = RIGS[name]
    line = np.column_stack([np.arange(3) * 0.125 * c1.w + c1.x0 + 8, np.arange(3) * 0.25 * c1.h + c1.y0 + 4])   # 3 collinear
    col1 = a1.astype(np.float64).copy()
    col1[:3] = line
    col2 = col1 @ np.array([[0.75, 0.125], [-0.25, 1.5]]).T + np.array([37.5, -12.25])
    same = np.tile(p1[:1], (64, 1)), np.tile(p2[:1], (64, 1))
    return [
        (p1[rep], p2[rep], 8, 1, "8pt"),
        (p1[rep], p2[rep], 7, 1, "7pt"),
        (a1, a2, 8, 2, "8pt"),
        (a1, a2, 7, 1, "7pt"),
        (p1[rep], p2[rep], 4, 2, "h"),
        (col1.astype(np.float32), col2.astype(np.float32), 4, 1, "h"),
        (same[0], same[1], 8, None, "8pt"),
        (same[0], same[1], 7, None, "7pt"),
        (same[0], same[1], 4, None, "h"),
    ]


# ====================================================================================================== kernels vs the reference (GPU)

THR = 3.0
# The kernels score in fp32 on raw pixel coordinates (division-free: num^2 <= thr^2 * |l|^2), so a decision can differ from
# the float64 one when the float64 error is within a rounding band of thr^2.  The band grows with the coordinates'
# magnitude; it is stated per pixel of the largest |coordinate| of the pair, at thr = 3 px.  Measured on a B200 with
# test_fp32_scoring_band_near_threshold: at most 6.6e-7 px^2 per pixel (5.1e-3 px^2 for H at 7680 wide; DESIGN.md §2
# lists every size), so 2e-6 leaves a margin of three.
FP32_BAND_PER_PX = 2e-6


def fp32_band(p1, p2):
    return FP32_BAND_PER_PX * max(np.abs(p1).max(), np.abs(p2).max())


def _rs():
    from sfm_b200 import ransac as rs
    return rs


def pack(pairs, cap=None):
    cap = cap or max(16, max(len(a) for a, _ in pairs))
    corr = np.zeros((len(pairs), cap, 4), np.float32)
    counts = np.zeros(len(pairs), np.int32)
    for k, (a, b) in enumerate(pairs):
        corr[k, : len(a), :2], corr[k, : len(a), 2:] = a, b
        counts[k] = len(a)
    return torch.from_numpy(corr).cuda(), torch.from_numpy(counts)


def sample_first(p1, p2, idx):
    """The correspondences reordered so that the sample `idx` is rows 0..len(idx)-1."""
    order = np.r_[idx, np.setdiff1d(np.arange(len(p1)), idx)]
    return p1[order], p2[order]


def run_sample(pairs, solver, score="sym_epipolar"):
    """Every pair's rows 0..7 as the minimal sample, repeated in every hypothesis (so the batch size does not matter), no
    LO, no early stop: the result is that sample's best model, or no model when it has no inlier.  Returns (model,
    n_inliers, mask) as numpy."""
    rs = _rs()
    corr, counts = pack(pairs)
    samples = np.tile(np.arange(8, dtype=np.uint32), (32, 1))
    kw = dict(samples=samples, max_iters=32, confidence=1.0, lo=False, thr=THR)
    vb = rs.verify_h_corr(corr, counts, **kw) if solver == "h" else rs.verify_corr(corr, counts, solver=solver, score=score, **kw)
    return vb.F.cpu().numpy(), vb.n_inliers.cpu().numpy(), vb.mask.cpu().numpy()


def assert_mask_is_float64_decision(mask, err, band):
    """mask == (err <= thr^2) wherever err is farther than `band` from thr^2.  Returns the largest |err - thr^2| of a
    decision that differs (0 when none does)."""
    m = np.asarray(mask).astype(bool)
    want = err <= THR * THR
    far = np.abs(err - THR * THR) > band
    assert np.array_equal(m[far], want[far]), f"{int((m[far] != want[far]).sum())} decisions differ outside +-{band:.2e} px^2"
    diff = m != want
    return float(np.abs(err[diff] - THR * THR).max()) if diff.any() else 0.0


@gpu_test
@pytest.mark.parametrize("name", RIG_NAMES)
def test_8pt_minimal_solver_matches_reference(name):
    """One explicit 8-point sample of noisy inliers per pair (their 8-point solution is not rank 2 by itself): F == the
    reference's normalised 8-point with its rank-2 projection to 1e-9 after unit-Frobenius scaling; F[2,2] == 1; the
    mask is the float64 decision on F.  A model with fewer inliers than the 8 points of its sample is no model."""
    s = rig_scene(name, 400, seed=21)
    p1, p2 = s["p1"], s["p2"]
    rng = np.random.default_rng(21)
    picks = [rng.choice(np.flatnonzero(s["gt"]), 8, replace=False) for _ in range(24)]
    pairs = [sample_first(p1, p2, idx) for idx in picks]
    F, n, mask = run_sample(pairs, "8pt")
    for k, idx in enumerate(picks):
        ref, _ = fundamental_8pt(p1[idx], p2[idx])
        a, b = pairs[k]
        if n[k] == 0:
            assert not F[k].any() and (f_errors(ref, a, b)[0] <= THR * THR + fp32_band(a, b)).sum() < 8
            continue
        assert F[k][2, 2] == 1.0 and n[k] == mask[k].sum()
        assert model_dist(F[k], ref) < 1e-9, (k, model_dist(F[k], ref))
        assert_mask_is_float64_decision(mask[k, : len(a)], f_errors(F[k], a, b)[0], fp32_band(a, b))
    assert (n > 0).sum() >= 20


@gpu_test
@pytest.mark.parametrize("name", RIG_NAMES)
def test_7pt_minimal_solver_returns_best_reference_root(name):
    """One explicit 7-point sample per pair: the returned F is one of the reference's cubic-root models.  For samples with
    three real, distinct roots and a winner that no fp32 rounding can overturn, it is THE winner (the root with the most
    float64 inliers), so a solver that loses roots picks the wrong model on some of them."""
    s = rig_scene(name, 400, seed=22, outlier_frac=0.2)
    p1, p2 = s["p1"], s["p2"]
    rng = np.random.default_rng(22)
    picks = [rng.choice(len(p1), 7, replace=False) for _ in range(64)]
    pairs = [sample_first(p1, p2, idx) for idx in picks]
    band = max(fp32_band(a, b) for a, b in pairs)
    F, n, mask = run_sample(pairs, "7pt")
    decisive = 0
    for k, idx in enumerate(picks):
        models, _ = fundamental_7pt(p1[idx], p2[idx])
        a, b = pairs[k]
        errs = [f_errors(M, a, b)[0] for M in models]
        if n[k] == 0:                                 # no root reaches the 7 inliers a model needs
            assert not F[k].any() and all((e <= THR * THR + band).sum() < 7 for e in errs)
            continue
        d = [model_dist(F[k], M) for M in models]
        assert n[k] >= 7 and min(d) < 1e-8, (k, d)
        if len(models) == 3 and min(model_dist(models[i], models[j]) for i, j in ((0, 1), (0, 2), (1, 2))) > 1e-3:
            lo_cnt = [int((e <= THR * THR - band).sum()) for e in errs]
            hi_cnt = [int((e <= THR * THR + band).sum()) for e in errs]
            w = int(np.argmax(lo_cnt))
            if all(lo_cnt[w] > hi_cnt[j] for j in range(3) if j != w):
                decisive += 1
                assert int(np.argmin(d)) == w, (k, d, lo_cnt, hi_cnt)
                assert lo_cnt[w] <= n[k] <= hi_cnt[w]
    assert decisive >= 6, decisive                    # enough three-root samples to catch a solver that loses roots


@gpu_test
@pytest.mark.parametrize("name", RIG_NAMES)
def test_4pt_homography_matches_reference(name):
    """One explicit 4-point sample of a planar scene per pair: H == the reference DLT to 1e-9 relative, H[2,2] == 1, the
    mask is the float64 transfer-error decision."""
    s = rig_scene(name, 400, planar=True, seed=23)
    p1, p2 = s["p1"], s["p2"]
    rng = np.random.default_rng(23)
    inl = np.flatnonzero(s["gt"])
    picks = [rng.choice(inl, 4, replace=False) for _ in range(24)]
    pairs = [sample_first(p1, p2, idx) for idx in picks]
    H, n, mask = run_sample(pairs, "h")
    for k, idx in enumerate(picks):
        ref, _ = homography_dlt(p1[idx], p2[idx])
        if n[k] == 0:             # rejected: the four points do not all keep one side of the line H sends to infinity
            w = to_h(p1[idx]) @ ref[2]
            assert not H[k].any() and not ((w > 0).all() or (w < 0).all())
            continue
        assert n[k] >= 4 and H[k][2, 2] == 1.0
        assert np.abs(H[k] - ref).max() / np.abs(ref).max() < 1e-9, (k, H[k], ref)
        a, b = pairs[k]
        assert_mask_is_float64_decision(mask[k, : len(a)], h_error(H[k], a, b), fp32_band(a, b))
    assert (n > 0).sum() >= 20


@gpu_test
@pytest.mark.parametrize("name", RIG_NAMES)
def test_degenerate_samples_give_no_model(name):
    """A repeated index, 8 (or 7) coplanar points for F, 3 collinear points of 4 for H, and identical points: the
    design matrix is rank-deficient (shown by the reference's singular values in
    test_reference_degenerate_samples_are_rank_deficient), so no model is returned: n_inliers == 0, F / H == 0, empty
    mask.  The coplanar and collinear samples are exact in float32; a sample that is degenerate only up to rounding is a
    (poor) regular sample and is not rejected."""
    cases = _degenerate_cases(name)
    for solver in ("8pt", "7pt", "h"):
        sel = [(a, b) for a, b, m, k, kind in cases if kind == solver]
        F, n, mask = run_sample(sel, solver)
        assert (n == 0).all() and not F.any() and not mask.any(), (solver, n)


def near_threshold(M, p1, p2, kind, rng, window=0.05):
    """Noise-free correspondences moved in image 2, each along its own random direction, until the float64 error of the
    model M reaches a random target within +-window px^2 of thr^2.  (Rounding to float32 moves the error a little more.)"""
    p1, p2 = np.asarray(p1, np.float64), np.asarray(p2, np.float64)
    ang = rng.uniform(0.0, 2.0 * np.pi, len(p1))
    d = np.column_stack([np.cos(ang), np.sin(ang)])
    target = THR * THR + rng.uniform(-window, window, len(p1))
    err = {"sym_epipolar": lambda q: f_errors(M, p1, q)[0], "sampson": lambda q: f_errors(M, p1, q)[1],
           "homography": lambda q: h_error(M, p1, q)}[kind]
    step = np.full(len(p1), THR)
    for _ in range(6):
        step *= np.sqrt(target / np.maximum(err(p2 + step[:, None] * d), 1e-30))
    return (p2 + step[:, None] * d).astype(np.float32)


@gpu_test
@pytest.mark.parametrize("kind", ["sym_epipolar", "sampson", "homography"])
def test_fp32_scoring_band_near_threshold(kind):
    """The fp32 inlier test where it is hardest: for every camera size, one model fixed by an explicit noise-free sample
    and ~8,000 correspondences whose float64 error is within 0.05 px^2 of thr^2.  Every decision farther than the fp32
    band from thr^2 is the float64 decision.  Prints the largest |err - thr^2| of a differing decision per rig: the
    figure FP32_BAND_PER_PX is set from (with a margin)."""
    rng = np.random.default_rng(61)
    pairs = []
    for k, name in enumerate(RIG_NAMES):
        s = rig_scene(name, 8192, planar=kind == "homography", seed=61 + k, sigma=0.0, outlier_frac=0.0)
        p1, p2 = s["p1"], s["p2"]
        M = homography_dlt(p1[:4], p2[:4])[0] if kind == "homography" else fundamental_8pt(p1[:8], p2[:8])[0]
        q2 = p2.copy()
        q2[8:] = near_threshold(M, p1[8:], p2[8:], kind, rng)
        pairs.append((p1, q2))
    M, n, mask = run_sample(pairs, "h" if kind == "homography" else "8pt", score="sampson" if kind == "sampson" else "sym_epipolar")
    worst = {}
    for k, (a, b) in enumerate(pairs):
        err = h_error(M[k], a, b) if kind == "homography" else f_errors(M[k], a, b)[kind == "sampson"]
        assert (np.abs(err[8:] - THR * THR) < 0.1).mean() > 0.95          # the data really sit at the threshold
        worst[RIG_NAMES[k]] = assert_mask_is_float64_decision(mask[k, : len(a)], err, fp32_band(a, b))
        assert n[k] == mask[k].sum()
    print(f"{kind}: largest |err - thr^2| of a differing decision, px^2: {worst}")


def _full_run_scenes():
    return [rig_scene(name, 3000, seed=31 + k, sigma=1.0, outlier_frac=0.4) for k, name in enumerate(RIG_NAMES)]


# LO's refit is fitted on the inliers of the previous model and scored on its own: on its final inlier set its algebraic
# residual may exceed that of the least-squares refit on exactly that set, by a little
LO_RESIDUAL_TOL = 1.25


@gpu_test
@pytest.mark.parametrize("score", ["sym_epipolar", "sampson"])
def test_full_run_mask_is_the_float64_decision(score):
    """Seeded RANSAC-F at every camera size, with and without LO: n_inliers == mask.sum(), F[2,2] == 1, and the mask
    equals `float64 error(F) <= thr^2` for every correspondence outside the fp32 band.  LO never loses inliers against
    the same-seed run without it; when it keeps the minimal model the results are identical, otherwise its F fits its
    own inliers about as well as the reference's least-squares refit on that set."""
    rs = _rs()
    scenes = _full_run_scenes()
    corr, counts = pack([(s["p1"], s["p2"]) for s in scenes])
    kw = dict(thr=THR, confidence=0.99, max_iters=1024, solver="7pt", score=score, seed=5)
    runs = {lo: rs.verify_corr(corr, counts, lo=lo, **kw) for lo in (False, True)}
    out = {lo: (v.F.cpu().numpy(), v.n_inliers.cpu().numpy(), v.mask.cpu().numpy()) for lo, v in runs.items()}
    worst = {}
    for k, s in enumerate(scenes):
        p1, p2, n = s["p1"], s["p2"], len(s["p1"])
        for lo in (False, True):
            F, ninl, mask = out[lo][0][k], out[lo][1][k], out[lo][2][k, :n]
            assert ninl >= 8 and ninl == mask.sum() and F[2, 2] == 1.0
            err = f_errors(F, p1, p2)[0 if score == "sym_epipolar" else 1]
            worst[(RIG_NAMES[k], lo)] = assert_mask_is_float64_decision(mask, err, fp32_band(p1, p2))
        (F0, n0, m0), (F1, n1, m1) = ((out[lo][0][k], out[lo][1][k], out[lo][2][k, :n]) for lo in (False, True))
        assert n1 >= n0
        if n1 == n0:
            assert np.array_equal(F1, F0) and np.array_equal(m1, m0)
        else:
            inl = m1.astype(bool)
            ref, _ = fundamental_8pt(p1[inl], p2[inl])
            r_lo, r_ref = algebraic_residual(F1, p1[inl], p2[inl]), algebraic_residual(ref, p1[inl], p2[inl])
            assert r_lo <= LO_RESIDUAL_TOL * r_ref, (RIG_NAMES[k], r_lo, r_ref)
    print(f"{score}: largest |err - thr^2| of a differing decision, px^2: {worst}")


@gpu_test
def test_full_run_homography_mask_is_the_float64_decision():
    """Seeded RANSAC-H on planar scenes at every camera size, with and without LO: the mask is the float64 transfer-error
    decision outside the fp32 band, n_inliers == mask.sum(), H[2,2] == 1, LO never loses inliers."""
    rs = _rs()
    scenes = [rig_scene(name, 3000, planar=True, seed=51 + k, sigma=1.0, outlier_frac=0.4) for k, name in enumerate(RIG_NAMES)]
    corr, counts = pack([(s["p1"], s["p2"]) for s in scenes])
    res = {lo: rs.verify_h_corr(corr, counts, thr=THR, confidence=0.995, max_iters=1024, lo=lo, seed=5) for lo in (False, True)}
    worst = {}
    for k, s in enumerate(scenes):
        p1, p2, n = s["p1"], s["p2"], len(s["p1"])
        for lo, v in res.items():
            H, ninl, mask = v.F[k].cpu().numpy(), int(v.n_inliers[k]), v.mask[k, :n].cpu().numpy()
            assert ninl >= 8 and ninl == mask.sum() and H[2, 2] == 1.0
            worst[(RIG_NAMES[k], lo)] = assert_mask_is_float64_decision(mask, h_error(H, p1, p2), fp32_band(p1, p2))
        assert int(res[True].n_inliers[k]) >= int(res[False].n_inliers[k])
    print(f"homography: largest |err - thr^2| of a differing decision, px^2: {worst}")


@gpu_test
def test_pose_with_two_cameras_vs_reference_cv2_and_oracle():
    """recover_pose_corr with camera_rows(K1, K2), K1 != K2, at every camera size: R, t == the reference to 1e-9, the same
    cheirality mask, points to 1e-5 relative; the same against cv2.recoverPose on coordinates normalised by each image's
    own K; bit for bit against oracle.two_view_pose; and the scene's true rotation."""
    from oracle import ransac_oracle as ro

    rs = _rs()
    scenes = [rig_scene(name, 2000, seed=41 + k) for k, name in enumerate(RIG_NAMES)]
    corr, counts = pack([(s["p1"], s["p2"]) for s in scenes])
    vb = rs.verify_corr(corr, counts, thr=THR, confidence=0.99, max_iters=1024, solver="7pt", lo=True, seed=5)
    cam = np.concatenate([rs.camera_rows(s["K1"], s["K2"]) for s in scenes])
    assert not np.array_equal(cam[:, :4], cam[:, 4:])
    pb = rs.recover_pose_corr(corr, counts, vb.F, cam, mask=vb.mask)
    F, fm = vb.F.cpu().numpy(), vb.mask.cpu().numpy()
    R, t, ng, pm, X = (x.cpu().numpy() for x in (pb.R, pb.t, pb.n_good, pb.mask, pb.points))
    for k, s in enumerate(scenes):
        p1, p2, n = s["p1"], s["p2"], len(s["p1"])
        inl = fm[k, :n].astype(bool)
        Rr, tr, good, Xr, votes = relative_pose(F[k], s["K1"], s["K2"], p1, p2, mask=inl)
        assert sorted(votes)[-1] > sorted(votes)[-2]                 # the vote is not a tie
        assert np.abs(R[k] - Rr).max() < 1e-9 and np.abs(t[k] - tr).max() < 1e-9, RIG_NAMES[k]
        assert np.array_equal(pm[k, :n].astype(bool), good) and ng[k] == good.sum() and (pm[k, n:] == 0).all()
        assert not X[k, :n][~good].any()
        assert (np.abs(X[k, :n][good] - Xr[good]).max(1) / np.abs(Xr[good]).max(1)).max() < 1e-5
        E = s["K2"].T @ F[k] @ s["K1"]
        nc, Rc, tc, mc, _ = cv2.recoverPose(E, normalise_pixels(p1[inl], s["K1"]), normalise_pixels(p2[inl], s["K2"]), np.eye(3),
                                            distanceThresh=50.0)
        assert ng[k] == nc and np.abs(R[k] - Rc).max() < 1e-9 and np.abs(t[k] - tc.ravel()).max() < 1e-9
        assert np.array_equal(pm[k, :n][inl], (mc.ravel() > 0).astype(np.uint8))
        on, oR, ot, _, om, oX = ro.two_view_pose(p1, p2, F[k], cam[k], mask=fm[k, :n])
        assert ng[k] == on and np.array_equal(R[k], oR) and np.array_equal(t[k], ot)
        assert np.array_equal(pm[k, :n], om) and np.array_equal(X[k, :n], oX)
        assert np.abs(R[k] - s["R"]).max() < 2e-2 and np.abs(t[k] - s["t"]).max() < 5e-2, RIG_NAMES[k]


@gpu_test
def test_pipeline_uses_each_images_own_camera():
    """match_and_verify(intrinsics=Ks) with a different K for every image, over ordered pairs (both (i, j) and (j, i)):
    every pair's R, t, n_pose, in_front and points3d equal recover_pose_corr with camera_rows(Ks[i], Ks[j]) on that pair's
    own matches, inlier mask and F -- so the pair's camera row is (image i's camera, image j's camera), in that order."""
    import sfm_b200
    from sfm_b200 import synth

    rs = _rs()
    sc = synth.make_scene(4, 1024, seed=8)
    bank = sfm_b200.DescriptorBank(4, 1024)
    bank.put(0, sc.desc, xy=sc.xy)
    pairs = sfm_b200.ordered_pairs(4)
    Ks = np.stack([np.array([[f, 0.0, cx], [0.0, f * a, cy], [0.0, 0.0, 1.0]])
                   for f, a, cx, cy in ((1000.0, 1.0, 960.0, 540.0), (1150.0, 1.01, 930.0, 560.0),
                                        (880.0, 0.99, 990.0, 525.0), (1300.0, 1.0, 955.0, 548.0))])
    h = sfm_b200.match_and_verify(bank, pairs, fetch=True, max_iters=256, seed=3, lo=True, intrinsics=Ks).to_host()
    for p, (i, j) in enumerate(pairs):
        sl = slice(h["offsets"][p], h["offsets"][p + 1])
        q, t = h["matches"][sl, 0], h["matches"][sl, 1]
        corr, counts = pack([(sc.xy[i][q], sc.xy[j][t])], cap=len(q))
        mask = torch.from_numpy(h["inlier"][sl][None].copy())
        pb = rs.recover_pose_corr(corr, counts, torch.from_numpy(h["F"][p][None].copy()), rs.camera_rows(Ks[i], Ks[j]), mask=mask)
        assert h["n_pose"][p] == int(pb.n_good[0]) > 0, (i, j)
        assert np.array_equal(h["R"][p], pb.R[0].cpu().numpy()) and np.array_equal(h["t"][p], pb.t[0].cpu().numpy()), (i, j)
        assert np.array_equal(h["in_front"][sl], pb.mask[0].cpu().numpy()), (i, j)
        assert np.array_equal(h["points3d"][sl], pb.points[0].cpu().numpy()), (i, j)
