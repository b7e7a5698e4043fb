"""CPU checks of registration: the parameter struct as the header declares it, the C-ABI argument checks of sfm_pnp_gather and
sfm_pnp_ransac (all before any CUDA call), the C oracle's P3P against cv2.solveP3P (P3P and AP3P), its whole estimate against
cv2.solvePnPRansac + cv2.solvePnPRefineLM, and the numpy gather oracle against a direct restatement of its definition."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import pnp_oracle as po

cv2 = pytest.importorskip("cv2")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["max_error", "confidence", "seed", "max_iters", "min_inliers", "min_inlier_ratio", "refine_iters", "reserved"]
K = np.array([[1000.0, 0.0, 960.0], [0.0, 1000.0, 540.0], [0.0, 0.0, 1.0]])


def test_params_struct_matches_header(tmp_path):
    from sfm_b200 import _lib

    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sfm_b200.h"\nint main(void){printf("%zu", sizeof(sfm_pnp_params));'
                   + "".join(f'printf(" %zu", offsetof(sfm_pnp_params, {f}));' for f in FIELDS) + "return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    for mirror in (_lib.PnpParams, po.PnpParams):
        assert [f[0] for f in mirror._fields_] == FIELDS
        assert [C.sizeof(mirror)] + [getattr(mirror, f).offset for f in FIELDS] == got
    assert got[0] == 64


def test_entry_points_reject_bad_arguments_without_a_gpu():
    """Every rejection returns SFM_ERR_ARG with its message before any CUDA call (pointers are fake and never read)."""
    from sfm_b200 import _lib
    from sfm_b200 import pnp

    L = _lib.lib()
    err = lambda: L.sfm_last_error().decode()  # noqa: E731

    def ransac(n_images=3, n_query=2, stride=64, prm=True, null=None, **fields):
        p = pnp.pnp_params()
        for k, v in fields.items():
            setattr(p, k, v)
        ptrs = {k: 0x1000 * (i + 1) for i, k in enumerate(("cams", "image", "xy", "X", "count", "pose", "ninl", "status", "mask", "counts"))}
        if null:
            ptrs[null] = None
        return L.sfm_pnp_ransac(n_images, ptrs["cams"], ptrs["image"], n_query, ptrs["xy"], ptrs["X"], stride, ptrs["count"],
                                C.byref(p) if prm else None, ptrs["pose"], ptrs["ninl"], ptrs["status"], ptrs["mask"], None, ptrs["counts"], None)

    assert ransac(prm=False) == -1 and "NULL params" in err()
    for name in ("cams", "image", "xy", "X", "count", "pose", "ninl", "status", "mask", "counts"):
        assert ransac(null=name) == -1 and "sfm_pnp_ransac: NULL argument" in err(), name
    assert ransac(n_images=0) == -1 and "positive" in err()
    assert ransac(stride=0) == -1 and "positive" in err()
    assert ransac(n_query=-1) == -1 and "non-negative" in err()
    assert ransac(max_iters=0) == -1 and "max_iters must be positive" in err()
    assert ransac(min_inliers=2) == -1 and "min_inliers must be at least 3, got 2" in err()
    for r in (-0.1, 1.5, float("nan")):
        assert ransac(min_inlier_ratio=r) == -1 and "min_inlier_ratio" in err(), r
    for r in (-1, 1001):
        assert ransac(refine_iters=r) == -1 and "refine_iters" in err(), r
    for e in (0.0, -1.0, float("nan"), float("inf")):
        assert ransac(max_error=e) == -1 and "max_error" in err(), e

    def gather(n_images=3, S=100, stride=128, max_tracks=10, n_query=2, null=None, xy=0x3000):
        ptrs = {k: 0x1000 * (i + 8) for i, k in enumerate(("track_of", "tc", "ps", "X", "image", "oxy", "oX", "of", "oc"))}
        if null:
            ptrs[null] = None
        return L.sfm_pnp_gather(n_images, S, ptrs["track_of"], ptrs["tc"], max_tracks, ptrs["ps"], ptrs["X"], xy, stride, ptrs["image"],
                                n_query, ptrs["oxy"], ptrs["oX"], ptrs["of"], ptrs["oc"], None)

    for name in ("track_of", "tc", "ps", "X", "image", "oxy", "oX", "of", "oc"):
        assert gather(null=name) == -1 and "sfm_pnp_gather: NULL argument" in err(), name
    assert gather(xy=None) == -1 and "NULL argument" in err()
    assert gather(n_images=0) == -1 and "positive" in err()
    assert gather(S=0) == -1 and "positive" in err()
    assert gather(n_images=65536, S=32768, stride=32768) == -1 and "2^31" in err()
    assert gather(stride=99) == -1 and "xy_stride" in err()
    assert gather(max_tracks=-1) == -1 and "negative" in err()
    assert gather(n_query=-1) == -1 and "negative" in err()
    assert gather(xy=0x3004) == -1 and "aligned" in err()
    for bad in (dict(min_inliers=2), dict(max_error=0.0), dict(min_inlier_ratio=2.0), dict(refine_iters=-1), dict(max_iters=0)):
        with pytest.raises(ValueError):
            pnp.pnp_params(**bad)


def random_rotation(rng):
    q = rng.normal(size=4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def test_oracle_p3p_equals_cv2():
    """Well-conditioned triplets (camera-frame points spread over the image at depth 3-6): every cv2 pose that puts the three
    points in front of the camera is an oracle root and every oracle root is such a cv2 pose, within 1e-6 (max abs difference
    of R and t); the true pose is always among the roots.  (AP3P also returns poses with a negative depth; the oracle drops
    those by contract.)"""
    rng = np.random.default_rng(0)
    matched = 0
    for _ in range(200):
        R, t = random_rotation(rng), rng.normal(size=3)
        Xc = np.stack([np.r_[rng.uniform(-1, 1, 2) * [0.9, 0.5], 1.0] * rng.uniform(3, 6) for _ in range(3)])
        Xw = (Xc - t) @ R
        nxy = Xc[:, :2] / Xc[:, 2:]
        roots = po.p3p(nxy, Xw)
        assert 1 <= len(roots) <= 4
        assert min(np.abs(Ro - R).max() + np.abs(to - t).max() for Ro, to in roots) < 1e-6
        for flag in (cv2.SOLVEPNP_P3P, cv2.SOLVEPNP_AP3P):
            _, rv, tv = cv2.solveP3P(Xw.reshape(3, 1, 3), (nxy * 1000 + [960, 540]).reshape(3, 1, 2), K, None, flags=flag)
            cv = [(cv2.Rodrigues(r)[0], np.ravel(tt)) for r, tt in zip(rv, tv)]
            cv = [(Rc, tc) for Rc, tc in cv if np.all(Xw @ Rc[2] + tc[2] > 0)]
            for Rc, tc in cv:
                assert min(np.abs(Rc - Ro).max() + np.abs(tc - to).max() for Ro, to in roots) < 1e-6
            for Ro, to in roots:
                assert min([np.abs(Rc - Ro).max() + np.abs(tc - to).max() for Rc, tc in cv] + [1.0]) < 1e-6
            matched += len(cv)
    assert matched > 400


def scene_query(seed, M=400, outlier_frac=0.3, noise=0.5):
    """M points at depth 4-8 seen by a random camera with `noise` px of pixel noise; a fraction moved 80-300 px away."""
    rng = np.random.default_rng(seed)
    R, t = random_rotation(rng), rng.normal(size=3)
    Xc = np.stack([rng.uniform(-2, 2, M), rng.uniform(-1.2, 1.2, M), rng.uniform(4, 8, M)], 1)
    Xw = (Xc - t) @ R
    px = Xc[:, :2] / Xc[:, 2:] * 1000 + [960, 540] + rng.normal(0, noise, (M, 2))
    out = rng.random(M) < outlier_frac
    px[out] += rng.choice([-1, 1], (out.sum(), 2)) * rng.uniform(80, 300, (out.sum(), 2))
    return px.astype(np.float32), Xw, out, R, t


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("outlier_frac", [0.0, 0.3, 0.6])
def test_oracle_estimate_equals_cv2_ransac_and_refine_lm(seed, outlier_frac):
    px, Xw, out, _, _ = scene_query(seed, outlier_frac=outlier_frac)
    cams = np.array([[1000.0, 1000.0, 960.0, 540.0] + [0.0] * 12])
    o = po.pnp_ransac(px[None], Xw[None], [len(px)], cams, [0], seed=seed)
    ok, rv, tv, inl = cv2.solvePnPRansac(Xw, px.astype(np.float64), K, None, reprojectionError=12.0, iterationsCount=2000, confidence=0.9999,
                                         flags=cv2.SOLVEPNP_P3P)
    assert ok
    rv, tv = cv2.solvePnPRefineLM(Xw[inl.ravel()], px.astype(np.float64)[inl.ravel()], K, None, rv, tv)
    assert o["status"].tolist() == [0] and o["counts"].tolist() == [1, 0, 0, 0, 0]
    mask = o["mask"][0].astype(bool)
    assert np.array_equal(mask, ~out) and sorted(np.nonzero(mask)[0]) == sorted(inl.ravel())
    assert o["n_inliers"][0] == (~out).sum()
    np.testing.assert_allclose(o["pose"][0, :9].reshape(3, 3), cv2.Rodrigues(rv)[0], rtol=0, atol=1e-6)
    np.testing.assert_allclose(o["pose"][0, 9:], tv.ravel(), rtol=0, atol=1e-6)


def test_oracle_statuses():
    """Invalid image and focal length, too few points, no model (collinear world points), too few inliers, registered."""
    px, Xw, _, _, _ = scene_query(1, M=64, outlier_frac=0.0)
    cams = np.tile(np.array([1000.0, 1000.0, 960.0, 540.0] + [0.0] * 12), (3, 1))
    cams[1, 0] = 0.0
    line = np.zeros((64, 3))
    line[:, 2] = np.linspace(4, 8, 64)
    xy = np.stack([px, px, px, px, px, px])
    X = np.stack([Xw, Xw, Xw, Xw, line, Xw])
    o = po.pnp_ransac(xy, X, [64, 64, 64, 2, 64, 64], cams, [5, 1, -1, 0, 0, 2], min_inliers=65, max_iters=100)
    assert o["status"].tolist() == [4, 4, 4, 1, 2, 3] and o["counts"].tolist() == [0, 1, 1, 1, 3]
    assert o["n_inliers"].tolist()[:5] == [0] * 5 and o["n_inliers"][5] == 64 and not o["mask"].any() and not o["pose"].any()
    assert o["iters"].tolist()[:4] == [0] * 4 and o["iters"][4] == 100
    o = po.pnp_ransac(xy[5:], X[5:], [64], cams, [2], min_inliers=64, min_inlier_ratio=1.0)
    assert o["status"].tolist() == [0] and o["mask"].all()


def _gather_by_definition(track_of, n_tracks, point_status, X, xy, image):
    n_images, S = track_of.shape
    rows = []
    for img in image:
        r = []
        if 0 <= img < n_images:
            for f in range(S):
                k = int(track_of[img, f])
                if 0 <= k < n_tracks and point_status[k] == 0:
                    r.append((f, xy[img, f], X[k]))
        rows.append(r)
    return rows


def test_numpy_gather_oracle_equals_its_definition():
    rng = np.random.default_rng(3)
    n_images, S, n_cap = 7, 300, 900
    track_of = rng.integers(-1, n_cap + 50, (n_images, S)).astype(np.int32)
    point_status = rng.integers(0, 5, n_cap).astype(np.uint8) * (rng.random(n_cap) < 0.4)
    X = rng.normal(size=(n_cap, 3))
    xy = rng.uniform(0, 1000, (n_images, S + 20, 2)).astype(np.float32)
    image = np.array([0, 3, 6, 7, -1, 3])
    for n_tracks in (0, 500, n_cap):
        got = po.gather(track_of, n_tracks, point_status, X, xy, image)
        want = _gather_by_definition(track_of, n_tracks, point_status, X, xy, image)
        for q, rows in enumerate(want):
            n = len(rows)
            assert got["count"][q] == n
            assert got["feature"][q, :n].tolist() == [f for f, _, _ in rows]
            assert np.array_equal(got["xy"][q, :n], np.array([p for _, p, _ in rows]).reshape(n, 2))
            assert np.array_equal(got["X"][q, :n], np.array([x for _, _, x in rows]).reshape(n, 3))
        assert got["count"][4] == 0 and got["count"][3] == 0 and (n_tracks == 0) == (got["count"].sum() == 0)
