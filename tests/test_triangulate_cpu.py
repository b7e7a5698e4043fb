"""CPU checks of the track triangulation: the parameter struct as the header declares it, the C-ABI argument checks of
sfm_triangulate_tracks (all before any CUDA call), the C oracle against an independent numpy float64 reference (SVD DLT) on
random well-conditioned tracks, the camera table of the public call, and the scene points of the synthetic scenes."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import triangulate_oracle as tro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["max_error", "min_angle", "confidence", "seed", "max_iters", "min_inliers", "reserved"]


def test_params_struct_matches_header(tmp_path):
    """sizeof and every field offset of sfm_triangulate_params, from the header compiled by the C compiler, equal the ctypes
    mirrors of the product and of the oracle."""
    from sfm_b200 import _lib

    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sfm_b200.h"\nint main(void){printf("%zu", sizeof(sfm_triangulate_params));'
                   + "".join(f'printf(" %zu", offsetof(sfm_triangulate_params, {f}));' for f in FIELDS) + "return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    for mirror in (_lib.TriangulateParams, tro.TriangulateParams):
        assert [f[0] for f in mirror._fields_] == FIELDS
        assert [C.sizeof(mirror)] + [getattr(mirror, f).offset for f in FIELDS] == got
    assert got[0] == 64


def test_entry_point_rejects_bad_arguments_without_a_gpu():
    """Every rejection returns SFM_ERR_ARG with its message before any CUDA call (pointers are fake and never read)."""
    from sfm_b200 import _lib

    L = _lib.lib()
    err = lambda: L.sfm_last_error().decode()  # noqa: E731

    def call(n_images=3, S=100, stride=256, max_tracks=10, prm=True, null=None, **fields):
        p = _lib.TriangulateParams(4.0, 1.5, 0.999, 0, 500, 2)
        for k, v in fields.items():
            setattr(p, k, v)
        ptrs = {k: 0x1000 * (i + 1) for i, k in enumerate(("offsets", "obs", "tc", "xy", "cams", "X", "ninl", "status", "oin", "oerr", "counts"))}
        if null:
            ptrs[null] = None
        return L.sfm_triangulate_tracks(n_images, S, ptrs["offsets"], ptrs["obs"], ptrs["tc"], max_tracks, ptrs["xy"], stride, ptrs["cams"],
                                        None, C.byref(p) if prm else None, ptrs["X"], ptrs["ninl"], ptrs["status"], ptrs["oin"],
                                        ptrs["oerr"], ptrs["counts"], None)

    assert call(prm=False) == -1 and "NULL params" in err()
    for name in ("offsets", "obs", "tc", "xy", "cams", "X", "ninl", "status", "oin", "oerr", "counts"):
        assert call(null=name) == -1 and "sfm_triangulate_tracks: NULL argument" in err(), name
    assert call(n_images=0) == -1 and "positive" in err()
    assert call(S=-1) == -1 and "positive" in err()
    assert call(n_images=65536, S=32768, stride=32768) == -1 and "2^31" in err()
    assert call(stride=99) == -1 and "xy_stride" in err()
    assert call(max_tracks=-1) == -1 and "capacity" in err()
    assert call(max_iters=0) == -1 and "max_iters must be positive" in err()
    assert call(max_iters=-5) == -1 and "max_iters" in err()
    assert call(min_inliers=1) == -1 and "min_inliers must be at least 2, got 1" in err()
    for a in (-0.5, 90.0, 120.0, float("nan")):
        assert call(min_angle=a) == -1 and "min_angle" in err(), a
    for e in (0.0, -1.0, float("nan"), float("inf")):
        assert call(max_error=e) == -1 and "max_error" in err(), e


# ------------------------------------------------------------------ independent float64 reference (numpy SVD)
def _rng_u32(seed, pair, hyp, ctr):
    m = (1 << 64) - 1
    x = (seed + 0x9E3779B97F4A7C15 * ((pair << 32) | hyp)) & m
    x ^= (0xD1B54A32D192ED03 * (ctr + 1)) & m
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & m
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & m
    x ^= x >> 31
    return x >> 32


def _draw_pair(seed, k, h, M):
    idx = []
    for j in range(2):
        v = 0
        for attempt in range(16):
            v = (_rng_u32(seed, k, h, j * 16 + attempt) * M) >> 32
            if v not in idx:
                break
        idx.append(v)
    return idx


def _should_stop(best, M, done, confidence):
    if confidence >= 1.0 or best <= 0:
        return False
    q = 1.0 - (best / M) ** 2
    return q <= 0 or q ** done <= 1.0 - confidence


def _batch(done):
    return 32 if done < 64 else (64 if done < 128 else 128)


def _dlt(P, x, f):
    """SVD of the stacked DLT rows: P [n,3,4] ([R|t]), x [n,2] normalised, each row scaled by its view's focal length f [n,2]."""
    A = np.concatenate([(x[:, :1] * P[:, 2] - P[:, 0]) * f[:, :1], (x[:, 1:] * P[:, 2] - P[:, 1]) * f[:, 1:]])
    v = np.linalg.svd(A)[2][-1]
    return None if not abs(v[3]) > 1e-300 else v[:3] / v[3]


def reference_triangulate(offsets, obs, xy, cams, registered, *, max_error, min_angle, max_iters, confidence, seed, min_inliers):
    n_images, S = xy.shape[:2]
    f, c = cams[:, :2], cams[:, 2:4]
    Rt = np.concatenate([cams[:, 4:13].reshape(-1, 3, 3), cams[:, 13:16, None]], axis=2)
    centers = -np.einsum("nji,nj->ni", Rt[:, :, :3], Rt[:, :, 3])
    out = []
    for k in range(len(offsets) - 1):
        o = obs[offsets[k]: offsets[k + 1]]
        if np.any((o[:, 0] < 0) | (o[:, 0] >= n_images) | (o[:, 1] < 0) | (o[:, 1] >= S)):
            out.append((4, None, None))
            continue
        use = np.ones(len(o), bool) if registered is None else registered[o[:, 0]] != 0
        img = o[use, 0]
        xn = (xy[img, o[use, 1]].astype(np.float64) - c[img]) / f[img]
        M = len(img)
        if M < 2:
            out.append((1, None, None))
            continue

        def inliers(X):
            p = Rt[img, :, :3] @ X + Rt[img, :, 3]
            with np.errstate(divide="ignore", invalid="ignore"):
                e2 = (((p[:, :2] / p[:, 2:]) - xn) * f[img]) ** 2
            return (p[:, 2] > 0) & (e2.sum(1) <= max_error ** 2)

        best, X, done = -1, None, 0
        while done < max_iters:
            nb = min(_batch(done), max_iters - done)
            for h in range(done, done + nb):
                a, b = sorted(_draw_pair(seed, k, h, M))
                Xh = _dlt(Rt[img[[a, b]]], xn[[a, b]], f[img[[a, b]]])
                if Xh is None or not (Rt[img[a], 2, :3] @ Xh + Rt[img[a], 2, 3] > 0) or not (Rt[img[b], 2, :3] @ Xh + Rt[img[b], 2, 3] > 0):
                    continue
                da, db = Xh - centers[img[a]], Xh - centers[img[b]]
                if not np.dot(da, db) / np.linalg.norm(da) / np.linalg.norm(db) <= np.cos(np.deg2rad(min_angle)):
                    continue
                n = int(inliers(Xh).sum())
                if n > best:
                    best, X = n, Xh
            done += nb
            if _should_stop(best, M, done, confidence):
                break
        if best < 0:
            out.append((2, None, None))
            continue
        cur = best
        for _ in range(2):
            if cur < 2:
                break
            m = inliers(X)
            Xr = _dlt(Rt[img[m]], xn[m], f[img[m]])
            if Xr is None or inliers(Xr).sum() < cur:
                break
            X, cur = Xr, int(inliers(Xr).sum())
        full = np.zeros(len(o), bool)
        full[np.nonzero(use)[0]] = inliers(X)
        out.append((0 if cur >= min_inliers else 3, X, full))
    return out


def random_scene_tracks(seed, n_tracks=60, n_images=12):
    """Tracks of random scene points seen by the synthetic arc cameras (0.5 px noise), up to 40 % outlier observations,
    some unregistered images, a few tracks too short to triangulate."""
    from sfm_b200 import synth

    rng = np.random.default_rng(seed)
    Ps = synth.make_cameras(n_images, baseline=3.0)
    Kinv = np.linalg.inv(synth.K_INTR)
    Rt = np.einsum("ij,njk->nik", Kinv, Ps)
    K = synth.K_INTR
    cams = np.concatenate([np.tile([K[0, 0], K[1, 1], K[0, 2], K[1, 2]], (n_images, 1)), Rt[:, :, :3].reshape(-1, 9), Rt[:, :, 3]], axis=1)
    S = 64
    xy = rng.uniform([0, 0], [1920, 1080], (n_images, S, 2)).astype(np.float32)
    offsets, obs, used = [0], [], np.zeros((n_images, S), bool)
    for k in range(n_tracks):
        X = np.array([rng.uniform(-2, 2), rng.uniform(-2, 2), rng.uniform(4, 8)])
        L = int(rng.integers(1, 11)) if k % 7 == 0 else int(rng.integers(2, n_images + 1))
        imgs = np.sort(rng.choice(n_images, L, replace=False))
        out_frac = rng.uniform(0.0, 0.4)
        for i in imgs:
            f = int(rng.choice(np.nonzero(~used[i])[0]))
            used[i, f] = True
            if rng.random() >= out_frac:
                p = Ps[i] @ np.append(X, 1.0)
                xy[i, f] = (p[:2] / p[2] + rng.normal(0, 0.5, 2)).astype(np.float32)
            obs.append((i, f))
        offsets.append(len(obs))
    registered = np.ones(n_images, np.uint8)
    registered[rng.choice(n_images, 2, replace=False)] = 0
    return np.array(offsets, np.int64), np.array(obs, np.int32).reshape(-1, 2), xy, cams, registered


@pytest.mark.parametrize("seed", range(3))
@pytest.mark.parametrize("min_angle,max_error", [(1.5, 4.0), (0.0, 2.0)])
def test_oracle_equals_numpy_svd_reference(seed, min_angle, max_error):
    offsets, obs, xy, cams, registered = random_scene_tracks(seed)
    prm = dict(max_error=max_error, min_angle=min_angle, max_iters=500, confidence=0.999, seed=seed, min_inliers=3)
    for reg in (None, registered):
        got = tro.triangulate_tracks(offsets, obs, xy, cams, reg, **prm)
        ref = reference_triangulate(offsets, obs, xy, cams, reg, **prm)
        statuses = [s for s, _, _ in ref]
        assert got["status"].tolist() == statuses
        assert got["counts"].tolist() == [statuses.count(s) for s in range(5)]
        assert statuses.count(0) > len(statuses) // 2
        for k, (s, X, inl) in enumerate(ref):
            seg = slice(offsets[k], offsets[k + 1])
            if s != 0:
                assert np.all(got["X"][k] == 0) and not got["obs_inlier"][seg].any() and np.isnan(got["obs_error"][seg]).all()
                continue
            assert np.array_equal(got["obs_inlier"][seg].astype(bool), inl), k
            assert got["n_inliers"][k] == inl.sum()
            np.testing.assert_allclose(got["X"][k], X, rtol=1e-9, atol=0)
            e = got["obs_error"][seg]
            assert np.all(e[inl] <= max_error) and np.all(~(e[~inl] <= max_error))


def test_oracle_statuses_on_hand_made_tracks():
    """An image outside [0, n_images), a feature outside [0, S), a lone view, and a clean two-view track of neighbouring
    cameras: triangulated at min_angle 1.5, no model at 60 degrees, too few inliers when 3 are required."""
    from sfm_b200 import synth

    _, _, xy, cams, _ = random_scene_tracks(7, n_tracks=1)
    Ps = synth.make_cameras(12, baseline=3.0)
    X = np.array([0.3, -0.2, 6.0, 1.0])
    for i, f in ((3, 60), (4, 61)):
        p = Ps[i] @ X
        xy[i, f] = p[:2] / p[2]
    tracks = [[[0, 3], [12, 0]], [[0, 99], [1, 2]], [[0, 3]], [[3, 60], [4, 61]]]
    offs = np.cumsum([0] + [len(t) for t in tracks]).astype(np.int64)
    obs = np.concatenate(tracks).astype(np.int32)
    got = tro.triangulate_tracks(offs, obs, xy, cams)
    assert got["status"].tolist() == [4, 4, 1, 0] and got["counts"].tolist() == [1, 1, 0, 0, 2]
    np.testing.assert_allclose(got["X"][3], X[:3], rtol=1e-6)
    assert got["n_inliers"].tolist() == [0, 0, 0, 2] and got["obs_inlier"].tolist() == [0, 0, 0, 0, 0, 1, 1]
    assert got["obs_error"][5:].max() < 1e-3 and np.isnan(got["obs_error"][:5]).all()
    assert tro.triangulate_tracks(offs, obs, xy, cams, min_angle=60)["status"].tolist() == [4, 4, 1, 2]
    assert tro.triangulate_tracks(offs, obs, xy, cams, min_inliers=3)["status"].tolist() == [4, 4, 1, 3]


def test_camera_table():
    from sfm_b200 import synth
    from sfm_b200 import triangulate as tri

    K = synth.K_INTR
    R = np.stack([np.eye(3), np.eye(3)[[1, 0, 2]]])
    t = np.array([[0, 0, 0], [1.0, 2.0, 3.0]])
    tab = tri.camera_table(K, R, t)
    assert tab.shape == (2, 16) and tab.dtype == np.float64
    assert tab[1].tolist() == [1000.0, 1000.0, 960.0, 540.0] + R[1].ravel().tolist() + [1.0, 2.0, 3.0]
    K2 = np.stack([K, K * [[2, 1, 1], [1, 2, 1], [1, 1, 1]]])
    assert tri.camera_table(K2, R, t)[1, :4].tolist() == [2000.0, 2000.0, 960.0, 540.0]
    skew = K.copy()
    skew[0, 1] = 0.5
    for bad in (skew, K + np.array([[0, 0, 0], [0.1, 0, 0], [0, 0, 0]]), K + np.array([[0, 0, 0], [0, 0, 0], [0.001, 0, 0]]),
                K * [[1, 1, 1], [1, 1, 1], [1, 1, 2]], np.stack([K, K, K])):
        with pytest.raises(ValueError):
            tri.camera_table(bad, R, t)
    with pytest.raises(ValueError):
        tri.camera_table(K, R[:, :2], t)
    with pytest.raises(ValueError):
        tri.camera_table(K, R, t[:1])
    with pytest.raises(ValueError):
        tri.triangulate_params(min_inliers=1)
    with pytest.raises(ValueError):
        tri.triangulate_params(min_angle=90)


def test_scene_points_project_to_their_features():
    """Scene.X holds the world points make_scene draws: every shared feature is the projection of its point (0.5 px noise)."""
    from sfm_b200 import synth

    sc = synth.make_scene(3, 512, seed=4)
    assert sc.X.dtype == np.float64 and sc.X.shape == (int(round(256 * 1.5)), 3)
    for i in range(3):
        m = sc.point[i] >= 0
        p = (sc.P[i] @ np.concatenate([sc.X[sc.point[i][m]], np.ones((m.sum(), 1))], axis=1).T).T
        assert np.abs(p[:, :2] / p[:, 2:] - sc.xy[i][m]).max() < 4.0
