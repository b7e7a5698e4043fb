"""CPU checks of incremental reconstruction: both parameter structs as the header declares them, the C-ABI argument checks of
sfm_next_images and sfm_filter_points (all before any CUDA call), the numpy oracle of both kernels on hand-worked cases, and
the initial-pair order."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import mapper_oracle as mo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FULL = 4 + 16 + 64 + 256 + 1024 + 4096          # one point: one cell at each of the 6 levels, weighted by d^2


def _layout(tmp_path, struct, fields):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / f"{struct}.c"
    src.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "sfm_b200.h"\nint main(void){{printf("%zu", sizeof({struct}));'
                   + "".join(f'printf(" %zu", offsetof({struct}, {f}));' for f in fields) + "return 0;}\n")
    exe = tmp_path / struct
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    return [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]


def test_params_structs_match_header(tmp_path):
    from sfm_b200 import _lib

    for mirror, struct in ((_lib.NextImagesParams, "sfm_next_images_params"), (_lib.FilterPointsParams, "sfm_filter_points_params")):
        fields = [f[0] for f in mirror._fields_]
        got = _layout(tmp_path, struct, fields)
        assert [C.sizeof(mirror)] + [getattr(mirror, f).offset for f in fields] == got
        assert got[0] == 64 and C.sizeof(mirror) == 64


def test_entry_points_reject_bad_arguments_without_a_gpu():
    """Every rejection returns SFM_ERR_ARG with its message before any CUDA call (pointers are fake and never read)."""
    from sfm_b200 import _lib
    from sfm_b200 import mapper

    L = _lib.lib()
    err = lambda: L.sfm_last_error().decode()  # noqa: E731
    fake = [0x1000 * (i + 1) for i in range(16)]

    def nxt(n_images=12, S=64, stride=64, null=None, **fields):
        p = mapper.next_images_params()
        for k, v in fields.items():
            setattr(p, k, v)
        a = list(fake)
        if null is not None:
            a[null] = None
        return L.sfm_next_images(n_images, S, a[0], a[1], 100, a[2], a[3], stride, a[4], a[5], a[6], C.byref(p), a[7], a[8], a[9], a[10], None)

    assert nxt(n_images=1025) == -1 and "[1, 1024]" in err()
    assert nxt(n_images=0) == -1 and "[1, 1024]" in err()
    assert nxt(stride=32) == -1 and "xy_stride" in err()
    assert nxt(levels=0) == -1 and "levels" in err()
    assert nxt(levels=9) == -1 and "levels" in err()
    assert nxt(max_select=0) == -1 and "max_select" in err()
    assert nxt(max_trials=0) == -1 and "max_trials" in err()
    assert nxt(null=7) == -1 and "NULL argument" in err()

    def flt(n_images=12, null=None, **fields):
        p = mapper.filter_params()
        for k, v in fields.items():
            setattr(p, k, v)
        a = list(fake)
        if null is not None:
            a[null] = None
        return L.sfm_filter_points(n_images, a[0], a[1], a[2], 100, a[3], a[4], a[5], C.byref(p), a[6], a[7], a[8], a[9], a[10], None)

    assert flt(n_images=0) == -1 and "positive" in err()
    assert flt(min_inliers=1) == -1 and "min_inliers" in err()
    assert flt(min_angle=90.0) == -1 and "min_angle" in err()
    assert flt(max_error=math.inf) == -1 and "max_error" in err()
    assert flt(null=4) == -1 and "NULL argument" in err()
    for bad in (dict(max_select=0), dict(levels=9), dict(max_trials=0), dict(min_visible=-1)):
        with pytest.raises(ValueError):
            mapper.next_images_params(**bad)
    for bad in (dict(max_error=-1.0), dict(min_angle=90), dict(min_inliers=1)):
        with pytest.raises(ValueError):
            mapper.filter_params(**bad)


def test_pyramid_score_hand_worked():
    w, h = 640, 480
    assert mo.pyramid_score([100.0], [100.0], w, h) == FULL
    assert mo.pyramid_score([], [], w, h) == 0
    # corners 0 and w: cell 0 and cell d - 1 (x = w gives floor(d) = d, clamped) at every level
    assert mo.pyramid_score([0.0, 640.0], [0.0, 0.0], w, h) == 2 * FULL
    # outside the image and NaN clamp to the border cells: -5 and NaN share x's cell 0 with 0, 1000 shares d - 1 with 640
    assert mo.pyramid_score([0.0, -5.0, np.nan, 640.0, 1000.0], [0.0] * 5, w, h) == 2 * FULL
    # x = w / 2 is the first cell of the right half at every level, one float32 ulp below it the last of the left half
    below = float(np.nextafter(np.float32(320.0), np.float32(0.0)))
    assert mo.pyramid_score([320.0, below], [0.0, 0.0], w, h) == 2 * FULL
    # x = 160 and 161 share a cell at every level up to d = 64 (16 and 16.1)
    assert mo.pyramid_score([160.0, 161.0], [0.0, 0.0], w, h) == FULL
    # x = 160 and 170 differ only at the finest level (d = 32: 8 and 8.5; d = 64: 16 and 17)
    assert mo.pyramid_score([160.0, 170.0], [0.0, 0.0], w, h) == FULL + 4096
    # a seventh level (d = 128) tells 160 and 165 apart (32 and 33) where six do not (16 and 16.5)
    assert mo.pyramid_score([160.0, 165.0], [0.0, 0.0], w, h) == FULL
    assert mo.pyramid_score([160.0, 165.0], [0.0, 0.0], w, h, levels=7) == FULL + 2 * 128 * 128
    # the cell uses the image's own size: with w = 320, x = 320 is the last cell
    assert mo.pyramid_score([319.0, 320.0], [0.0, 0.0], 320, 240) == FULL


def _images(xy_lists, S=8):
    n = len(xy_lists)
    track_of = np.full((n, S), -1, np.int32)
    xy = np.zeros((n, S, 2), np.float32)
    k = 0
    for i, pts in enumerate(xy_lists):
        for f, p in enumerate(pts):
            track_of[i, f] = k
            xy[i, f] = p
            k += 1
    return track_of, k, xy


def test_next_images_order_trials_and_padding():
    # image 0: 2 points in one cell; 1: 2 points in different cells; 2: like 1; 3: 3 points in one cell; 4: registered
    track_of, T, xy = _images([[(10, 10), (11, 11)], [(10, 10), (600, 400)], [(600, 400), (10, 10)], [(10, 10), (11, 10), (10, 11)],
                               [(10, 10), (600, 400)]])
    status = np.zeros(T, np.uint8)
    size = np.tile([640, 480], (5, 1))
    reg = np.array([0, 0, 0, 0, 1], np.uint8)
    trials = np.zeros(5, np.int32)
    o = mo.next_images(track_of, T, status, xy, size, reg, trials, max_select=8, min_visible=2)
    assert o["score"].tolist() == [FULL, 2 * FULL, 2 * FULL, FULL, 2 * FULL]
    assert o["visible"].tolist() == [2, 2, 2, 3, 2]
    # score ties: 1 before 2 (image ascending); 3 before 0 (more visible)
    assert o["images"].tolist() == [1, 2, 3, 0, -1, -1, -1, -1] and o["n_selected"] == 4
    assert o["trials"].tolist() == [1, 1, 1, 1, 0]
    # max_select 2: only the first two are selected and counted
    o2 = mo.next_images(track_of, T, status, xy, size, reg, trials, max_select=2, min_visible=2)
    assert o2["images"].tolist() == [1, 2] and o2["trials"].tolist() == [0, 1, 1, 0, 0]
    # max_trials: images 1 and 2 have used theirs
    o3 = mo.next_images(track_of, T, status, xy, size, reg, np.array([0, 3, 3, 2, 0], np.int32), max_select=3, min_visible=2)
    assert o3["images"].tolist() == [3, 0, -1] and o3["trials"].tolist() == [1, 3, 3, 3, 0]
    # min_visible 3 leaves image 3; a point whose track has no point (status != 0) is not visible
    st = status.copy()
    st[track_of[3, 0]] = 2
    o4 = mo.next_images(track_of, T, st, xy, size, reg, trials, max_select=4, min_visible=2)
    assert o4["visible"][3] == 2 and o4["images"].tolist() == [1, 2, 0, 3]
    assert mo.next_images(track_of, T, status, xy, size, reg, trials, max_select=4, min_visible=3)["images"].tolist() == [3, -1, -1, -1]


def _ring_cams(n, radius=10.0):
    cams = np.zeros((n, 16))
    for i in range(n):
        a = 2 * np.pi * i / n
        C = np.array([radius * np.sin(a), 0.0, -radius * np.cos(a)])
        z = -C / np.linalg.norm(C)
        x = np.cross([0.0, 1.0, 0.0], z)
        x /= np.linalg.norm(x)
        R = np.stack([x, np.cross(z, x), z])
        cams[i, :4] = [1000.0, 1000.0, 320.0, 240.0]
        cams[i, 4:13] = R.ravel()
        cams[i, 13:] = -R @ C
    return cams


def test_filter_points_hand_worked():
    cams = _ring_cams(8)
    reg = np.ones(8, np.uint8)
    reg[7] = 0
    f4 = np.float32(4.0)
    up = np.nextafter(f4, np.float32(np.inf))
    # track 0: errors NaN, +inf, exactly 4, one ulp above 4 -> 1 inlier left -> status 3
    # track 1: three inliers, one in an unregistered image -> stays, n_inliers 2
    # track 2: status 1 already -> untouched
    # track 3: two views of neighbouring cameras (45 degrees apart) -> stays
    obs = np.array([[0, 0], [1, 0], [2, 0], [3, 0], [0, 1], [2, 1], [7, 1], [5, 2], [6, 2], [1, 3], [2, 3]], np.int32)
    offsets = np.array([0, 4, 7, 9, 11], np.int64)
    err = np.array([np.nan, np.inf, 4.0, up, 0.5, 0.5, 0.5, 0.1, 0.1, 1.0, 1.0], np.float32)
    X = np.zeros((4, 3))
    X[2] = 7.0
    status = np.array([0, 0, 1, 0], np.uint8)
    inl = np.ones(11, np.uint8)
    inl[7:9] = 0
    o = mo.filter_points(offsets, obs, cams, reg, X, [4, 3, 0, 2], status, inl, err)
    assert o["status"].tolist() == [3, 0, 1, 0]
    assert o["obs_inlier"].tolist() == [0, 0, 0, 0, 1, 1, 0, 0, 0, 1, 1]
    assert o["n_inliers"].tolist() == [1, 2, 0, 2]
    assert np.array_equal(o["X"][2], [7.0] * 3) and not o["X"][0].any()
    assert o["counts"].tolist() == [2, 1, 0, 1, 0]
    # max_error 3.99 drops track 0's exact-4 observation as well (0 inliers left); min_inliers 3 makes track 1 status 3 too
    o = mo.filter_points(offsets, obs, cams, reg, X, [4, 3, 0, 2], status, inl, err, min_inliers=3)
    assert o["status"].tolist() == [3, 3, 1, 3] and o["n_inliers"].tolist() == [1, 2, 0, 2] and not o["obs_inlier"].any()


def test_filter_angle_exactly_at_the_threshold():
    """A point seen by two cameras whose rays meet at exactly min_angle (cos equal to cos(min_angle) to the bit) is kept; one
    double above that angle, status 2."""
    cams = _ring_cams(64, radius=10.0)
    X = np.array([0.3, 0.2, 0.1])
    Ca, Cb = mo.camera_center(cams[0]), mo.camera_center(cams[1])
    c = mo.ray_cos(list(X), Ca, Cb)
    m = math.degrees(math.acos(c))
    hit = None
    for _ in range(4000):                        # walk the doubles around acos(c) until cos reproduces c exactly
        cm = mo.cos_min_of(m)
        if cm == c:
            hit = m
            break
        m = math.nextafter(m, math.inf if cm > c else -math.inf)
    assert hit is not None
    above = hit
    while mo.cos_min_of(above) >= c:
        above = math.nextafter(above, math.inf)
    args = (np.array([0, 2], np.int64), np.array([[0, 0], [1, 0]], np.int32), cams, np.ones(64, np.uint8), X[None], [2],
            np.array([0], np.uint8), np.ones(2, np.uint8), np.zeros(2, np.float32))
    assert mo.filter_points(*args, min_angle=hit)["status"].tolist() == [0]
    o = mo.filter_points(*args, min_angle=above)
    assert o["status"].tolist() == [2] and o["n_inliers"].tolist() == [0] and not o["obs_inlier"].any() and not o["X"].any()


def test_initial_pair_order():
    from sfm_b200 import mapper

    n_pose = np.array([150, 300, 99, 300, 500, 200, 120])
    n_inl = np.array([200, 400, 300, 400, 600, 210, 200])
    n_h = np.array([100, 100, 0, 320, 481, 150, 90])
    # pair 2: too few; 4: H explains 481 > 0.8 * 600; 3: 320 <= 320 passes; ties on n_pose by pair index
    assert mapper.initial_pair_order(n_pose, n_inl, n_h, min_inliers=100, max_h_ratio=0.8).tolist() == [1, 3, 5, 0, 6]
    assert mapper.initial_pair_order(n_pose, n_inl, None, min_inliers=100).tolist() == [4, 1, 3, 5, 0, 6]
    assert mapper.initial_pair_order(n_pose, n_inl, n_h, min_inliers=1000).tolist() == []
    assert mapper.round_launches(50) == 2 + 2 + 1 + 4 + 5 * 50 + 1
