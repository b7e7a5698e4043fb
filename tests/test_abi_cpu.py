"""CPU-side checks of the boundary: the C-ABI library loads and exports every symbol include/sfm_b200.h
declares, argument validation fails loudly, and the product never routes through oracle/."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "sfm_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sfm_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_header_symbol():
    import sfm_b200

    L = sfm_b200._lib.lib()
    syms = _header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/sfm_b200.h but not exported"
    assert sorted(sfm_b200._lib.EXPORTS) == syms
    assert L.sfm_abi_version() == 2


def test_struct_layouts_match_header():
    from sfm_b200 import _lib

    assert C.sizeof(_lib.MatchParams) == 32
    assert C.sizeof(_lib.FilterParams) == 48
    assert C.sizeof(_lib.RansacParams) == 56
    from oracle.ransac_oracle import RansacParams as OracleParams

    assert C.sizeof(OracleParams) == C.sizeof(_lib.RansacParams)
    assert [f[0] for f in OracleParams._fields_] == [f[0] for f in _lib.RansacParams._fields_]


def test_argument_errors_are_reported_without_a_gpu():
    import sfm_b200

    L = sfm_b200._lib.lib()
    n = C.c_size_t(0)
    assert L.sfm_bank_storage_bytes(0, 10, 0, C.byref(n)) == -1
    assert b"positive" in L.sfm_last_error()
    assert L.sfm_bank_storage_bytes(4, 10, 7, C.byref(n)) == -1
    assert L.sfm_bank_storage_bytes(50, 8192, 0, C.byref(n)) == 0
    # desc 50*8192*128 + ext (1/4 of that /4...) + norms + xy + counts
    rows = 50 * 8192
    assert n.value >= rows * 128 + rows // 128 * 4096 + rows * 4 + rows * 8 + 50 * 4
    assert n.value < rows * (128 + 32 + 4 + 8) * 1.01 + 8192
    with pytest.raises(sfm_b200.SfmError):
        sfm_b200._lib.check(-1, "unit-test")

    # RANSAC-F / RANSAC-H launchers: every rejection returns before any CUDA call.  Pointers are fake and never read.
    from sfm_b200.ransac import ransac_params

    def ransac(entry, corr=0x1000, size=64, n_pairs=1, null=None, **fields):
        prm = ransac_params(solver="8pt")
        for k, v in fields.items():
            setattr(prm, k, v)
        a = {"corr": corr, "idx": 0x2000, "prm": C.byref(prm), "out": 0x3000, "ninl": 0x4000, "mask": 0x5000}
        if null:
            a[null] = None
        head = [a["corr"], size, a["idx"], n_pairs] if entry.endswith("_batch") else [a["corr"], a["idx"], n_pairs, size]
        opt = [None] * (3 if "_h_" in entry else 2)            # pair_id, samples (, stop_target)
        rc = getattr(L, entry)(*head, *opt, a["prm"], a["out"], a["ninl"], a["mask"], None, None)
        return rc, L.sfm_last_error().decode()

    for entry in ("sfm_ransac_f_batch", "sfm_ransac_f_packed", "sfm_ransac_h_batch", "sfm_ransac_h_packed"):
        model = entry.rsplit("_", 1)[0]
        assert ransac(entry, null="idx") == (-1, f"{entry}: NULL argument")
        for null in ("corr", "prm", "out", "ninl", "mask"):
            assert ransac(entry, null=null) == (-1, f"{model}: NULL argument"), (entry, null)
        assert ransac(entry, max_iters=0) == (-1, "max_iters and threshold must be positive")
        assert ransac(entry, threshold=0.0) == (-1, "max_iters and threshold must be positive")
        assert ransac(entry, size=0) == (-1, "bad sizes")
        assert ransac(entry, n_pairs=-1) == (-1, "bad sizes")
        assert ransac(entry, corr=0x1004) == (-1, "corr must be 16-byte aligned")
        assert ransac(entry, n_pairs=0)[0] == 0
        if model == "sfm_ransac_f":
            assert ransac(entry, solver=5) == (-1, "solver must be 7 or 8, got 5")
            assert ransac(entry, score=2) == (-1, "unknown score 2")
        else:                                                  # RANSAC-H ignores both fields
            assert ransac(entry, n_pairs=0, solver=5, score=2)[0] == 0


def test_no_cpu_fallback_without_cuda(monkeypatch):
    import torch

    import sfm_b200

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(sfm_b200.SfmError, match="no CPU fallback"):
        sfm_b200.DescriptorBank(2, 64)
    import feature_matching as fm

    img = np.zeros((64, 64), np.uint8)
    with pytest.raises(sfm_b200.SfmError, match="no CPU fallback"):
        fm.extract_and_match(img, img)                    # extraction itself runs on the device: loud failure, never cv2 in its place
    monkeypatch.setattr(fm, "GPU_DESCRIPTORS", False)     # (SFM_ORB_DESCRIPTORS=cv2: extraction left to cv2 as the north star allows)
    fm._ORB_CACHE.clear()
    assert fm.extract_and_match(img, img) == []          # no keypoints -> [] before any GPU work
    with pytest.raises(ValueError):
        fm.extract_and_match(img.astype(np.float32), img)


def test_product_never_imports_the_oracle():
    """The product path must not import, include, link or execute anything under oracle/."""
    pkg = os.path.join(ROOT, "sfm-project_b200")
    for dirpath, _, files in os.walk(pkg):
        if os.path.basename(dirpath) in ("build", "__pycache__", "lib"):
            continue
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".h", "Makefile")):
                continue
            text = open(os.path.join(dirpath, f)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f"{f} imports oracle"
            for ln in text.splitlines():
                code = ln.split("//")[0].split("#")[0] if not ln.lstrip().startswith("#include") else ln
                assert "oracle" not in code or ln.lstrip().startswith(("//", "#", "*", '"""')) or "oracle" in ln.split("//")[-1], (f, ln)


def test_dropin_module_surface_matches_reference():
    """Names code/pipeline.py relies on via `from feature_matching import*` (SURVEY §8b)."""
    import feature_matching as fm
    import geometric_verification as gv

    for name in ("extract_and_match", "extract_and_match_draw", "read_img", "os", "cv2", "np", "math", "plt", "bisect"):
        assert hasattr(fm, name), name
    assert not hasattr(fm, "__all__")
    for name in ("verify_pair", "verify_pairs", "verify_matches"):
        assert hasattr(gv, name), name
    assert not hasattr(gv, "__all__")


def test_pair_enumerations():
    from sfm_b200 import synth

    assert len(synth.exhaustive_pairs(50)) == 1225
    assert len(synth.exhaustive_pairs(200)) == 19900
    assert len(synth.windowed_pairs(1000, 20)) == 19790
    from sfm_b200 import pairs as pl

    bp = pl.blocked_exhaustive_pairs(200, 32)
    assert len(bp) == 19900 and sorted(map(tuple, bp.tolist())) == sorted(map(tuple, synth.exhaustive_pairs(200).tolist()))
    assert len({(a // 32, b // 32) for a, b in bp[:496].tolist()}) == 1          # the first square: 32 images against themselves
    assert np.array_equal(pl.blocked_exhaustive_pairs(20, 32), synth.exhaustive_pairs(20))
    op = synth.ordered_pairs(4)
    assert len(op) == 12 and op[0].tolist() == [0, 1] and op[3].tolist() == [1, 0]


def test_synthetic_scene_properties():
    from sfm_b200 import synth

    sc = synth.make_scene(3, 512, seed=1)
    assert sc.desc.shape == (3, 512, 128) and sc.desc.dtype == np.uint8
    norms = np.linalg.norm(sc.desc.astype(np.float64), axis=2)
    assert 400 < np.median(norms) < 620
    shared = (sc.point[0] >= 0).sum()
    assert shared == 256
    F = sc.true_fundamental(0, 1)
    both = np.intersect1d(sc.point[0][sc.point[0] >= 0], sc.point[1][sc.point[1] >= 0])
    i0 = np.array([np.nonzero(sc.point[0] == b)[0][0] for b in both[:50]])
    i1 = np.array([np.nonzero(sc.point[1] == b)[0][0] for b in both[:50]])
    from oracle import ransac_oracle as ro

    assert np.median(ro.sym_epipolar_err(F, sc.xy[0][i0], sc.xy[1][i1])) < 4.0


def test_two_view_host_logic_without_a_gpu():
    """Host-side pieces of the §8f stages that need no device: camera rows, per-image intrinsics, edge classification."""
    import numpy as np

    from sfm_b200 import plan as pl
    from sfm_b200 import ransac as rs

    K = np.array([[1000.0, 0, 960], [0, 1100.0, 540], [0, 0, 1]])
    rows = rs.camera_rows(K, None, 3)
    assert rows.shape == (3, 8) and rows[1].tolist() == [1000.0, 1100.0, 960.0, 540.0] * 2
    K2 = np.stack([K, 2 * K, 3 * K])
    K2[:, 2, 2] = 1
    both = rs.camera_rows(K, K2, 3)
    assert both[2].tolist() == [1000.0, 1100.0, 960.0, 540.0, 3000.0, 3300.0, 2880.0, 1620.0]
    for bad in (np.eye(4), np.array([[1.0, 0.5, 0], [0, 1, 0], [0, 0, 1]])):
        with pytest.raises(ValueError):
            rs.camera_rows(bad)
    assert pl.intrinsics_rows(K, 4).tolist() == [[1000.0, 1100.0, 960.0, 540.0]] * 4
    assert pl.intrinsics_rows(K2, 3)[2].tolist() == [3000.0, 3300.0, 2880.0, 1620.0]
    assert pl.intrinsics_rows(np.array([[1.0, 2, 3, 4]] * 5), 5).shape == (5, 4)
    for bad, n in ((K2, 4), (np.zeros((3, 4)), 3), (np.ones((3, 5)), 3)):
        with pytest.raises(ValueError):
            pl.intrinsics_rows(bad, n)

    import sys

    sys.modules.pop("geometric_verification", None)
    import geometric_verification as gv

    cls = gv.classify_pairs([100, 100, 10, 0], [50, 81, 10, 0], calibrated=True)
    assert list(cls) == [gv.CALIBRATED, gv.PLANAR_OR_PANORAMIC, gv.DEGENERATE, gv.DEGENERATE]
    assert list(gv.classify_pairs([100], [80])) == [gv.UNCALIBRATED]            # exactly the ratio: not planar
    assert list(gv.classify_pairs([20], [19], min_inliers=30)) == [gv.DEGENERATE]
    for name in ("verify_pair", "verify_pairs", "verify_matches", "find_homography", "find_homographies", "recover_pose",
                 "recover_poses", "classify_pairs", "two_view_geometry"):
        assert callable(getattr(gv, name))


def test_extract_and_match_draw_runs_under_stubbed_pyplot(monkeypatch):
    """code/feature_matching.py:15-37 executed once: extraction, the matcher call, cv2.drawMatches with the reference's
    arguments, plt.imshow + plt.show, and the match list handed back.  No GPU here, so the device matcher is replaced by a
    recorder; the GPU twin (tests/test_gpu_matcher.py) checks the real list."""
    import cv2
    import feature_matching as fm

    rng = np.random.default_rng(4)
    g1 = cv2.GaussianBlur((rng.random((240, 320)) * 255).astype(np.uint8), (5, 5), 0)
    g2 = np.roll(g1, 3, axis=1)
    calls = {}
    fake = [cv2.DMatch(0, 1, 0, 7.0), cv2.DMatch(2, 0, 0, 11.0)]

    def fake_match(des1, des2, max_distance=fm.MAX_HAMMING_DISTANCE, _keys=None):
        calls["match"] = (None if des1 is None else des1.shape, None if des2 is None else des2.shape, _keys)
        return list(fake)

    def fake_draw(img1, kp1, img2, kp2, matches, out, **kw):
        calls["draw"] = (img1 is g1, img2 is g2, len(kp1), len(kp2), [m.queryIdx for m in matches], out, kw)
        return np.zeros((4, 4, 3), np.uint8)

    class Plt:
        def imshow(self, img):
            calls["imshow"] = img.shape

        def show(self):
            calls["show"] = True

    monkeypatch.setattr(fm, "GPU_DESCRIPTORS", False)        # no device here: cv2 computes the descriptors, the matcher is the recorder
    monkeypatch.setattr(fm, "match_descriptors_hamming", fake_match)
    monkeypatch.setattr(fm.cv2, "drawMatches", fake_draw)
    monkeypatch.setattr(fm, "plt", Plt())
    out = fm.extract_and_match_draw(g1, g2)
    assert [(m.queryIdx, m.trainIdx, m.distance) for m in out] == [(0, 1, 7.0), (2, 0, 11.0)]
    kp1, des1 = cv2.ORB_create().detectAndCompute(g1, None)
    assert calls["match"][0] == des1.shape and calls["match"][2][0] != calls["match"][2][1]
    assert calls["draw"][:2] == (True, True) and calls["draw"][2] == len(kp1) and calls["draw"][4] == [0, 2] and calls["draw"][5] is None
    assert calls["draw"][6] == {"flags": cv2.DrawMatchesFlags_NOT_DRAW_SINGLE_POINTS}
    assert calls["imshow"] == (4, 4, 3) and calls["show"] is True
    with pytest.raises(ValueError):
        fm.extract_and_match_draw(g1.astype(np.float32), g2)


def test_image_cache_key_fast_path_is_safe():
    """The drop-in keys its ORB cache on image CONTENT; an ndarray object seen before skips the full hash, but never when
    the object was modified in place, replaced at the same address, or is another view."""
    import feature_matching as fm

    rng = np.random.default_rng(1)
    a = (rng.random((480, 640)) * 255).astype(np.uint8)
    k1 = fm._content_key(a)
    assert fm._content_key(a) == k1 and id(a) in fm._SEEN
    b = a.copy()
    assert fm._content_key(b) == k1                       # same content, other object: same key through the hash
    a[::15, ::20] ^= 0xFF                                 # in-place edit that hits the sparse fingerprint
    k2 = fm._content_key(a)
    assert k2 != k1 and fm._content_key(a) == k2
    v = a[:, ::-1]
    assert fm._content_key(v) != k2                       # a view with other strides is another image
