"""CPU checks of bundle adjustment: the parameter and summary structs as the header declares them, the C-ABI argument checks of
sfm_bundle_workspace_bytes and sfm_bundle_adjust (all before any CUDA call), and the float64 reference (tests/bundle_reference.py)
against scipy.optimize.least_squares and against first-order optimality by central finite differences."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.spatial.transform import Rotation

import bundle_reference as br

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _layout(tmp_path, struct, fields):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / f"{struct}.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sfm_b200.h"\nint main(void){' + f'printf("%zu", sizeof({struct}));'
                   + "".join(f'printf(" %zu", offsetof({struct}, {f}));' for f in fields) + "return 0;}\n")
    exe = tmp_path / struct
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    return [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]


def test_structs_match_header(tmp_path):
    from sfm_b200 import _lib

    for mirror, name in ((_lib.BundleParams, "sfm_bundle_params"), (_lib.BundleSummary, "sfm_bundle_summary")):
        fields = [f[0] for f in mirror._fields_]
        got = _layout(tmp_path, name, fields)
        assert [C.sizeof(mirror)] + [getattr(mirror, f).offset for f in fields] == got
        assert got[0] == 64


def test_entry_points_reject_bad_arguments_without_a_gpu():
    """Every rejection returns SFM_ERR_ARG with its message before any CUDA call (pointers are fake and never read)."""
    from sfm_b200 import _lib
    from sfm_b200 import bundle

    L = _lib.lib()
    err = lambda: L.sfm_last_error().decode()  # noqa: E731
    n = C.c_size_t(0)
    assert L.sfm_bundle_workspace_bytes(12, 100, 400, None) == -1 and "NULL" in err()
    for bad in (0, 1025, -3):
        assert L.sfm_bundle_workspace_bytes(bad, 100, 400, C.byref(n)) == -1 and "n_images must lie in [1, 1024]" in err(), bad
    assert L.sfm_bundle_workspace_bytes(12, -1, 400, C.byref(n)) == -1 and "max_tracks" in err()
    assert L.sfm_bundle_workspace_bytes(12, 100, 1 << 31, C.byref(n)) == -1 and "max_obs" in err()
    assert L.sfm_bundle_workspace_bytes(12, 100, 400, C.byref(n)) == 0
    need = n.value
    assert need >= (6 * 12) ** 2 * 8
    names = ("offsets", "obs", "tc", "ps", "oi", "X", "xy", "cams", "ws", "pose", "oX", "oe", "sum")

    def call(n_images=12, S=64, stride=64, max_tracks=100, max_obs=400, prm=True, null=None, ws_bytes=None, ws=0x100000, **fields):
        p = bundle.bundle_params()
        for k, v in fields.items():
            setattr(p, k, v)
        ptrs = {k: 0x1000 * (i + 1) for i, k in enumerate(names)}
        ptrs["ws"] = ws
        if null:
            ptrs[null] = None
        return L.sfm_bundle_adjust(n_images, S, ptrs["offsets"], ptrs["obs"], ptrs["tc"], max_tracks, max_obs, ptrs["ps"], ptrs["oi"], ptrs["X"],
                                   ptrs["xy"], stride, ptrs["cams"], None, None, C.byref(p) if prm else None, ptrs["ws"],
                                   need if ws_bytes is None else ws_bytes, ptrs["pose"], ptrs["oX"], ptrs["oe"], ptrs["sum"], None)

    assert call(prm=False) == -1 and "NULL params" in err()
    for name in names:
        assert call(null=name) == -1 and "sfm_bundle_adjust: NULL argument" in err(), name
    assert call(n_images=1025, stride=64) == -1 and "n_images must lie in [1, 1024], got 1025" in err()
    assert call(n_images=0) == -1 and "n_images" in err()
    assert call(S=0) == -1 and "S must be positive" in err()
    assert call(stride=63) == -1 and "xy_stride" in err()
    assert call(max_tracks=-1) == -1 and "max_tracks" in err()
    for it in (0, 10001):
        assert call(max_iters=it) == -1 and "max_iters must lie in [1, 10000]" in err(), it
    for v in (-1e-6, float("nan"), float("inf")):
        assert call(function_tolerance=v) == -1 and "function_tolerance" in err(), v
        assert call(parameter_tolerance=v) == -1 and "parameter_tolerance" in err(), v
    assert call(ws_bytes=need - 1) == -1 and "workspace" in err()
    assert call(ws=0x100010) == -1 and "aligned" in err()
    for bad in (dict(max_iters=0), dict(max_iters=10001), dict(function_tolerance=-1.0), dict(parameter_tolerance=float("nan"))):
        with pytest.raises(ValueError):
            bundle.bundle_params(**bad)


def small_problem(seed, n_cams=4, n_pts=60, sigma=0.5):
    """n_cams cameras (fx != fy, off-centre principal points) around n_pts points, every point seen by every camera with
    sigma px noise; cameras and points perturbed (about 0.3 degree, 1 % of the depth) as a bundle adjustment would start."""
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1.0, 1.0, (n_pts, 3))
    cams = np.zeros((n_cams, 16))
    xy = []
    for i in range(n_cams):
        a = -0.4 + 0.8 * i / max(n_cams - 1, 1)
        C0 = np.array([5 * np.sin(a), 0.3 * rng.normal(), -5 * np.cos(a)])
        z = -C0 / np.linalg.norm(C0)
        x = np.cross([0.0, 1.0, 0.0], z)
        x /= np.linalg.norm(x)
        R = np.stack([x, np.cross(z, x), z])
        cams[i] = np.concatenate([[900.0 + 40 * i, 880.0 + 35 * i, 640.0 + 7 * i, 360.0 - 5 * i], R.ravel(), -R @ C0])
    cam = np.repeat(np.arange(n_cams), n_pts)
    pt = np.tile(np.arange(n_pts), n_cams)
    xy = br.residuals(cams, X, cam, pt, np.zeros((len(cam), 2))).reshape(-1, 2) + rng.normal(0, sigma, (len(cam), 2))
    c0 = cams.copy()
    for i in range(1, n_cams):
        dR = Rotation.from_rotvec(rng.normal(size=3) * np.radians(0.3) / np.sqrt(3)).as_matrix()
        R = dR @ cams[i, 4:13].reshape(3, 3)
        C = -cams[i, 4:13].reshape(3, 3).T @ cams[i, 13:] + rng.normal(size=3) * 0.05 / np.sqrt(3)
        c0[i, 4:13], c0[i, 13:] = R.ravel(), -R @ C
    X0 = X + rng.normal(size=X.shape) * 0.01
    return c0, X0, cam, pt, xy


def test_reference_equals_least_squares():
    cams, X, cam, pt, xy = small_problem(3)
    var = np.array([False, True, True, True])
    adj = np.ones(len(X), bool)
    ref = br.bundle_adjust(cams, X, cam, pt, xy, var, adj)

    def unpack(z):
        c = cams.copy()
        for j, i in enumerate(np.nonzero(var)[0]):
            c[i, 4:13] = Rotation.from_rotvec(z[6 * j: 6 * j + 3]).as_matrix().ravel()
            c[i, 13:] = z[6 * j + 3: 6 * j + 6]
        return c, z[6 * var.sum():].reshape(-1, 3)

    z0 = np.concatenate([np.concatenate([Rotation.from_matrix(cams[i, 4:13].reshape(3, 3)).as_rotvec(), cams[i, 13:]]) for i in np.nonzero(var)[0]]
                        + [X.ravel()])
    ls = least_squares(lambda z: br.residuals(*unpack(z), cam, pt, xy), z0, method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-15, x_scale="jac")
    ls_cost = float(ls.fun @ ls.fun)
    print(f"\nreference cost {ref['cost']:.12e} ({ref['iterations']} iterations), least_squares {ls_cost:.12e}, start {ref['initial_cost']:.4e}; "
          f"max residual difference {np.abs(ref['residuals'] - ls.fun).max():.3e} px")
    assert ref["cost"] < 0.01 * ref["initial_cost"]
    assert abs(ref["cost"] - ls_cost) <= 1e-10 * ls_cost
    assert np.abs(ref["residuals"] - ls.fun).max() < 1e-6


def test_reference_gradient_vanishes_at_its_optimum():
    """Central finite differences of the cost in the reference's own parameters at the optimum: every component is a tiny fraction
    of the gradient at the start."""
    cams, X, cam, pt, xy = small_problem(5)
    var = np.array([False, True, True, True])
    adj = np.ones(len(X), bool)
    ref = br.bundle_adjust(cams, X, cam, pt, xy, var, adj)
    n = 6 * var.sum() + 3 * adj.sum()

    def cost(c, Xs):
        r = br.residuals(c, Xs, cam, pt, xy)
        return float(r @ r)

    def fd_grad(c, Xs, eps=1e-6):
        g = np.zeros(n)
        for j in range(n):
            h = np.zeros(n)
            h[j] = eps
            g[j] = (cost(*br.apply_step(c, Xs, h, var, adj)) - cost(*br.apply_step(c, Xs, -h, var, adj))) / (2 * eps)
        return g

    g0 = fd_grad(cams, X)
    g1 = fd_grad(ref["cams"], ref["X"])
    analytic = 2 * br.gradient(ref["cams"], ref["X"], cam, pt, xy, var, adj)
    print(f"\n|grad| at the start {np.abs(g0).max():.3e}, at the optimum {np.abs(g1).max():.3e} (analytic {np.abs(analytic).max():.3e})")
    assert np.abs(g1).max() < 1e-6 * np.abs(g0).max()
    assert np.abs(analytic).max() < 1e-6 * np.abs(g0).max()
    assert np.allclose(2 * br.gradient(cams, X, cam, pt, xy, var, adj), g0, rtol=1e-5, atol=1e-6 * np.abs(g0).max())


def test_problem_selects_used_observations():
    offsets = np.array([0, 3, 5, 7, 8])
    obs = np.array([[0, 1], [1, 4], [2, 2], [0, 5], [2, 0], [1, 1], [3, 3], [1, 7]])
    status = np.array([0, 0, 2, 0], np.uint8)
    inl = np.array([1, 1, 0, 1, 1, 1, 1, 1], np.uint8)
    cam, pt, o, var, adj = br.problem(offsets, obs, status, inl, 4, registered=[1, 1, 1, 0])
    assert o.tolist() == [0, 1, 3, 4, 7] and cam.tolist() == [0, 1, 0, 2, 1] and pt.tolist() == [0, 0, 1, 1, 3]
    assert adj.tolist() == [True, True, False, False] and var.tolist() == [False, True, True, False]
