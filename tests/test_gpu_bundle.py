"""Bundle adjustment on the GPU (csrc/bundle.cu) against the independent float64 reference (tests/bundle_reference.py): the
optimum (final cost and every residual; poses and points directly with two fixed cameras) on the 12-camera mixed rig at world
offsets 0 and 1e5; first-order optimality; ground truth (perturbation recovery and the incremental loop of test_gpu_pnp.py);
invariants and bit-identity (run to run, another stream, extra unregistered images); the fixed launch count and a CUDA-graph
replay; edge cases and the public call.  Measured numbers are printed and recorded in DESIGN §4 "Bundle adjustment"."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # collected on CPU boxes, skipped there
    pytest.skip("needs a GPU", allow_module_level=True)

from scipy.optimize import least_squares  # noqa: E402
from scipy.spatial.transform import Rotation  # noqa: E402

import bundle_reference as br  # noqa: E402
import geometric_verification as gv  # noqa: E402
import sfm_b200  # noqa: E402
from sfm_b200 import bundle, synth  # noqa: E402
from sfm_b200 import pnp  # noqa: E402
from sfm_b200 import triangulate as tri  # noqa: E402
from sfm_b200 import tracks as tr  # noqa: E402
from test_gpu_register_reference import CAMERAS, track_scene  # noqa: E402

TIGHT = dict(function_tolerance=1e-12, parameter_tolerance=1e-12, max_iters=200)
# Measured on one B200 (DESIGN §4 "Bundle adjustment"): 8.3e-15 / 2.5e-10 relative cost and 6.3e-9 / 7.2e-7 px per residual at
# world offsets 0 / 1e5.  The bounds are ceilings well above both.
COST_REL = 1e-8
RESID_PX = 1e-5


def umeyama(src, dst):
    """s, Q, c with dst ~ s Q src + c (least squares)."""
    ms, md = src.mean(0), dst.mean(0)
    a, b = src - ms, dst - md
    U, D, Vt = np.linalg.svd(b.T @ a / len(src))
    S = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        S[2, 2] = -1
    Q = U @ S @ Vt
    return np.trace(np.diag(D) @ S) / a.var(0).sum(), Q, md - (np.trace(np.diag(D) @ S) / a.var(0).sum()) * Q @ ms


def rot_err(Ra, Rb):
    return float(np.degrees(Rotation.from_matrix(Ra @ Rb.T).magnitude()))


def perturb(cams, seed, depth=8.0):
    """Rotations of about 0.3 degree and centres moved about 1 % of the depth."""
    rng = np.random.default_rng(seed)
    out = cams.copy()
    for i in range(len(cams)):
        R = cams[i, 4:13].reshape(3, 3)
        C = -R.T @ cams[i, 13:]
        Rn = Rotation.from_rotvec(rng.normal(size=3) * np.radians(0.3) / np.sqrt(3)).as_matrix() @ R
        Cn = C + rng.normal(size=3) * 0.01 * depth / np.sqrt(3)
        out[i, 4:13], out[i, 13:] = Rn.ravel(), -Rn @ Cn
    return out


def rig_problem(offset, seed=0, n_tracks=400, n_views=12):
    """The 12-camera mixed rig (640x480 to 7680x4320, fx != fy) around n_tracks points; cameras perturbed; points triangulated
    on the device from the perturbed cameras.  Returns (scene dict, true cams, start cams, Tracks, TrackPoints, xy)."""
    s = track_scene([c for _, c in CAMERAS], n_tracks, seed, offset=offset, outlier_frac=0.0, n_views=n_views)
    start = perturb(s["cams"], seed + 100)
    dev = torch.device("cuda")
    counts = torch.tensor([n_tracks, len(s["obs"]), 0, 0, 0], dtype=torch.int64, device=dev)
    t = tr.Tracks(offsets_buf=torch.from_numpy(s["offsets"]).to(dev), obs_buf=torch.from_numpy(s["obs"]).to(dev),
                  track_of_buf=torch.zeros((n_views, n_tracks), dtype=torch.int32, device=dev), counts_dev=counts)
    xy = torch.from_numpy(np.ascontiguousarray(s["xy"])).to(dev)
    pts = tri.triangulate_tracks_device(t, xy, torch.from_numpy(start).to(dev), max_error=1e4)
    assert pts.counts["triangulated"] == n_tracks
    return s, start, t, pts, xy


def reference_of(s, start, pts, fixed=None, n_images=12):
    h = pts.to_host()
    cam, pt, o, var, adj = br.problem(s["offsets"], s["obs"], h["status"], h["obs_inlier"], n_images, fixed=fixed)
    xy = s["xy"][cam, s["obs"][o, 1]].astype(np.float64)
    return br.bundle_adjust(start, h["X"], cam, pt, xy, var, adj), (cam, pt, o, var, adj, xy)


def gpu_residuals(res, start, cam, pt, xy):
    c = start.copy()
    c[:, 4:] = res["pose"]
    return br.residuals(c, res["X"], cam, pt, xy), c


@pytest.fixture(scope="module", params=[0.0, 1e5], ids=["offset0", "offset1e5"])
def rig(request):
    s, start, t, pts, xy = rig_problem(request.param)
    cams = torch.from_numpy(start).cuda()
    res = bundle.bundle_adjust_device(t, pts, xy, cams, **TIGHT).to_host()
    ref, prob = reference_of(s, start, pts)
    return request.param, s, start, t, pts, xy, res, ref, prob


def test_optimum_equals_the_reference(rig):
    offset, s, start, t, pts, xy, res, ref, (cam, pt, o, var, adj, pxy) = rig
    r, _ = gpu_residuals(res, start, cam, pt, pxy)
    cost = float(r @ r)
    rel = abs(res["final_cost"] - ref["cost"]) / ref["cost"]
    dres = np.abs(r - ref["residuals"]).max()
    print(f"\noffset {offset:g}: status {res['status']} after {res['iterations']} iterations ({res['accepted']} accepted); cost "
          f"{res['initial_cost']:.6e} -> {res['final_cost']:.12e}, reference {ref['cost']:.12e} ({ref['iterations']} iterations): "
          f"relative difference {rel:.3e}, max residual difference {dres:.3e} px, own cost recomputed {abs(cost - res['final_cost']) / cost:.3e}")
    assert res["status"] in ("function_tolerance", "parameter_tolerance", "no_progress")
    assert res["variable_cameras"] == 11 and res["adjusted_points"] == 400 and res["used_obs"] == 400 * 12
    assert rel <= COST_REL
    assert dres <= RESID_PX
    assert abs(cost - res["final_cost"]) <= 1e-9 * cost


@pytest.mark.parametrize("offset", [0.0, 1e5])
def test_two_fixed_cameras_pin_poses_and_points(offset):
    s, start, t, pts, xy = rig_problem(offset, seed=1)
    fixed = np.zeros(12, np.uint8)
    fixed[[0, 6]] = 1
    res = bundle.bundle_adjust_device(t, pts, xy, torch.from_numpy(start).cuda(), fixed=fixed, **TIGHT).to_host()
    ref, _ = reference_of(s, start, pts, fixed=fixed)
    dpose = np.abs(res["pose"] - ref["cams"][:, 4:]).max()
    Ct = np.stack([-res["R"][i].T @ res["t"][i] for i in range(12)])
    Cr = np.stack([-ref["cams"][i, 4:13].reshape(3, 3).T @ ref["cams"][i, 13:] for i in range(12)])
    dX = np.abs(res["X"] - ref["X"]).max()
    dC = np.abs(Ct - Cr).max()
    print(f"\noffset {offset:g}: max |R, t| difference {dpose:.3e}, centre {dC:.3e}, point {dX:.3e} (cost {res['final_cost']:.10e} vs "
          f"{ref['cost']:.10e})")
    assert dC <= 1e-5 and dX <= 1e-5
    assert np.abs(res["pose"][:, :9] - ref["cams"][:, 4:13]).max() <= 1e-7


def test_first_order_optimality(rig):
    offset, s, start, t, pts, xy, res, ref, (cam, pt, o, var, adj, pxy) = rig
    _, c = gpu_residuals(res, start, cam, pt, pxy)
    g0 = np.abs(br.gradient(start, pts.to_host()["X"], cam, pt, pxy, var, adj)).max()
    g1 = np.abs(br.gradient(c, res["X"], cam, pt, pxy, var, adj)).max()
    print(f"\noffset {offset:g}: max |J^T r| {g0:.3e} at the start, {g1:.3e} at the GPU optimum (ratio {g1 / g0:.3e})")
    assert g1 <= 1e-6 * g0


def test_perturbation_recovery_against_ground_truth(rig):
    """After a similarity alignment the camera and point errors fall back to those of points triangulated from the true cameras."""
    offset, s, start, t, pts, xy, res, ref, _ = rig
    C_true = np.stack([-R.T @ tt for R, tt in zip(s["Rs"], s["ts"])])
    C_est = np.stack([-res["R"][i].T @ res["t"][i] for i in range(12)])
    sc, Q, c = umeyama(C_est - C_true.mean(0), C_true - C_true.mean(0))
    cen = np.linalg.norm((sc * (Q @ (C_est - C_true.mean(0)).T)).T + c - (C_true - C_true.mean(0)), axis=1)
    rot = [rot_err(res["R"][i] @ Q.T, s["Rs"][i]) for i in range(12)]
    Xa = (sc * (Q @ (res["X"] - C_true.mean(0)).T)).T + c + C_true.mean(0)
    true_pts = tri.triangulate_tracks_device(t, xy, torch.from_numpy(s["cams"]).cuda(), max_error=1e4).to_host()["X"]
    e_ba = np.median(np.linalg.norm(Xa - s["X"], axis=1))
    e_true = np.median(np.linalg.norm(true_pts - s["X"], axis=1))
    C0 = np.stack([-start[i, 4:13].reshape(3, 3).T @ start[i, 13:] for i in range(12)])
    print(f"\noffset {offset:g}: start centre error median {np.median(np.linalg.norm(C0 - C_true, axis=1)):.4f}; after BA rotation "
          f"median {np.median(rot):.5f} deg, centre median {np.median(cen):.6f}; point error median {e_ba:.6f} vs {e_true:.6f} from the "
          f"true cameras")
    assert np.median(rot) < 0.05 and np.median(cen) < 0.003
    assert e_ba <= 1.5 * e_true


def test_invariants_and_bit_identity():
    s, start, t, pts, xy = rig_problem(0.0, seed=2, n_tracks=300)
    reg = np.ones(12, np.uint8)
    reg[5] = 0                                                 # unregistered
    fixed = np.zeros(12, np.uint8)
    fixed[[0, 3]] = 1
    status = pts.status_buf.clone()
    pts.status_buf[7] = 2                                      # a point without status 0 stays as it was
    inl = pts.obs_inlier_buf.clone()
    pts.obs_inlier_buf[s["offsets"][0]: s["offsets"][-1]].view(-1, 12)[:, 9] = 0     # camera 9: no used observation
    cams = torch.from_numpy(start).cuda()
    a = bundle.bundle_adjust_device(t, pts, xy, cams, reg, fixed=fixed, **TIGHT)
    ha = a.to_host()
    for i in (0, 3, 5, 9):
        assert np.array_equal(ha["pose"][i].view(np.uint8), start[i, 4:].view(np.uint8)), i
    assert np.array_equal(ha["X"][7].view(np.uint8), pts.X_buf[7].cpu().numpy().view(np.uint8))
    assert ha["final_cost"] <= ha["initial_cost"] and ha["variable_cameras"] == 8
    # run to run, on another stream, with extra unregistered images
    b = bundle.bundle_adjust_device(t, pts, xy, cams, reg, fixed=fixed, **TIGHT).to_host()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        c = bundle.bundle_adjust_device(t, pts, xy, cams, reg, fixed=fixed, **TIGHT)
    side.synchronize()
    c = c.to_host()
    xy_big = torch.cat([xy, torch.zeros((5,) + tuple(xy.shape[1:]), dtype=xy.dtype, device=xy.device)]).contiguous()
    cams_big = torch.cat([cams, cams[:5]]).contiguous()
    d = bundle.bundle_adjust_device(t, pts, xy_big, cams_big, np.concatenate([reg, np.zeros(5, np.uint8)]),
                                    fixed=np.concatenate([fixed, np.zeros(5, np.uint8)]), **TIGHT).to_host()
    for other in (b, c, d):
        assert np.array_equal(ha["pose"].view(np.uint8), other["pose"][:12].view(np.uint8))
        assert np.array_equal(ha["X"].view(np.uint8), other["X"].view(np.uint8))
        assert np.array_equal(ha["obs_error"].view(np.uint8), other["obs_error"].view(np.uint8))
        assert (other["iterations"], other["final_cost"]) == (ha["iterations"], ha["final_cost"])
    pts.status_buf.copy_(status)
    pts.obs_inlier_buf.copy_(inl)


def test_launch_count_and_graph_replay():
    s, start, t, pts, xy = rig_problem(0.0, seed=3, n_tracks=200)
    cams = torch.from_numpy(start).cuda()
    ws = torch.empty(bundle.workspace_bytes(12, pts.X_buf.shape[0], pts.obs_inlier_buf.numel()), dtype=torch.uint8, device="cuda")
    prm = dict(max_iters=20, function_tolerance=1e-10)
    torch.cuda.synchronize()
    n0 = sfm_b200.launch_count()
    eager = bundle.bundle_adjust_device(t, pts, xy, cams, workspace=ws, **prm)
    assert sfm_b200.launch_count() - n0 == bundle.bundle_launches(20) == 4 + 5 * 20
    eager = eager.to_host()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            cap = bundle.bundle_adjust_device(t, pts, xy, cams, workspace=ws, **prm)
    g.replay()
    torch.cuda.synchronize()
    h = cap.to_host()
    assert np.array_equal(h["pose"].view(np.uint8), eager["pose"].view(np.uint8))
    assert np.array_equal(h["X"].view(np.uint8), eager["X"].view(np.uint8))
    assert h["final_cost"] == eager["final_cost"] and h["iterations"] == eager["iterations"]


@pytest.fixture(scope="module")
def scene():
    sc = synth.make_scene(12, 4096, seed=21)
    bank = sfm_b200.DescriptorBank(12, 4096)
    bank.put(0, sc.desc, xy=sc.xy)
    res = sfm_b200.match_and_verify(bank, synth.exhaustive_pairs(12), tracks=True, max_iters=512, seed=9, solver="8pt")
    Rt = np.einsum("ij,njk->nik", np.linalg.inv(synth.K_INTR), sc.P)
    return sc, bank, res, Rt


def loop_errors(R, t, Rt, depth):
    C_est = np.stack([-R[i].T @ t[i] for i in range(12)])
    C_true = np.stack([-Rt[i, :, :3].T @ Rt[i, :, 3] for i in range(12)])
    s, Q, c = umeyama(C_est, C_true)
    cen = np.linalg.norm((s * (Q @ C_est.T)).T + c - C_true, axis=1)
    rot = [rot_err(R[i] @ Q.T, Rt[i, :, :3]) for i in range(12)]
    return float(np.median(rot)), float(100 * np.median(cen) / depth)


def test_incremental_loop_then_bundle_adjustment(scene):
    """test_gpu_pnp.py::test_incremental_loop_on_the_device, then triangulation from all twelve and bundle adjustment: the median
    rotation and centre errors drop to at most half of the unadjusted loop's."""
    sc, bank, res, Rt = scene
    two = sfm_b200.match_and_verify(bank, [[0, 1]], fetch=True, max_iters=512, seed=5, solver="8pt").to_host()
    m = two["matches"][two["inlier"].astype(bool)]
    g = gv.two_view_geometry(sc.xy[0][m[:, 0]], sc.xy[1][m[:, 1]], synth.K_INTR, synth.K_INTR, seed=3)
    R = np.tile(np.eye(3), (12, 1, 1))
    t = np.zeros((12, 3))
    R[1], t[1] = g["R"], g["t"]
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, R, t)).cuda()
    reg = torch.zeros(12, dtype=torch.uint8, device="cuda")
    reg[:2] = 1
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, reg, S=bank.max_feats)
    pnp.register_images_device(res.tracks, pts, bank.xy, cams, np.arange(2, 12), update=True, registered=reg, seed=4)
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, reg, S=bank.max_feats)
    second = pnp.register_images_device(res.tracks, pts, bank.xy, cams, np.arange(12), update=True, registered=reg, seed=4).to_host()
    assert second["registered"] == 12
    depth = float(np.median(sc.X @ Rt[0, 2, :3] + Rt[0, 2, 3]))
    before = loop_errors(second["R"], second["t"], Rt, depth)
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, reg, S=bank.max_feats)
    torch.cuda.synchronize()
    n0 = sfm_b200.launch_count()
    out = bundle.bundle_adjust_device(res.tracks, pts, bank.xy, cams, reg, update=True, S=bank.max_feats)
    assert sfm_b200.launch_count() - n0 == bundle.bundle_launches(50)
    h = out.to_host()
    after = loop_errors(h["R"], h["t"], Rt, depth)
    assert np.array_equal(cams[:, 4:].cpu().numpy(), h["pose"])
    assert np.array_equal(pts.X.cpu().numpy().view(np.uint8), h["X"].view(np.uint8))
    print(f"\nincremental loop: rotation error median {before[0]:.4f} deg, centre error median {before[1]:.4f} % of the median depth; "
          f"after BA ({h['status']}, {h['iterations']} iterations, RMS {np.sqrt(h['final_cost'] / h['used_obs']):.4f} px over "
          f"{h['used_obs']} observations): {after[0]:.4f} deg, {after[1]:.4f} %")
    assert after[0] <= 0.5 * before[0] and after[1] <= 0.5 * before[1]
    assert h["final_cost"] < h["initial_cost"]


def test_edge_cases(scene):
    sc, bank, res, Rt = scene
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])).cuda()
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, S=bank.max_feats)
    # no used observation: nothing registered
    h = bundle.bundle_adjust_device(res.tracks, pts, bank.xy, cams, np.zeros(12, np.uint8), S=bank.max_feats).to_host()
    assert h["status"] == "nothing_to_adjust" and h["iterations"] == 0 and h["used_obs"] == 0
    assert np.array_equal(h["pose"], cams[:, 4:].cpu().numpy()) and np.array_equal(h["X"], pts.X.cpu().numpy())
    # one variable camera
    fixed = np.ones(12, np.uint8)
    fixed[4] = 0
    h = bundle.bundle_adjust_device(res.tracks, pts, bank.xy, cams, fixed=fixed, S=bank.max_feats).to_host()
    assert h["variable_cameras"] == 1 and h["final_cost"] <= h["initial_cost"]
    assert np.array_equal(np.delete(h["pose"], 4, 0), np.delete(cams[:, 4:].cpu().numpy(), 4, 0))
    # out-of-range observation: status 5, everything returned as it came
    bad = tr.Tracks(offsets_buf=res.tracks.offsets_buf, obs_buf=res.tracks.obs_buf.clone(), track_of_buf=res.tracks.track_of_buf,
                    counts_dev=res.tracks.counts_dev)
    k = int(np.nonzero(pts.status.cpu().numpy() == 0)[0][0])
    bad.obs_buf[int(res.tracks.offsets_buf[k]), 0] = 12
    h = bundle.bundle_adjust_device(bad, pts, bank.xy, cams, S=bank.max_feats).to_host()
    assert h["status"] == "invalid" and np.array_equal(h["pose"], cams[:, 4:].cpu().numpy())
    # n_images 1025 is rejected on the host
    with pytest.raises(ValueError, match="1 to 1024"):
        bundle.bundle_adjust_device(res.tracks, pts, torch.zeros((1025, 4096, 2), dtype=torch.float32, device="cuda"),
                                    torch.zeros((1025, 16), dtype=torch.float64, device="cuda"))
    with pytest.raises(sfm_b200.SfmError, match="1024"):
        bundle.workspace_bytes(1025, 10, 10)


def per_point_ls(cams, q, xy):
    """The offset d minimising the pixel error of X0 + d over every view, with q = R X0 + t formed once per view so that far
    worlds lose no digits to the cancellation in R X + t."""
    R = cams[:, 4:13].reshape(-1, 3, 3)

    def res(d):
        p = q + R @ d
        return np.concatenate([cams[:, 0] * p[:, 0] / p[:, 2] + cams[:, 2] - xy[:, 0], cams[:, 1] * p[:, 1] / p[:, 2] + cams[:, 3] - xy[:, 1]])

    return least_squares(res, np.zeros(3), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, x_scale="jac").x


def test_all_cameras_fixed_refines_each_point_alone():
    s, start, t, pts, xy = rig_problem(1e5, seed=4, n_tracks=100)
    h = bundle.bundle_adjust_device(t, pts, xy, torch.from_numpy(start).cuda(), fixed=np.ones(12, np.uint8), **TIGHT).to_host()
    assert h["variable_cameras"] == 0 and np.array_equal(h["pose"], start[:, 4:])
    X0 = pts.to_host()["X"]
    worst = 0.0
    R = start[:, 4:13].reshape(-1, 3, 3)
    for k in range(100):
        ls = per_point_ls(start, R @ X0[k] + start[:, 13:], s["xy"][:, k].astype(np.float64))
        worst = max(worst, float(np.abs(X0[k] + ls - h["X"][k]).max()))
    print(f"\nall cameras fixed ({h['status']}, {h['iterations']} iterations): max point difference to the per-point least squares "
          f"{worst:.3e} (world offset 1e5)")
    # measured 5.3e-6 on one B200: the kernel evaluates R X + t at |X| ~ 1e5, so its cost resolves ~2e-8 relative and its points
    # ~5e-6; the per-point solution forms R X0 + t once and does not share that floor
    assert worst <= 2e-5


def test_public_call_on_host_inputs():
    s, start, t, pts, xy = rig_problem(0.0, seed=5, n_tracks=150)
    host_tracks = {"offsets": s["offsets"], "obs": s["obs"], "track_of": np.zeros((12, 150), np.int32), "n_tracks": 150,
                   "n_obs": len(s["obs"]), "n_conflicting": 0, "n_short": 0, "n_invalid_rows": 0}
    Ks = np.stack([np.array([[c[0], 0, c[2]], [0, c[1], c[3]], [0, 0, 1.0]]) for c in start])
    out = gv.bundle_adjust(host_tracks, pts, s["xy"], Ks, start[:, 4:13].reshape(-1, 3, 3), start[:, 13:], max_iters=100)
    dev = bundle.bundle_adjust_device(t, pts, xy, torch.from_numpy(start).cuda(), max_iters=100).to_host()
    assert out["status"] in bundle.STATUS_NAMES and out["final_cost"] < out["initial_cost"]
    assert np.array_equal(out["R"], dev["R"]) and np.array_equal(out["X"], dev["X"]) and out["iterations"] == dev["iterations"]
