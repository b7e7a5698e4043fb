"""Incremental reconstruction on the GPU (csrc/mapper.cu, sfm_b200/mapper.py): sfm_next_images and sfm_filter_points against
the numpy oracle (oracle/mapper_oracle.py) bit for bit; reconstruct_device end to end on a ring of cameras that each see only
their own frustum, against the same loop written here from the public device calls and against the ground truth; determinism
and the per-round launch count; disconnected scenes, scenes without an initial pair, an explicit initial pair and the
argument checks.  Measured numbers are printed and recorded in DESIGN §4 "Incremental reconstruction"."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # collected on CPU boxes, skipped there
    pytest.skip("needs a GPU", allow_module_level=True)

from scipy.spatial.transform import Rotation  # noqa: E402

import geometric_verification as gv  # noqa: E402
import sfm_b200  # noqa: E402
from oracle import mapper_oracle as mo  # noqa: E402
from sfm_b200 import bundle, mapper, pnp, synth  # noqa: E402
from sfm_b200 import triangulate as tri  # noqa: E402
from sfm_b200 import tracks as tr  # noqa: E402

K = synth.K_INTR
N_FEATS = 2048
# Measured on one B200 at a 1,000 W power limit on the 24-camera ring (DESIGN §4 "Incremental reconstruction"); the bounds
# are ceilings well above the measurement.
ROT_DEG = 0.05          # measured 0.0155 degree (median rotation error after a similarity alignment)
CEN_PCT = 0.2           # measured 0.054 % of the ring radius (median centre error)
RMS_PX = 0.6            # measured 0.427 px over the inlier observations (pixel noise 0.5 px per coordinate)


def ring_scene(n_cams, *, seed, radius=10.0, centre=(0.0, 0.0, 0.0), n_points=12000, max_seen=1200):
    """Cameras on a horizontal circle looking outward at points on a surrounding cylinder (radius + 4 to radius + 8, heights
    -2 to 2): each camera sees only its own frustum, so tracks chain across neighbours and distant cameras share nothing.
    ``radius`` 0 puts every camera at one centre (pure rotation)."""
    rng = np.random.default_rng(seed)
    c0 = np.asarray(centre, np.float64)
    phi = rng.uniform(0, 2 * np.pi, n_points)
    rr = radius + rng.uniform(4.0, 8.0, n_points)
    X = np.stack([rr * np.sin(phi), rng.uniform(-2.0, 2.0, n_points), rr * np.cos(phi)], 1) + c0
    base = synth.sift_like(rng, n_points)
    P = np.zeros((n_cams, 3, 4))
    desc = np.empty((n_cams, N_FEATS, 128), np.uint8)
    xy = np.empty((n_cams, N_FEATS, 2), np.float32)
    for i in range(n_cams):
        a = 2 * np.pi * i / n_cams
        C = c0 + radius * np.array([np.sin(a), 0.0, np.cos(a)])
        z = np.array([np.sin(a), 0.0, np.cos(a)])
        x = np.cross([0.0, 1.0, 0.0], z)
        R = np.stack([x, np.cross(z, x), z])
        t = -R @ C
        P[i] = K @ np.concatenate([R, t[:, None]], 1)
        q = (P[i] @ np.concatenate([X, np.ones((n_points, 1))], 1).T).T
        px = q[:, :2] / q[:, 2:3]
        seen = np.nonzero((q[:, 2] > 0.5) & (px[:, 0] >= 0) & (px[:, 0] < synth.IMG_W) & (px[:, 1] >= 0) & (px[:, 1] < synth.IMG_H))[0]
        seen = rng.permutation(seen)[:max_seen]
        slot = rng.permutation(N_FEATS)
        s_sh, s_cl = slot[: len(seen)], slot[len(seen):]
        desc[i, s_sh] = synth.observe(rng, base[seen])
        xy[i, s_sh] = (px[seen] + rng.normal(0.0, 0.5, (len(seen), 2))).astype(np.float32)
        desc[i, s_cl] = synth.sift_like(rng, len(s_cl))
        xy[i, s_cl] = rng.uniform([0, 0], [synth.IMG_W, synth.IMG_H], (len(s_cl), 2)).astype(np.float32)
    return desc, xy, P, X


def verified(desc, xy, *, keep_conflicts=False):
    n = desc.shape[0]
    bank = sfm_b200.DescriptorBank(n, N_FEATS)
    bank.put(0, desc, xy=xy)
    res = sfm_b200.match_and_verify(bank, synth.exhaustive_pairs(n), tracks=True, homography=True, intrinsics=K, max_iters=512,
                                    seed=9, solver="8pt", keep_conflicts=keep_conflicts)
    return bank, res


@pytest.fixture(scope="module")
def ring():
    desc, xy, P, X = ring_scene(24, seed=11)
    bank, res = verified(desc, xy)
    Rt = np.einsum("ij,njk->nik", np.linalg.inv(K), P)
    return bank, res, Rt, xy


def umeyama(src, dst):
    ms, md = src.mean(0), dst.mean(0)
    a, b = src - ms, dst - md
    U, D, Vt = np.linalg.svd(b.T @ a / len(src))
    S = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        S[2, 2] = -1
    Q = U @ S @ Vt
    s = np.trace(np.diag(D) @ S) / a.var(0).sum()
    return s, Q, md - s * Q @ ms


def errors(R, t, Rt, idx):
    """Median rotation error (degrees) and median centre error (% of the ring radius) of images idx after a similarity
    alignment of the centres."""
    C_est = np.stack([-R[i].T @ t[i] for i in idx])
    C_true = np.stack([-Rt[i, :, :3].T @ Rt[i, :, 3] for i in idx])
    s, Q, c = umeyama(C_est, C_true)
    cen = np.linalg.norm((s * (Q @ C_est.T)).T + c - C_true, axis=1)
    rot = [np.degrees(Rotation.from_matrix(R[i] @ Q.T @ Rt[i, :, :3].T).magnitude()) for i in idx]
    return float(np.median(rot)), float(np.median(cen) / 10.0 * 100)


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def host_points(p):
    h = p.to_host()
    return {k: h[k] for k in ("X", "n_inliers", "status", "obs_inlier", "obs_error")}


# ------------------------------------------------------------------------------------------------------ sfm_next_images
def check_next(tracks, points, xy, registered, trials, size, **prm):
    """Run sfm_next_images and its oracle on the same inputs; every output equal, out_visible equal to the gather's counts."""
    n = int(tracks.track_of_buf.shape[0])
    tr_h = trials.cpu().numpy()
    ref = mo.next_images(tracks.track_of_buf.cpu().numpy(), min(int(tracks.counts_dev[0]), points.status_buf.numel()),
                         points.status_buf.cpu().numpy(), xy[:n].cpu().numpy(), size.cpu().numpy(), registered.cpu().numpy(), tr_h, **prm)
    got = mapper.next_images_device(tracks, points, xy, registered, trials, image_size=size, **prm).to_host()
    for k in ("images", "visible", "score", "n_selected"):
        assert same(got[k], ref[k]) if k != "n_selected" else got[k] == ref[k], (k, got[k], ref[k])
    assert same(trials.cpu().numpy(), ref["trials"])
    _, _, _, count = pnp.gather_device(tracks, points, xy, np.arange(n))
    assert same(count.cpu().numpy(), got["visible"])
    return got


def test_next_images_equals_the_oracle(ring):
    bank, res, Rt, _ = ring
    trk = res.tracks
    cams = torch.from_numpy(tri.camera_table(K, Rt[:, :, :3], Rt[:, :, 3])).cuda()
    size = mapper.image_sizes(cams)
    for subset in ([0, 1], [0, 1, 2, 3], list(range(0, 24, 2)), list(range(10))):
        reg = torch.zeros(24, dtype=torch.uint8, device="cuda")
        reg[subset] = 1
        pts = tri.triangulate_tracks_device(trk, bank.xy, cams, reg, S=bank.max_feats)
        trials = torch.zeros(24, dtype=torch.int32, device="cuda")
        trials[5] = 3
        for max_select in (1, 4, 16, 64):
            got = check_next(trk, pts, bank.xy, reg, trials, size, max_select=max_select)
            assert 5 not in got["images"].tolist()
        for prm in (dict(max_select=8, min_visible=0, max_trials=100), dict(max_select=3, levels=1), dict(max_select=5, levels=8)):
            check_next(trk, pts, bank.xy, reg, torch.zeros(24, dtype=torch.int32, device="cuda"), size, **prm)
    # keep_conflicts tracks, and an image whose features are all clutter (no tracks)
    desc, xy, P, X = ring_scene(12, seed=5, n_points=6000)
    desc[7] = synth.sift_like(np.random.default_rng(1), N_FEATS)
    bank2, res2 = verified(desc, xy, keep_conflicts=True)
    Rt2 = np.einsum("ij,njk->nik", np.linalg.inv(K), P)
    cams2 = torch.from_numpy(tri.camera_table(K, Rt2[:, :, :3], Rt2[:, :, 3])).cuda()
    reg2 = torch.zeros(12, dtype=torch.uint8, device="cuda")
    reg2[[0, 1, 2]] = 1
    pts2 = tri.triangulate_tracks_device(res2.tracks, bank2.xy, cams2, reg2, S=bank2.max_feats)
    check_next(res2.tracks, pts2, bank2.xy, reg2, torch.zeros(12, dtype=torch.int32, device="cuda"), mapper.image_sizes(cams2),
               max_select=12, min_visible=0)


def synthetic_tracks(n_images, S, seed):
    """Random track_of / point status / xy (with NaN, negative, past-the-edge coordinates, zero-feature images and score ties)
    for the selection alone: sfm_next_images reads nothing else."""
    rng = np.random.default_rng(seed)
    T = 5000
    track_of = rng.integers(-1, T + 50, (n_images, S)).astype(np.int32)
    track_of[rng.random(n_images) < 0.1] = -1
    track_of[:: 7] = track_of[0]                                # identical rows: score and visible ties
    xy = rng.uniform(-50, 700, (n_images, S, 2)).astype(np.float32)
    xy[:: 7] = xy[0]
    xy[rng.random((n_images, S)) < 0.01] = np.nan
    status = rng.integers(0, 5, T + 64).astype(np.uint8)
    status[rng.random(T + 64) < 0.6] = 0
    dev = torch.device("cuda")
    t = tr.Tracks(offsets_buf=torch.zeros(T + 1, dtype=torch.int64, device=dev), obs_buf=torch.zeros((1, 2), dtype=torch.int32, device=dev),
                  track_of_buf=torch.from_numpy(track_of).to(dev), counts_dev=torch.tensor([T, 0, 0, 0, 0], dtype=torch.int64, device=dev))
    p = tri.TrackPoints(tracks=t, X_buf=torch.zeros((T + 64, 3), dtype=torch.float64, device=dev),
                        n_inliers_buf=torch.zeros(T + 64, dtype=torch.int32, device=dev), status_buf=torch.from_numpy(status).to(dev),
                        obs_inlier_buf=torch.zeros(1, dtype=torch.uint8, device=dev), obs_error_buf=torch.zeros(1, dtype=torch.float32, device=dev),
                        counts_dev=torch.zeros(5, dtype=torch.int64, device=dev))
    size = torch.from_numpy(np.tile([640, 480], (n_images, 1)).astype(np.int32)).to(dev)
    return t, p, torch.from_numpy(xy).to(dev), size


@pytest.mark.parametrize("n_images", [1, 2, 37, 1024])
def test_next_images_sizes_and_ties(n_images):
    t, p, xy, size = synthetic_tracks(n_images, 256, seed=n_images)
    rng = np.random.default_rng(n_images)
    reg = torch.from_numpy((rng.random(n_images) < 0.3).astype(np.uint8)).cuda()
    trials = torch.from_numpy(rng.integers(0, 4, n_images).astype(np.int32)).cuda()
    for prm in (dict(max_select=16, min_visible=10), dict(max_select=2000, min_visible=0), dict(max_select=1, min_visible=50, levels=3)):
        check_next(t, p, xy, reg, trials, size, **prm)
    if n_images == 1024:
        with pytest.raises(ValueError, match="1 to 1024"):
            t2, p2, xy2, size2 = synthetic_tracks(1025, 8, seed=0)
            mapper.next_images_device(t2, p2, xy2, torch.zeros(1025, dtype=torch.uint8, device="cuda"),
                                      torch.zeros(1025, dtype=torch.int32, device="cuda"), image_size=size2)


# ------------------------------------------------------------------------------------------------------ sfm_filter_points
def test_filter_points_equals_the_oracle(ring):
    bank, res, Rt, _ = ring
    trk = res.tracks
    rng = np.random.default_rng(3)
    R0, t0 = Rt[:, :, :3].copy(), Rt[:, :, 3].copy()
    for i in range(1, 24):
        C = -R0[i].T @ t0[i] + rng.normal(size=3) * 0.02
        R0[i] = Rotation.from_rotvec(rng.normal(size=3) * np.radians(0.3)).as_matrix() @ R0[i]
        t0[i] = -R0[i] @ C
    cams = torch.from_numpy(tri.camera_table(K, R0, t0)).cuda()
    reg = torch.ones(24, dtype=torch.uint8, device="cuda")
    reg[[5, 17]] = 0
    pts = tri.triangulate_tracks_device(trk, bank.xy, cams, reg, S=bank.max_feats)
    bundle.bundle_adjust_device(trk, pts, bank.xy, cams, reg, update=True, S=bank.max_feats)
    # injected errors: NaN, +inf, exactly 4, one ulp above, large, on a fifth of the observations
    err = pts.obs_error.clone()
    n_obs = err.numel()
    pick = torch.from_numpy(rng.choice(n_obs, n_obs // 5, replace=False)).cuda()
    four = np.float32(4.0)
    vals = torch.tensor([np.nan, np.inf, four, np.nextafter(four, np.float32(np.inf)), 50.0, 3.999], dtype=torch.float32, device="cuda")
    err[pick] = vals[torch.arange(pick.numel(), device="cuda") % vals.numel()]
    pts.obs_error_buf[:n_obs] = err
    reg_f = reg.clone()
    reg_f[9] = 0                                               # an image that the filter no longer counts
    th = trk.to_host()
    before = host_points(pts)
    for prm in (dict(), dict(min_angle=10.0), dict(min_inliers=4, max_error=2.0)):
        p = tri.TrackPoints(tracks=trk, X_buf=pts.X_buf.clone(), n_inliers_buf=pts.n_inliers_buf.clone(), status_buf=pts.status_buf.clone(),
                            obs_inlier_buf=pts.obs_inlier_buf.clone(), obs_error_buf=pts.obs_error_buf.clone(), counts_dev=pts.counts_dev.clone())
        torch.cuda.synchronize()
        n0 = sfm_b200.launch_count()
        mapper.filter_points_device(p, cams, reg_f, **prm)
        assert sfm_b200.launch_count() - n0 == mapper.FILTER_LAUNCHES
        ref = mo.filter_points(th["offsets"], th["obs"], cams.cpu().numpy(), reg_f.cpu().numpy(), before["X"], before["n_inliers"],
                               before["status"], before["obs_inlier"], before["obs_error"], **prm)
        h = host_points(p)
        for k in ("X", "n_inliers", "status", "obs_inlier"):
            assert same(h[k], ref[k]), k
        assert same(h["obs_error"], before["obs_error"])
        c = p.counts
        assert [c[n] for n in tri.STATUS_NAMES] == ref["counts"].tolist() == np.bincount(h["status"], minlength=5).tolist()
        # triangulation's invariants
        bad = h["status"] != 0
        assert not h["X"][bad].any() and not h["n_inliers"][h["status"] == 2].any()
        owner = np.repeat(np.arange(len(h["status"])), np.diff(th["offsets"]))
        assert not h["obs_inlier"][bad[owner]].any()
        ok = h["status"] == 0
        assert (h["n_inliers"][ok] >= prm.get("min_inliers", 2)).all()
        assert (np.bincount(owner, weights=h["obs_inlier"], minlength=len(ok))[ok] == h["n_inliers"][ok]).all()
        e = h["obs_error"][h["obs_inlier"] == 1].astype(np.float64)
        assert (e <= prm.get("max_error", 4.0)).all()
        print(f"\nfilter {prm}: {dict(c)}; inlier observations {int(before['obs_inlier'].sum())} -> {int(h['obs_inlier'].sum())}")


# ------------------------------------------------------------------------------------------------------ reconstruct_device
def manual_loop(res, xy, *, init_pair, max_per_round=16, check_oracle=True):
    """reconstruct_device with init_pair given, restated from the public device calls (and each round's selection checked
    against the oracle on that round's inputs)."""
    trk = res.tracks
    n = int(xy.shape[0])
    S = int(trk.track_of_buf.shape[1])
    pairs = res.pairs.cpu().numpy()
    p = int(np.nonzero((pairs[:, 0] == init_pair[0]) & (pairs[:, 1] == init_pair[1]))[0][0])
    i, j = init_pair
    R = np.tile(np.eye(3), (n, 1, 1))
    t = np.zeros((n, 3))
    R[j], t[j] = res.R[p].cpu().numpy(), res.t[p].cpu().numpy()
    cams = torch.from_numpy(tri.camera_table(K, R, t)).cuda()
    reg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    reg[[i, j]] = 1
    fixed = torch.zeros(n, dtype=torch.uint8, device="cuda")
    fixed[i] = 1
    pts = tri.triangulate_tracks_device(trk, xy, cams, reg, S=S)
    bundle.bundle_adjust_device(trk, pts, xy, cams, reg, fixed=fixed, update=True, S=S)
    mapper.filter_points_device(pts, cams, reg)
    trials = torch.zeros(n, dtype=torch.int32, device="cuda")
    size = mapper.image_sizes(cams)
    launches = []
    while True:
        if check_oracle:
            check_next(trk, pts, xy, reg, trials.clone(), size, max_select=max_per_round)
        torch.cuda.synchronize()
        n0 = sfm_b200.launch_count()
        nxt = mapper.next_images_device(trk, pts, xy, reg, trials, image_size=size, max_select=max_per_round)
        out = pnp.register_images_device(trk, pts, xy, cams, nxt.images, update=True, registered=reg)
        n_sel, n_reg = int(nxt.n_selected.cpu()[0]), out.counts["registered"]
        if n_sel == 0:
            break
        if n_reg:
            pts = tri.triangulate_tracks_device(trk, xy, cams, reg, S=S)
            bundle.bundle_adjust_device(trk, pts, xy, cams, reg, fixed=fixed, update=True, S=S)
            mapper.filter_points_device(pts, cams, reg)
        launches.append((n_reg, sfm_b200.launch_count() - n0))
    return cams, reg, pts, launches


def test_reconstruct_ring_end_to_end(ring):
    bank, res, Rt, xy_h = ring
    torch.cuda.synchronize()
    n0 = sfm_b200.launch_count()
    rec = mapper.reconstruct_device(res, bank.xy, K)
    launched = sfm_b200.launch_count() - n0
    h = rec.to_host()
    print(f"\nring of 24: init pair {h['init_pair']}, {len(h['rounds']) - 1} rounds, round of each image {h['round'].tolist()}")
    for e in h["rounds"]:
        print(f"  {e}")
    assert h["status"] == "ok" and h["registered"].all() and (h["round"] >= 0).all()
    i, j = h["init_pair"]
    assert h["round"][i] == 0 and h["round"][j] == 0
    # points: every status-0 point has >= 2 inliers, every inlier error <= 4 px
    th = res.tracks.to_host()
    owner = np.repeat(np.arange(len(h["point_status"])), np.diff(th["offsets"]))
    ok = h["point_status"] == 0
    n_inl = np.bincount(owner, weights=h["obs_inlier"], minlength=len(ok))
    assert (n_inl[ok] >= 2).all() and not h["obs_inlier"][~ok[owner]].any()
    e = h["obs_error"][h["obs_inlier"] == 1].astype(np.float64)
    assert (e <= 4.0).all()
    rms = float(np.sqrt(np.mean(e ** 2)))
    rot, cen = errors(h["R"], h["t"], Rt, range(24))
    print(f"  {int(ok.sum())} points, {len(e)} inlier observations, RMS {rms:.4f} px; after a similarity alignment: rotation error "
          f"median {rot:.5f} deg, centre error median {cen:.5f} % of the ring radius; {launched} launches")
    assert rot < ROT_DEG and cen < CEN_PCT and rms < RMS_PX
    # the same loop from the public device calls, with each round's selection checked against the oracle: bit-identical
    cams, reg, pts, launches = manual_loop(res, bank.xy, init_pair=(i, j))
    assert same(cams.cpu().numpy(), rec.cams.cpu().numpy()) and same(reg.cpu().numpy(), h["registered"])
    mh = host_points(pts)
    for k in ("X", "obs_inlier", "obs_error"):
        assert same(mh[k], h[k]), k
    assert same(mh["status"], h["point_status"])
    # the per-round launch count: a registering round is round_launches(50), any other NEXT_IMAGES_LAUNCHES + PNP_LAUNCHES
    for n_reg, n in launches:
        assert n == (mapper.round_launches(50) if n_reg else mapper.NEXT_IMAGES_LAUNCHES + pnp.PNP_LAUNCHES), (n_reg, n)
    # reconstruct_device's whole count: the candidates it triangulated, the initial adjustment and filter, then the rounds
    n_tried = launched - 1 - bundle.bundle_launches(50) - sum(n for _, n in launches) - mapper.NEXT_IMAGES_LAUNCHES - pnp.PNP_LAUNCHES
    assert 1 <= n_tried <= 10


def test_reconstruct_is_deterministic_and_stream_independent(ring):
    bank, res, Rt, _ = ring
    a = mapper.reconstruct_device(res, bank.xy, K, max_per_round=4).to_host()
    b = mapper.reconstruct_device(res, bank.xy, K, max_per_round=4).to_host()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c = mapper.reconstruct_device(res, bank.xy, K, max_per_round=4)
    torch.cuda.current_stream().wait_stream(s)
    c = c.to_host()
    for other in (b, c):
        for k in ("R", "t", "registered", "round", "X", "point_status", "obs_inlier", "obs_error"):
            assert same(a[k], other[k]), k
        assert a["rounds"] == other["rounds"] and a["init_pair"] == other["init_pair"]
    # the public drop-in call returns the same
    g = gv.reconstruct(res, bank, K, max_per_round=4)
    assert same(g["R"], a["R"]) and same(g["X"], a["X"]) and g["status"] == "ok"


def test_explicit_init_pair_and_no_initial_pair(ring):
    bank, res, Rt, _ = ring
    auto = mapper.reconstruct_device(res, bank.xy, K).init_pair
    order = mapper.initial_pair_order(res.n_pose.cpu().numpy(), res.n_inliers.cpu().numpy(), res.n_inliers_h.cpu().numpy())
    pairs = res.pairs.cpu().numpy()
    other = next(tuple(int(v) for v in pairs[p]) for p in order if tuple(pairs[p]) != auto)
    rec = mapper.reconstruct_device(res, bank.xy, K, init_pair=other)
    h = rec.to_host()
    print(f"\nexplicit initial pair {other} (the search takes {auto}): {int(h['registered'].sum())} of 24 registered in "
          f"{len(h['rounds']) - 1} rounds")
    assert h["init_pair"] == other and h["round"][other[0]] == 0 and h["round"][other[1]] == 0
    assert h["rounds"][0]["selected"] == list(other)
    # the reversed order names the stored pair
    assert mapper.reconstruct_device(res, bank.xy, K, init_pair=other[::-1]).init_pair == other
    none = mapper.reconstruct_device(res, bank.xy, K, init_min_inliers=10 ** 6).to_host()
    assert none["status"] == "no_initial_pair" and none["init_pair"] is None and (none["round"] == -1).all() and not none["registered"].any()
    with pytest.raises(ValueError, match="init_pair"):
        mapper.reconstruct_device(res, bank.xy, K, init_pair=(0, 99))


def test_pure_rotation_scene_has_no_initial_pair():
    desc, xy, P, X = ring_scene(8, seed=4, radius=0.0, n_points=6000)
    bank, res = verified(desc, xy)
    h = gv.reconstruct(res, bank, K)
    assert h["status"] == "no_initial_pair" and (h["round"] == -1).all()


def test_two_disconnected_rings():
    da, xa, Pa, _ = ring_scene(24, seed=6)
    db, xb, Pb, _ = ring_scene(24, seed=7, centre=(500.0, 0.0, 0.0))
    bank, res = verified(np.concatenate([da, db]), np.concatenate([xa, xb]))
    h = mapper.reconstruct_device(res, bank.xy, K).to_host()
    i, j = h["init_pair"]
    comp = slice(0, 24) if i < 24 else slice(24, 48)
    other = slice(24, 48) if i < 24 else slice(0, 24)
    print(f"\ntwo rings: initial pair {(i, j)}, registered {np.nonzero(h['registered'])[0].tolist()}")
    assert h["registered"][comp].all() and (h["round"][comp] >= 0).all()
    assert not h["registered"][other].any() and (h["round"][other] == -1).all()


def test_argument_errors(ring):
    bank, res, Rt, _ = ring
    no_tracks = sfm_b200.match_and_verify(bank, [[0, 1]], intrinsics=K)
    with pytest.raises(ValueError, match="tracks"):
        mapper.reconstruct_device(no_tracks, bank.xy, K)
    no_pose = sfm_b200.match_and_verify(bank, [[0, 1], [1, 2]], tracks=True)
    with pytest.raises(ValueError, match="pose"):
        mapper.reconstruct_device(no_pose, bank.xy, K)
    with pytest.raises(ValueError, match="1024"):
        mapper.reconstruct_device(res, torch.zeros((1025, N_FEATS, 2), dtype=torch.float32, device="cuda"), K)
