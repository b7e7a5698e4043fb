"""Track triangulation on the GPU (csrc/triangulate.cu) against the C oracle (oracle/triangulate.c), array for array: random
tracks of 2-64 observations plus tracks of 1,000 and 100,000, outliers, unregistered images, points behind cameras, same-image
and zero-baseline views, invalid observations and every status, over a parameter sweep; then ground truth on a synthetic scene,
the two-view bridge to pose.cu's points, the pipeline path with its launch count, and empty / degenerate inputs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # collected on CPU boxes, skipped there
    pytest.skip("needs a GPU", allow_module_level=True)

import geometric_verification as gv  # noqa: E402
import sfm_b200  # noqa: E402
from oracle import triangulate_oracle as tro  # noqa: E402
from sfm_b200 import synth  # noqa: E402
from sfm_b200 import tracks as tr  # noqa: E402
from sfm_b200 import triangulate as tri  # noqa: E402

KEYS = ("X", "n_inliers", "status", "obs_inlier", "obs_error")


def device_tracks(offsets, obs, spare=5):
    """A Tracks object from host arrays, with `spare` unused slots of capacity past the last track (the kernel reads the track
    count on the device and must not look beyond it)."""
    T = len(offsets) - 1
    off = np.concatenate([offsets, np.full(spare, offsets[-1])]).astype(np.int64)
    counts = torch.tensor([T, int(offsets[-1]), 0, 0, 0], dtype=torch.int64)
    return tr.Tracks(offsets_buf=torch.from_numpy(off).cuda(), obs_buf=torch.from_numpy(np.ascontiguousarray(obs, np.int32)).cuda(),
                     track_of_buf=torch.zeros((1, 1), dtype=torch.int32, device="cuda"), counts_dev=counts.cuda())


def assert_same(got, ref):
    h = got.to_host() if isinstance(got, tri.TrackPoints) else got
    for k in KEYS:
        a, b = np.asarray(h[k]), np.asarray(ref[k])
        assert a.dtype == b.dtype and a.shape == b.shape, (k, a.shape, b.shape)
        if a.dtype.kind == "f":                                             # bit for bit, any NaN matching any NaN
            a, b = a.ravel(), b.ravel()
            assert np.array_equal(np.isnan(a), np.isnan(b)), k
            m = ~np.isnan(a)
            assert np.array_equal(a[m].view(np.uint8), b[m].view(np.uint8)), k
        else:
            assert np.array_equal(a, b), k
    ref_counts = ref["counts"].tolist() if "counts" in ref else [ref[n] for n in tri.STATUS_NAMES]
    assert [h[n] for n in tri.STATUS_NAMES] == ref_counts


def cameras():
    """14 cameras on the synthetic arc, a twin of camera 0 (same centre, rotated: zero baseline) and one looking away from the
    scene (every scene point is behind it).  Returns P [16,3,4], cams [16,16]."""
    K = synth.K_INTR
    Ps = list(synth.make_cameras(14, baseline=3.0))
    Rt0 = np.linalg.inv(K) @ Ps[0]
    c = np.array([0.05, 0.03, 0.0])
    Rz = np.array([[np.cos(c[0]), -np.sin(c[0]), 0], [np.sin(c[0]), np.cos(c[0]), 0], [0, 0, 1.0]])
    C0 = -Rt0[:, :3].T @ Rt0[:, 3]
    R1 = Rz @ Rt0[:, :3]
    Ps.append(K @ np.concatenate([R1, (-R1 @ C0)[:, None]], axis=1))
    Rb = np.diag([-1.0, 1.0, -1.0])                                     # looks along -z from (0, 0, 2)
    Ps.append(K @ np.concatenate([Rb, (-Rb @ np.array([0.0, 0.0, 2.0]))[:, None]], axis=1))
    Ps = np.stack(Ps)
    Rt = np.einsum("ij,njk->nik", np.linalg.inv(K), Ps)
    cams = np.concatenate([np.tile([K[0, 0], K[1, 1], K[0, 2], K[1, 2]], (len(Ps), 1)), Rt[:, :, :3].reshape(-1, 9), Rt[:, :, 3]], axis=1)
    return Ps, np.ascontiguousarray(cams)


def random_tracks(seed, n_tracks=600, S=8192):
    rng = np.random.default_rng(seed)
    Ps, cams = cameras()
    n_images = len(Ps)
    xy = rng.uniform([0, 0], [1920, 1080], (n_images, S, 2)).astype(np.float32)
    nxt = np.zeros(n_images, np.int64)
    offsets, obs = [0], []

    def add(imgs, X, out_frac):
        for i in imgs:
            f = int(nxt[i] % S)
            nxt[i] += 1
            if rng.random() >= out_frac:
                p = Ps[i] @ np.append(X, 1.0)
                xy[i, f] = (p[:2] / p[2] + rng.normal(0, 0.5, 2)).astype(np.float32)
            obs.append((i, f))
        offsets.append(len(obs))

    lengths = list(rng.integers(2, 65, n_tracks)) + [1000, 100_000]
    for k, L in enumerate(lengths):
        X = np.array([rng.uniform(-2, 2), rng.uniform(-2, 2), rng.uniform(4, 8)])
        kind = k % 10
        if L > 64:
            add(rng.integers(0, n_images, L), X, 0.1)
        elif kind == 0:                                                  # a lone view
            add([int(rng.integers(0, 14))], X, 0.0)
        elif kind == 1:                                                  # zero baseline: camera 0 and its twin
            add([0, 14], X, 0.0)
        elif kind == 2:                                                  # behind the last camera
            add([15, int(rng.integers(0, 14))], X, 0.0)
        elif kind == 3:                                                  # same image twice, plus others
            add(np.sort(np.concatenate([[3, 3], rng.choice(14, min(L, 14) - 2, replace=False)])), X, rng.uniform(0, 0.3))
        else:
            imgs = rng.choice(n_images, min(L, n_images), replace=False) if L <= n_images else rng.integers(0, n_images, L)
            add(np.sort(imgs), X, rng.uniform(0, 0.6))
    offsets, obs = np.array(offsets, np.int64), np.array(obs, np.int32)
    for k in rng.choice(n_tracks, 12, replace=False):                      # invalid observations
        o = offsets[k] + int(rng.integers(0, offsets[k + 1] - offsets[k]))
        obs[o] = [(n_images, 0), (-1, 0), (0, S), (2, -3)][k % 4]
    return offsets, obs, xy, cams


@pytest.fixture(scope="module")
def tracks_data():
    return {seed: random_tracks(seed) for seed in (0, 1)}


@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("min_inliers", [2, 3])
@pytest.mark.parametrize("max_error", [1.0, 4.0])
@pytest.mark.parametrize("min_angle", [0.0, 1.5, 10.0])
def test_bit_exact_vs_oracle(tracks_data, seed, min_angle, max_error, min_inliers):
    offsets, obs, xy, cams = tracks_data[seed]
    rng = np.random.default_rng([seed, int(min_angle), int(max_error), min_inliers])
    registered = None if min_inliers == 2 else (rng.random(len(cams)) > 0.2).astype(np.uint8)
    prm = dict(max_error=max_error, min_angle=min_angle, max_iters=500, confidence=0.999, seed=seed + 11, min_inliers=min_inliers)
    got = tri.triangulate_tracks_device(device_tracks(offsets, obs), torch.from_numpy(xy).cuda(), torch.from_numpy(cams).cuda(),
                                        registered, **prm)
    ref = tro.triangulate_tracks(offsets, obs, xy, cams, registered, **prm)
    assert_same(got, ref)
    c = ref["counts"]
    assert c[0] > 200 and c[1] > 0 and c[2] > 0 and c[4] == 12
    if min_inliers == 3:
        assert c[3] > 0
    st = ref["status"]
    assert st[-1] == 0 and ref["n_inliers"][-1] > 40_000 and st[-2] == 0            # the long tracks


def test_ground_truth_on_a_synthetic_scene():
    """make_scene(12, 4096) -> match_and_verify(tracks=True) -> triangulation with the true cameras.  Measured on one B200:
    3,072 tracks, all triangulated; median reprojection error of the inliers 0.526 px (pixel noise 0.5 px); median 3-D error
    0.00316 at a median depth of 6.03 (0.052 %).  Asserted: >= 99 % triangulated, median reprojection error < 1 px, median 3-D
    error < 1 % of the median depth."""
    sc = synth.make_scene(12, 4096, seed=21)
    bank = sfm_b200.DescriptorBank(12, 4096)
    bank.put(0, sc.desc, xy=sc.xy)
    res = sfm_b200.match_and_verify(bank, synth.exhaustive_pairs(12), tracks=True, max_iters=512, seed=9, solver="8pt")
    Rt = np.einsum("ij,njk->nik", np.linalg.inv(synth.K_INTR), sc.P)
    pts = gv.triangulate_tracks(res.tracks, bank, synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])
    h, t = pts.to_host(), res.tracks.to_host()
    ok = h["status"] == 0
    frac = ok.mean()
    seg = np.repeat(np.arange(t["n_tracks"]), np.diff(t["offsets"]))
    err = h["obs_error"][ok[seg] & (h["obs_inlier"] == 1)]
    pid = sc.point[t["obs"][t["offsets"][:-1], 0], t["obs"][t["offsets"][:-1], 1]]
    d3 = np.linalg.norm(h["X"][ok] - sc.X[pid[ok]], axis=1)
    depth = np.median(sc.X[pid[ok]] @ Rt[0, 2, :3] + Rt[0, 2, 3])                 # in camera 0
    print(f"\n{t['n_tracks']} tracks: {frac:.4f} triangulated, median reprojection error {np.median(err):.3f} px, "
          f"median 3-D error {np.median(d3):.5f} (median depth {depth:.2f}: {100 * np.median(d3) / depth:.4f} %), "
          f"statuses {[h[n] for n in tri.STATUS_NAMES]}")
    assert frac >= 0.99
    assert np.median(err) < 1.0
    assert np.median(d3) < 0.01 * depth


def test_two_view_bridge_reproduces_pose_points():
    """Two images, cameras [I|0] and recover_pose's (R, t): each track's point equals pose.cu's points3d of its match row
    (measured on one B200: all 683 compared points equal exactly in float32; asserted with rtol 1e-6)."""
    sc = synth.make_scene(2, 2048, seed=3)
    bank = sfm_b200.DescriptorBank(2, 2048)
    bank.put(0, sc.desc, xy=sc.xy)
    res = sfm_b200.match_and_verify(bank, [[0, 1]], fetch=True, tracks=True, intrinsics=synth.K_INTR, max_iters=512, seed=5, solver="7pt",
                                    lo=True)
    h = res.to_host()
    R, t = h["R"][0], h["t"][0]
    pts = gv.triangulate_tracks(res.tracks, bank, synth.K_INTR, np.stack([np.eye(3), R]), np.stack([np.zeros(3), t]),
                                registered=[1, 1]).to_host()
    track_of = res.tracks.track_of.cpu().numpy()
    m, front = h["matches"], h["in_front"].astype(bool)
    k = track_of[0, m[front, 0]]
    same = (k >= 0) & (k == track_of[1, m[front, 1]])      # rows whose two features form one track (not a dropped conflict)
    ok = same & (pts["status"][np.maximum(k, 0)] == 0)
    assert ok.mean() > 0.95
    got = pts["X"][k[ok]].astype(np.float32)
    want = h["points3d"][front][ok]
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=0)
    print(f"\n{ok.sum()} tracks: {np.mean(np.all(got == want, axis=1)):.4f} of the points equal pose.cu's float32 points exactly")


def test_pipeline_path_launches_and_equals_host_tracks():
    sc = synth.make_scene(12, 4096, seed=21)
    bank = sfm_b200.DescriptorBank(12, 4096)
    bank.put(0, sc.desc, xy=sc.xy)
    pairs = synth.exhaustive_pairs(12)
    Rt = np.einsum("ij,njk->nik", np.linalg.inv(synth.K_INTR), sc.P)
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])).cuda()
    reg = torch.ones(12, dtype=torch.uint8, device="cuda")
    reg[5] = 0
    torch.cuda.synchronize()
    res = sfm_b200.match_and_verify(bank, pairs, fetch=True, tracks=True, max_iters=512, seed=9, solver="8pt")
    n0 = sfm_b200.launch_count()
    pts = sfm_b200.triangulate_tracks_device(res.tracks, bank.xy, cams, reg, S=bank.max_feats, seed=4)
    assert sfm_b200.launch_count() - n0 == tri.TRIANGULATE_LAUNCHES
    host_tracks = gv.build_tracks(res.to_host(), 12, 4096).to_host()
    ref = gv.triangulate_tracks(host_tracks, sc.xy, synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3], registered=reg.cpu().numpy(), seed=4)
    assert_same(pts, ref.to_host())
    assert pts.counts["triangulated"] > 1000


def test_empty_and_degenerate_inputs():
    Ps, cams = cameras()
    cams_d = torch.from_numpy(cams).cuda()
    xy = torch.zeros((len(cams), 64, 2), dtype=torch.float32, device="cuda")
    z = np.zeros(0, np.int32)
    empty = sfm_b200.build_tracks_device(z, z, z, np.zeros((0, 3), np.int32), None, None, len(cams), 64)
    e = tri.triangulate_tracks_device(empty, xy, cams_d).to_host()
    assert e["X"].shape == (0, 3) and e["obs_error"].shape == (0,) and all(e[n] == 0 for n in tri.STATUS_NAMES)
    offsets, obs, xyh, _ = random_tracks(5, n_tracks=50, S=64)
    offsets, obs = offsets[:51], obs[: offsets[50]]
    none = np.zeros(len(cams), np.uint8)
    got = tri.triangulate_tracks_device(device_tracks(offsets, obs), torch.from_numpy(xyh).cuda(), cams_d, none)
    ref = tro.triangulate_tracks(offsets, obs, xyh, cams, none)
    assert_same(got, ref)
    st = got.to_host()["status"]
    assert (st == 4).sum() == 12 and (st == 1).sum() == 38 and np.isnan(got.to_host()["obs_error"]).all()
