"""Registration on the GPU (csrc/pnp.cu) against the C oracle (oracle/pnp.c), array for array: queries of 0 to 20,000
correspondences (past the shared-memory stage), outlier fractions 0 to 0.9, points behind the camera, collinear and coplanar
points, invalid images and intrinsics and every status, over a parameter sweep; batch independence; the gather against its numpy
oracle on pipeline tracks; ground truth on a synthetic scene; an incremental reconstruction loop on the device; the pipeline path
with its launch count; and empty / degenerate inputs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # collected on CPU boxes, skipped there
    pytest.skip("needs a GPU", allow_module_level=True)

import geometric_verification as gv  # noqa: E402
import sfm_b200  # noqa: E402
from oracle import pnp_oracle as po  # noqa: E402
from sfm_b200 import pnp  # noqa: E402
from sfm_b200 import synth  # noqa: E402
from sfm_b200 import triangulate as tri  # noqa: E402

KEYS = ("pose", "n_inliers", "status", "mask", "iters")


def assert_same(got, ref):
    h = got.to_host()
    for k in KEYS:
        a, b = np.asarray(h[k]), np.asarray(ref[k])
        assert a.dtype == b.dtype and a.shape == b.shape, (k, a.shape, b.shape)
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (k, np.nonzero(np.any((a != b).reshape(len(a), -1), axis=1))[0][:10])
    assert [h[n] for n in pnp.STATUS_NAMES] == ref["counts"].tolist()


def random_rotation(rng):
    q = rng.normal(size=4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def make_queries(seed):
    """A batch of queries, one per image.  Returns xy [Q, stride, 2], X [Q, stride, 3], count [Q], cams [n_images, 16], image [Q]."""
    rng = np.random.default_rng(seed)
    n_images = 40
    cams = np.zeros((n_images, 16))
    cams[:, :4] = [1000.0, 1000.0, 960.0, 540.0]
    cams[:, 4:13] = np.eye(3).ravel()
    cams[30, 0] = 0.0                                                   # invalid intrinsics
    cams[31, 1] = np.inf
    cams[32, 0] = np.nan
    cams[33, 1] = -1000.0
    queries = []                                                        # (image, Xc camera-frame points, outlier mask, world transform)

    def add(img, M, outlier_frac=0.0, behind=0.0, kind="scene"):
        Xc = np.stack([rng.uniform(-2, 2, M), rng.uniform(-1.2, 1.2, M), rng.uniform(4, 8, M)], 1)
        if kind == "coplanar":
            Xc[:, 2] = 6.0 + 0.3 * Xc[:, 0]
        px = Xc[:, :2] / Xc[:, 2:] * 1000.0 + [960, 540]
        px = px + rng.normal(0, 0.5, (M, 2))
        out = rng.random(M) < outlier_frac
        px[out] += rng.choice([-1, 1], (out.sum(), 2)) * rng.uniform(20, 400, (out.sum(), 2))
        back = rng.random(M) < behind
        Xc[back] *= [1, 1, -1]                                           # same ray direction up to sign, behind the camera
        R, t = random_rotation(rng), rng.normal(size=3)
        Xw = (Xc - t) @ R
        if kind == "collinear":
            Xw = np.stack([np.full(M, 1.5), np.full(M, -0.5), np.linspace(4, 8, M)], 1)     # exactly: every sample degenerate
        queries.append((img, px.astype(np.float32), Xw))

    add(0, 0)
    add(1, 2)
    add(2, 3)
    add(3, 4)
    add(4, 4096)
    add(5, 4096, 0.3)
    add(6, 4096, 0.6)
    add(7, 1000, 0.9)
    add(8, 20_000, 0.4)                                                  # beyond the shared-memory stage
    add(9, 600, 0.2, behind=0.3)
    add(10, 300, kind="collinear")
    add(11, 500, 0.2, kind="coplanar")
    add(12, 40, 0.85)                                                    # a handful of inliers
    add(13, 200, 0.7)
    for img in (30, 31, 32, 33, -1, n_images, 1 << 20):
        add(img, 100)
    add(14, 64, 1.0)                                                     # outliers only
    stride = max(len(p) for _, p, _ in queries)
    Q = len(queries)
    xy = np.zeros((Q, stride, 2), np.float32)
    X = np.zeros((Q, stride, 3), np.float64)
    count = np.zeros(Q, np.int32)
    for q, (img, p, Xw) in enumerate(queries):
        xy[q, : len(p)] = p
        X[q, : len(p)] = Xw
        count[q] = len(p)
    image = np.array([img for img, _, _ in queries], np.int32)
    return xy, X, count, cams, image


@pytest.fixture(scope="module")
def queries():
    return make_queries(0)


def run_gpu(xy, X, count, cams, image, **prm):
    return pnp.pnp_ransac_device(torch.from_numpy(xy).cuda(), torch.from_numpy(X).cuda(), torch.from_numpy(count).cuda(),
                                 torch.from_numpy(cams).cuda(), image, **prm)


SWEEP = [dict(max_error=12.0, confidence=0.9999, min_inliers=30, min_inlier_ratio=0.25, refine_iters=10),
         dict(max_error=2.0, confidence=0.99, min_inliers=3, min_inlier_ratio=0.0, refine_iters=0),
         dict(max_error=12.0, confidence=0.99, min_inliers=100, min_inlier_ratio=0.5, refine_iters=10),
         dict(max_error=4.0, confidence=0.9999, min_inliers=3, min_inlier_ratio=0.0, refine_iters=10),
         dict(max_error=12.0, confidence=1.0, min_inliers=3, min_inlier_ratio=0.25, refine_iters=0, max_iters=300)]


@pytest.mark.parametrize("case", range(len(SWEEP)))
def test_bit_exact_vs_oracle(queries, case):
    xy, X, count, cams, image = queries
    prm = dict(max_iters=2000, seed=case + 7, **SWEEP[case]) if "max_iters" not in SWEEP[case] else dict(seed=case + 7, **SWEEP[case])
    got = run_gpu(xy, X, count, cams, image, **prm)
    ref = po.pnp_ransac(xy, X, count, cams, image, **prm)
    assert_same(got, ref)
    st, c = ref["status"], ref["counts"]
    assert st[:2].tolist() == [1, 1] and st[10] == 2 and c[4] == 7 and c[2] >= 1
    assert st[4] == 0 and st[5] == 0 and st[8] == 0 and st[11] == 0
    assert ref["n_inliers"][8] > 9000
    if SWEEP[case]["min_inliers"] >= 30 or SWEEP[case]["min_inlier_ratio"] >= 0.25:
        assert c[3] > 0
    print(f"\ncase {case}: statuses {c.tolist()}, hypotheses {ref['iters'].tolist()}")


def test_batch_independence(queries):
    """A query alone, in a permuted batch and in a larger batch (with a second copy of the whole set under other image ids)
    gives the same bits: the sampler's stream is the image id."""
    xy, X, count, cams, image = queries
    prm = dict(max_iters=500, seed=3)
    full = run_gpu(xy, X, count, cams, image, **prm).to_host()
    perm = np.random.default_rng(1).permutation(len(image))
    p = run_gpu(xy[perm], X[perm], count[perm], cams, image[perm], **prm).to_host()
    cams2 = np.concatenate([cams, cams])
    img2 = np.concatenate([image, np.where((image >= 0) & (image < 40), image + 40, image)]).astype(np.int32)
    big = run_gpu(np.concatenate([xy, xy[::-1]]), np.concatenate([X, X[::-1]]), np.concatenate([count, count[::-1]]), cams2,
                  np.concatenate([image, img2[len(image):][::-1]]), **prm).to_host()
    for q in (2, 5, 8, 9, 12):
        alone = run_gpu(xy[q: q + 1], X[q: q + 1], count[q: q + 1], cams, image[q: q + 1], **prm).to_host()
        j = int(np.nonzero(perm == q)[0][0])
        for k in KEYS:
            a = alone[k][:1].view(np.uint8)
            assert np.array_equal(a, full[k][q: q + 1].view(np.uint8)), (q, k)
            assert np.array_equal(a, p[k][j: j + 1].view(np.uint8)), (q, k)
            assert np.array_equal(a, big[k][q: q + 1].view(np.uint8)), (q, k)


@pytest.fixture(scope="module")
def scene():
    sc = synth.make_scene(12, 4096, seed=21)
    bank = sfm_b200.DescriptorBank(12, 4096)
    bank.put(0, sc.desc, xy=sc.xy)
    res = sfm_b200.match_and_verify(bank, synth.exhaustive_pairs(12), tracks=True, max_iters=512, seed=9, solver="8pt")
    Rt = np.einsum("ij,njk->nik", np.linalg.inv(synth.K_INTR), sc.P)
    return sc, bank, res, Rt


def rotation_error_deg(Ra, Rb):
    c = (np.trace(Ra @ Rb.T) - 1.0) / 2.0
    return float(np.degrees(np.arccos(np.clip(c, -1.0, 1.0))))


def test_gather_equals_numpy_oracle(scene):
    sc, bank, res, Rt = scene
    reg = np.ones(12, np.uint8)
    reg[4] = 0
    pts = gv.triangulate_tracks(res.tracks, bank, synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3], registered=reg, min_inliers=3)
    n_tracks = res.tracks.n_tracks
    assert res.tracks.offsets_buf.numel() - 1 > n_tracks + 1000          # capacity past the live track count
    images = np.array([3, 0, 11, 4, -2, 12, 7], np.int32)
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])).cuda()
    out = pnp.register_images_device(res.tracks, pts, bank.xy, cams, images, seed=2)
    ref = po.gather(res.tracks.track_of.cpu().numpy(), n_tracks, pts.status.cpu().numpy(), pts.X.cpu().numpy(), sc.xy, images)
    h = out.to_host()
    assert h["count"].tolist() == ref["count"].tolist()
    assert ref["count"][[0, 1, 2, 3]].min() > 1000 and ref["count"][4] == 0 and ref["count"][5] == 0
    for q, n in enumerate(ref["count"]):
        assert np.array_equal(h["feature"][q, :n], ref["feature"][q, :n])
    o = po.pnp_ransac(ref["xy"], ref["X"], ref["count"], cams.cpu().numpy(), images, seed=2)
    assert_same(out, o)
    assert h["status"].tolist() == [0, 0, 0, 0, 4, 4, 0]


def test_ground_truth_on_a_synthetic_scene(scene):
    """Each image registered against the points triangulated from the other eleven.  Measured on one B200: see DESIGN §4
    "Absolute pose registration".  Asserted: every image registered, median rotation error < 0.5 degree, median camera-centre
    error < 1 % of the median depth."""
    sc, bank, res, Rt = scene
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])).cuda()
    rot, cen, inl = [], [], []
    depth = None
    for i in range(12):
        reg = np.ones(12, np.uint8)
        reg[i] = 0
        pts = gv.triangulate_tracks(res.tracks, bank, synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3], registered=reg)
        h = pnp.register_images_device(res.tracks, pts, bank.xy, cams, [i], seed=1).to_host()
        assert h["status"].tolist() == [0], (i, h["status"])
        R, t = h["R"][0], h["t"][0]
        rot.append(rotation_error_deg(R, Rt[i, :, :3]))
        C, Ct = -R.T @ t, -Rt[i, :, :3].T @ Rt[i, :, 3]
        cen.append(float(np.linalg.norm(C - Ct)))
        inl.append(h["n_inliers"][0] / h["count"][0])
        if depth is None:
            depth = float(np.median(sc.X @ Rt[0, 2, :3] + Rt[0, 2, 3]))
    print(f"\n12 images: median rotation error {np.median(rot):.5f} deg (max {max(rot):.5f}), median centre error {np.median(cen):.6f} "
          f"= {100 * np.median(cen) / depth:.4f} % of the median depth {depth:.2f} (max {100 * max(cen) / depth:.4f} %), "
          f"median inlier fraction {np.median(inl):.4f}")
    assert np.median(rot) < 0.5
    assert np.median(cen) < 0.01 * depth


def umeyama(src, dst):
    """s, Q, c with dst ~ s Q src + c (least squares)."""
    ms, md = src.mean(0), dst.mean(0)
    a, b = src - ms, dst - md
    U, D, Vt = np.linalg.svd(b.T @ a / len(src))
    S = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        S[2, 2] = -1
    Q = U @ S @ Vt
    s = np.trace(np.diag(D) @ S) / a.var(0).sum()
    return s, Q, md - s * Q @ ms


def test_incremental_loop_on_the_device(scene):
    """Two-view initialisation on images (0, 1) (camera 0 = [I|0], |t| = 1), triangulation from those two, registration of the
    other ten in one batch (writing into cams and registered on the device), triangulation from all twelve, registration of all
    twelve again.  After a similarity alignment of the camera centres every image is registered within loose bounds."""
    sc, bank, res, Rt = scene
    two = sfm_b200.match_and_verify(bank, [[0, 1]], fetch=True, max_iters=512, seed=5, solver="8pt").to_host()
    m = two["matches"][two["inlier"].astype(bool)]
    g = gv.two_view_geometry(sc.xy[0][m[:, 0]], sc.xy[1][m[:, 1]], synth.K_INTR, synth.K_INTR, seed=3)
    assert g["n_pose"] > 100
    R = np.tile(np.eye(3), (12, 1, 1))
    t = np.zeros((12, 3))
    R[1], t[1] = g["R"], g["t"]
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, R, t)).cuda()
    reg = torch.zeros(12, dtype=torch.uint8, device="cuda")
    reg[:2] = 1
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, reg, S=bank.max_feats)
    first = pnp.register_images_device(res.tracks, pts, bank.xy, cams, np.arange(2, 12), update=True, registered=reg, seed=4)
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, reg, S=bank.max_feats)
    second = pnp.register_images_device(res.tracks, pts, bank.xy, cams, np.arange(12), update=True, registered=reg, seed=4)
    h1, h2 = first.to_host(), second.to_host()
    assert h1["registered"] == 10 and h2["registered"] == 12 and reg.cpu().numpy().tolist() == [1] * 12
    assert np.array_equal(cams[:, 4:].cpu().numpy(), h2["pose"])
    Rs, ts = h2["R"], h2["t"]
    C_est = np.stack([-Rs[i].T @ ts[i] for i in range(12)])
    C_true = np.stack([-Rt[i, :, :3].T @ Rt[i, :, 3] for i in range(12)])
    s, Q, c = umeyama(C_est, C_true)
    cen = np.linalg.norm((s * (Q @ C_est.T)).T + c - C_true, axis=1)
    rot = [rotation_error_deg(Rs[i] @ Q.T, Rt[i, :, :3]) for i in range(12)]
    depth = float(np.median(sc.X @ Rt[0, 2, :3] + Rt[0, 2, 3]))
    print(f"\nincremental: rotation error median {np.median(rot):.4f} max {max(rot):.4f} deg; centre error median "
          f"{100 * np.median(cen) / depth:.4f} % max {100 * max(cen) / depth:.4f} % of the median depth; scale {s:.4f}")
    assert max(rot) < 2.0
    assert max(cen) < 0.05 * depth


def test_pipeline_path_launches(scene):
    sc, bank, res, Rt = scene
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])).cuda()
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, S=bank.max_feats)
    torch.cuda.synchronize()
    n0 = sfm_b200.launch_count()
    out = sfm_b200.register_images_device(res.tracks, pts, bank.xy, cams, np.arange(12), seed=6)
    assert sfm_b200.launch_count() - n0 == pnp.PNP_LAUNCHES
    assert out.counts["registered"] == 12
    ref_g = po.gather(res.tracks.track_of.cpu().numpy(), res.tracks.n_tracks, pts.status.cpu().numpy(), pts.X.cpu().numpy(), sc.xy,
                      np.arange(12))
    assert_same(out, po.pnp_ransac(ref_g["xy"], ref_g["X"], ref_g["count"], cams.cpu().numpy(), np.arange(12), seed=6))
    h = gv.register_images(res.tracks.to_host(), pts, sc.xy, synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3], np.arange(12), seed=6).to_host()
    assert np.array_equal(h["pose"], out.to_host()["pose"])


def test_estimate_absolute_pose_public_call():
    rng = np.random.default_rng(5)
    R, t = random_rotation(rng), rng.normal(size=3)
    Xc = np.stack([rng.uniform(-2, 2, 300), rng.uniform(-1.2, 1.2, 300), rng.uniform(4, 8, 300)], 1)
    px = Xc[:, :2] / Xc[:, 2:] * 1000 + [960, 540] + rng.normal(0, 0.5, (300, 2))
    px[:60] += 150.0
    Xw = (Xc - t) @ R
    n, Re, te, mask = gv.estimate_absolute_pose(px, Xw, synth.K_INTR)
    assert n == 240 and mask.shape == (300, 1) and mask[:60].sum() == 0 and mask[60:].all()
    assert rotation_error_deg(Re, R) < 0.1 and np.linalg.norm(te - t) < 0.05
    res = gv.estimate_absolute_poses([px, px[:2], px[:40] + 500.0], [Xw, Xw[:2], Xw[:40]], synth.K_INTR)
    assert [r[0] for r in res][1:] == [0, 0] and res[0][0] == 240 and not res[2][1].any()
    with pytest.raises(ValueError):
        gv.estimate_absolute_pose(px, Xw, synth.K_INTR + np.array([[0, 0.5, 0], [0, 0, 0], [0, 0, 0]]))


def test_empty_and_degenerate_inputs(scene):
    sc, bank, res, Rt = scene
    cams = torch.from_numpy(tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])).cuda()
    pts = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, S=bank.max_feats)
    e = pnp.register_images_device(res.tracks, pts, bank.xy, cams, np.zeros(0, np.int32)).to_host()
    assert e["pose"].shape == (0, 12) and all(e[n] == 0 for n in pnp.STATUS_NAMES)
    none = pnp.pnp_ransac_device(torch.zeros((0, 8, 2), dtype=torch.float32, device="cuda"), torch.zeros((0, 8, 3), dtype=torch.float64, device="cuda"),
                                 torch.zeros(0, dtype=torch.int32, device="cuda"), cams, []).to_host()
    assert none["status"].shape == (0,) and all(none[n] == 0 for n in pnp.STATUS_NAMES)
    # no tracks at all
    z = np.zeros(0, np.int32)
    empty = sfm_b200.build_tracks_device(z, z, z, np.zeros((0, 3), np.int32), None, None, 12, 4096)
    ept = tri.triangulate_tracks_device(empty, bank.xy, cams, S=bank.max_feats)
    h = pnp.register_images_device(empty, ept, bank.xy, cams, np.arange(12)).to_host()
    assert h["count"].tolist() == [0] * 12 and h["too_few_points"] == 12 and not h["pose"].any()
    # tracks, but no triangulated point (no image registered)
    npt = tri.triangulate_tracks_device(res.tracks, bank.xy, cams, np.zeros(12, np.uint8), S=bank.max_feats)
    h = pnp.register_images_device(res.tracks, npt, bank.xy, cams, np.arange(12)).to_host()
    assert h["count"].tolist() == [0] * 12 and h["too_few_points"] == 12
