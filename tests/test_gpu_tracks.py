"""Feature tracks on the GPU (csrc/tracks.cu) against the numpy oracle (oracle/track_oracle.py), array for array: random
graphs (small S, long chains, one component of 131,073 nodes, every flag source, the pair filter, empty inputs), order
independence, the end-to-end paths of the pipeline (host result, in-plan hooks, the sharded row sink, the reference's
pair_matches list), launch counts and the two-GPU gather."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # collected on CPU boxes, skipped there
    pytest.skip("needs a GPU", allow_module_level=True)

import geometric_verification as gv  # noqa: E402
import sfm_b200  # noqa: E402
from oracle import track_oracle as to  # noqa: E402
from sfm_b200 import dist as sdist  # noqa: E402
from sfm_b200 import synth  # noqa: E402
from sfm_b200 import tracks as tr  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRM = dict(max_iters=512, seed=9, solver="8pt")


def assert_same(got, ref):
    h = got.to_host() if isinstance(got, tr.Tracks) else got
    for k in ("offsets", "obs", "track_of"):
        assert h[k].dtype == ref[k].dtype and h[k].shape == ref[k].shape, (k, h[k].shape, ref[k].shape)
        assert np.array_equal(h[k], ref[k]), k
    for k in tr.COUNT_NAMES:
        assert h[k] == ref[k], (k, h[k], ref[k])


def random_rows(rng, n_images, S, P, max_rows):
    pairs = rng.integers(0, n_images, (P, 2)).astype(np.int32)
    n_rows = rng.integers(0, max_rows + 1, P).astype(np.int32)
    start = np.concatenate([[0], np.cumsum(n_rows)[:-1]]).astype(np.int64)
    rows = rng.integers(0, S, (int(n_rows.sum()), 3)).astype(np.int32)
    flags = {f: (rng.random(len(rows)) < 0.6).astype(np.uint8) for f in ("inlier", "inlier_h", "in_front")}
    n_inl = rng.integers(0, 40, P).astype(np.int32)
    return pairs, start, n_rows, rows, flags, n_inl


@pytest.mark.parametrize("flag", [None, "inlier", "inlier_h", "in_front"])
@pytest.mark.parametrize("min_length,keep", [(2, False), (3, False), (2, True), (3, True)])
def test_random_graphs_equal_oracle(flag, min_length, keep):
    rng = np.random.default_rng([tr.FLAG_FIELDS.index(flag), min_length, int(keep)])
    for n_images, S, P, max_rows in ((4, 7, 40, 9), (9, 64, 300, 40), (30, 1000, 2000, 300)):
        pairs, start, n_rows, rows, flags, n_inl = random_rows(rng, n_images, S, P, max_rows)
        row_flag = None if flag is None else flags[flag]
        for mpi in (0, 15):
            kw = dict(min_pair_inliers=mpi, min_length=min_length, keep_conflicts=keep)
            got = sfm_b200.build_tracks_device(pairs, start, n_rows, rows, row_flag, n_inl, n_images, S, **kw)
            assert_same(got, to.build_tracks(pairs, start, n_rows, rows, row_flag, n_inl, n_images, S, **kw))


def test_long_chain_in_random_order():
    """100,000 images x 1 feature linked into one chain in random order: deep unions, one non-conflicting track of 10^5
    observations (CTA sort with merge passes), and the same chain split by one missing link."""
    rng = np.random.default_rng(5)
    n = 100_000
    perm = rng.permutation(n).astype(np.int32)
    pairs = np.stack([perm[:-1], perm[1:]], axis=1)
    order = rng.permutation(n - 1)
    pairs = pairs[order]
    rows = np.zeros((n - 1, 3), np.int32)
    start, n_rows = np.arange(n - 1, dtype=np.int64), np.ones(n - 1, np.int32)
    got = sfm_b200.build_tracks_device(pairs, start, n_rows, rows, None, None, n, 1)
    ref = to.build_tracks(pairs, start, n_rows, rows, None, None, n, 1)
    assert ref["n_tracks"] == 1 and ref["n_obs"] == n
    assert_same(got, ref)
    flag = np.ones(n - 1, np.uint8)
    flag[np.nonzero(order == n // 3)[0]] = 0
    assert_same(sfm_b200.build_tracks_device(pairs, start, n_rows, rows, flag, None, n, 1),
                to.build_tracks(pairs, start, n_rows, rows, flag, None, n, 1))


def test_chain_built_without_any_find_walking_it():
    """Edges (k, k+1) in descending k: every find meets a root at once, so link-by-index leaves one chain of 200,000 nodes
    that only finalize's compression walks.  Images x 1 feature, one pair per edge, one row each."""
    n = 200_000
    k = np.arange(n - 2, -1, -1, dtype=np.int32)
    pairs = np.stack([k, k + 1], axis=1)
    rows = np.zeros((n - 1, 3), np.int32)
    start, n_rows = np.arange(n - 1, dtype=np.int64), np.ones(n - 1, np.int32)
    for order in (slice(None), slice(None, None, -1)):
        got = sfm_b200.build_tracks_device(pairs[order], start, n_rows, rows, None, None, n, 1)
        ref = to.build_tracks(pairs[order], start, n_rows, rows, None, None, n, 1)
        assert ref["n_tracks"] == 1 and ref["n_obs"] == n
        assert_same(got, ref)


@pytest.mark.parametrize("keep", [False, True])
def test_one_component_of_131073_nodes(keep):
    """Feature 0 of image 0 matched to every feature of image 1 (S = 131072), rows shuffled: one conflicting candidate of
    131,073 nodes -- dropped, or kept and sorted through the long-slice path -- plus a small clean track beside it."""
    rng = np.random.default_rng(6)
    S = 131072
    t = rng.permutation(S).astype(np.int32)
    rows = np.stack([np.zeros(S, np.int32), t, np.zeros(S, np.int32)], axis=1)
    pairs = np.array([[0, 1], [2, 0]], np.int32)
    rows = np.concatenate([rows, [[9, 5, 0]]]).astype(np.int32)          # pair (2, 0): the clean track {0:5, 2:9}
    start, n_rows = np.array([0, S], np.int64), np.array([S, 1], np.int32)
    got = sfm_b200.build_tracks_device(pairs, start, n_rows, rows, None, None, 3, S, keep_conflicts=keep)
    ref = to.build_tracks(pairs, start, n_rows, rows, None, None, 3, S, keep_conflicts=keep)
    assert ref["n_conflicting"] == 1 and ref["n_tracks"] == (2 if keep else 1)
    assert_same(got, ref)


def test_empty_inputs():
    """P == 0, and pairs whose rows all fail the flag or the pair filter: no track, every count zero, track_of all -1."""
    z = np.zeros(0, np.int32)
    for got in (sfm_b200.build_tracks_device(z, z, z, np.zeros((0, 3), np.int32), None, None, 3, 50),
                sfm_b200.build_tracks_device([[0, 1]], [0], [3], np.ones((3, 3), np.int32), np.zeros(3, np.uint8), None, 3, 50),
                sfm_b200.build_tracks_device([[0, 1]], [0], [3], np.ones((3, 3), np.int32), None, [14], 3, 50)):
        h = got.to_host()
        assert h["offsets"].tolist() == [0] and h["obs"].shape == (0, 2) and (h["track_of"] == -1).all()
        assert all(h[k] == 0 for k in tr.COUNT_NAMES)


def test_invalid_rows_are_counted_and_raise():
    rows = np.array([[1, 2, 0], [3, 50, 0]], np.int32)
    got = sfm_b200.build_tracks_device([[0, 1]], [0], [2], rows, None, None, 2, 50)
    assert int(got.counts_dev[4]) == 1
    with pytest.raises(sfm_b200.SfmError, match="outside"):
        got.to_host()
    with pytest.raises(sfm_b200.SfmError, match="outside"):
        got.track_of


def test_order_independence():
    """The output depends only on the set of used edges: rows shuffled within and across pairs, pairs permuted and split,
    every row duplicated, every pair also given reversed with swapped (q, t) -- identical arrays."""
    rng = np.random.default_rng(8)
    n_images, S = 12, 300
    pairs, start, n_rows, rows, flags, n_inl = random_rows(rng, n_images, S, 400, 60)
    base = sfm_b200.build_tracks_device(pairs, start, n_rows, rows, flags["inlier"], n_inl, n_images, S).to_host()
    u, v, _ = to.used_edges(pairs, start, n_rows, rows, flags["inlier"], n_inl, n_images, S)
    rec = np.stack([u // S, v // S, u % S, v % S], axis=1)
    rec = np.concatenate([rec, rec, rec[:, [1, 0, 3, 2]]])               # duplicates and both directions
    rec = rec[rng.permutation(len(rec))]
    key = rec[:, 0] * n_images + rec[:, 1]
    groups = [np.nonzero(key == k)[0] for k in rng.permutation(np.unique(key))]
    pl, rl, cnt = [], [], []
    for g in groups:
        for part in np.array_split(g, min(len(g), rng.integers(1, 3))):                # some pairs appear twice
            pl.append(rec[part[0], :2])
            rl.append(np.stack([rec[part, 2], rec[part, 3], np.zeros(len(part), np.int64)], axis=1))
            cnt.append(len(part))
    cnt = np.asarray(cnt)
    got = sfm_b200.build_tracks_device(np.asarray(pl), np.concatenate([[0], np.cumsum(cnt)[:-1]]), cnt, np.concatenate(rl),
                                       None, None, n_images, S)
    assert base["n_tracks"] > 10
    assert_same(got, base)


# ------------------------------------------------------------------ end to end on a synthetic scene
N_IMG, N_FEAT = 12, 4096


@pytest.fixture(scope="module")
def scene():
    sc = synth.make_scene(N_IMG, N_FEAT, seed=21)
    bank = sfm_b200.DescriptorBank(N_IMG, N_FEAT)
    bank.put(0, sc.desc, xy=sc.xy)
    return sc, bank, synth.exhaustive_pairs(N_IMG)


@pytest.fixture(scope="module")
def host_result(scene):
    sc, bank, pairs = scene
    return sfm_b200.match_and_verify(bank, pairs, fetch=True, homography=True, **PRM).to_host()


def test_scene_tracks_equal_oracle_and_ground_truth(scene, host_result):
    sc, bank, pairs = scene
    for flags in ("inlier", "inlier_h", None):
        got = gv.build_tracks(host_result, N_IMG, N_FEAT, flags=flags)
        assert_same(got, to.build_tracks_host(host_result, N_IMG, N_FEAT, flags=flags))
    t = gv.build_tracks(host_result, N_IMG, N_FEAT).to_host()
    assert t["n_tracks"] > 1000
    pt = sc.point[t["obs"][:, 0], t["obs"][:, 1]]
    seg = np.repeat(np.arange(t["n_tracks"]), np.diff(t["offsets"]))
    first = pt[t["offsets"][:-1]]
    pure = np.ones(t["n_tracks"], bool)
    np.logical_and.at(pure, seg, (pt == first[seg]) & (pt >= 0))
    frac = pure.mean()
    print(f"\n{t['n_tracks']} tracks, {t['n_obs']} observations, {t['n_conflicting']} conflicting, {t['n_short']} short; "
          f"{frac:.4f} of the tracks observe one scene point; mean length {t['n_obs'] / t['n_tracks']:.2f}")
    assert frac > 0.5
    # every observation of a kept track is in a distinct image
    assert (np.diff(t["obs"][:, 0])[np.diff(seg) == 0] > 0).all()


@pytest.mark.parametrize("overlap", [True, False])
@pytest.mark.parametrize("pair_batch", [2048, 7])
def test_in_plan_tracks_equal_standalone(scene, host_result, overlap, pair_batch):
    """tracks=True hooks every batch inside the plan (several batches rotate the output sets); fetch=False keeps no rows."""
    sc, bank, pairs = scene
    res = sfm_b200.match_and_verify(bank, pairs, homography=True, tracks=True, overlap=overlap, pair_batch=pair_batch, **PRM)
    assert res.host is None
    assert_same(res.tracks, to.build_tracks_host(host_result, N_IMG, N_FEAT))
    res_h = sfm_b200.match_and_verify(bank, pairs, homography=True, tracks=True, track_flags="inlier_h", min_length=3,
                                      overlap=overlap, pair_batch=pair_batch, **PRM)
    assert_same(res_h.tracks, to.build_tracks_host(host_result, N_IMG, N_FEAT, flags="inlier_h", min_length=3))


def test_sharded_row_sink_tracks_equal_standalone(scene, host_result):
    """World size 1: the sharded call gathers the rows into device arrays and builds the tracks from them (path b)."""
    sc, bank, pairs = scene
    out, _ = sdist.match_and_verify_sharded(bank, pairs, pair_batch=5, homography=True, tracks=True, **PRM)
    ref = to.build_tracks_host(host_result, N_IMG, N_FEAT)
    assert_same(out["tracks"], ref)
    assert_same(gv.build_tracks(out, N_IMG, N_FEAT), ref)
    with pytest.raises(ValueError):
        sdist.match_and_verify_sharded(bank, pairs, gather="summaries", tracks=True, **PRM)


def test_launch_counts(scene):
    """tracks=True adds one init, one hook per batch and the finalize launches of the library (each hook is preceded by a
    torch copy that widens the batch's int32 offsets, not counted here); the same job without it is unchanged."""
    sc, bank, pairs = scene
    kw = dict(pair_batch=8, overlap=False, **PRM)

    def count(**extra):
        n0 = sfm_b200.launch_count()
        sfm_b200.match_and_verify(bank, pairs, **kw, **extra)
        torch.cuda.synchronize()
        return sfm_b200.launch_count() - n0

    before = count()
    with_tracks = count(tracks=True)
    after = count()
    assert before == after
    n_batches = -(-len(pairs) // 8)
    assert with_tracks - before == 1 + n_batches + tr.FINALIZE_LAUNCHES


def test_empty_job_with_tracks(scene):
    sc, bank, pairs = scene
    res = sfm_b200.match_and_verify(bank, np.zeros((0, 2), np.int32), tracks=True, **PRM)
    assert res.tracks.n_tracks == 0 and res.tracks.track_of.shape == (N_IMG, N_FEAT)


def test_reference_pair_matches_equal_oracle(golden_dir):
    """The drop-in extract_and_match over the golden ORB images through the reference loop (code/pipeline.py:36-47) gives
    pair_matches; build_tracks of that list equals the oracle on the same rows."""
    import feature_matching as fm

    images = np.load(os.path.join(golden_dir, "ref_orb_hamming.npz"))["images"]
    pair_matches = []
    for i in range(images.shape[0]):
        for j in range(images.shape[0]):
            if i != j:
                match = fm.extract_and_match(images[i], images[j])
                if match:
                    pair = sfm_b200.Pair()
                    pair.img_inx_1, pair.img_inx_2, pair.matches = i, j, match
                    pair_matches.append(pair)
    assert len(pair_matches) == 6
    S = 1 + max(max(m.queryIdx, m.trainIdx) for p in pair_matches for m in p.matches)
    pairs = np.array([(p.img_inx_1, p.img_inx_2) for p in pair_matches], np.int32)
    cnt = np.array([len(p.matches) for p in pair_matches])
    rows = np.array([(m.queryIdx, m.trainIdx, 0) for p in pair_matches for m in p.matches], np.int32)
    ref = to.build_tracks(pairs, np.concatenate([[0], np.cumsum(cnt)[:-1]]), cnt, rows, None, None, images.shape[0], S)
    assert ref["n_tracks"] > 0
    assert_same(gv.build_tracks(pair_matches, images.shape[0], S), ref)


# ------------------------------------------------------------------ two GPUs
def _worker(rank, ws, port, q):
    import faulthandler

    faulthandler.dump_traceback_later(150, exit=True)
    try:
        _worker_body(rank, ws, port, q)
    except Exception:
        import traceback

        q.put({"error": f"rank {rank}: {traceback.format_exc()}"})
        raise
    finally:
        faulthandler.cancel_dump_traceback_later()


def _worker_body(rank, ws, port, q):
    for p in (ROOT, os.path.join(ROOT, "sfm-project_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    import sfm_b200
    from sfm_b200 import dist as sdist
    from sfm_b200 import synth

    n_img, n_feat = 7, 2048
    sc = synth.make_scene(n_img, n_feat, seed=77)
    pairs = synth.exhaustive_pairs(n_img)
    bank = sfm_b200.DescriptorBank(n_img, n_feat, device=dev)
    if rank == 0:
        bank.put(0, sc.desc, xy=sc.xy)
    sdist.broadcast_bank(bank, src=0)
    prm = dict(max_iters=512, solver="8pt", seed=9)
    report = {}
    for mode in ("block", "cyclic"):
        out, _ = sdist.match_and_verify_sharded(bank, pairs, mode=mode, pair_batch=4, tracks=True, **prm)
        torch.cuda.synchronize()
        if rank == 0:
            one = sfm_b200.match_and_verify(bank, pairs, pair_batch=4, tracks=True, **prm).tracks.to_host()
            got = out["tracks"].to_host()
            report[mode] = one["n_tracks"] > 0 and all(np.array_equal(np.asarray(got[k]), np.asarray(one[k])) for k in one)
    if rank == 0:
        q.put(report)
    dist.barrier()
    for reg in bank.__dict__.get("_gather_regions", {}).values():
        reg.close()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_two_gpu_tracks_equal_one_gpu_tracks():
    import queue as _queue
    import time

    import torch.multiprocessing as mp

    ws = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, ws, port, q)) for r in range(ws)]
    for p in procs:
        p.start()
    report, t0 = None, time.time()
    while report is None and time.time() - t0 < 420:
        try:
            report = q.get(timeout=2)
        except _queue.Empty:
            if any(p.exitcode not in (None, 0) for p in procs):
                break
    if report is None or "error" in report:
        for p in procs:
            if p.is_alive():
                p.kill()
        raise AssertionError(f"multi-GPU workers failed: {report}")
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert report and all(report.values()), report
