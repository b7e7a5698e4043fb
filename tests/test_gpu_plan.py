"""One-GPU tests of the execution plan (sfm_b200/plan.py): rows pushed to a device sink through the three-set rotation,
the one-stream form of the pipeline, the empty pair list with every stage, the D2H byte count with every stage, and the
argument checks of sfm_refine_filter_packed."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # collected on CPU boxes, skipped there
    pytest.skip("needs a GPU", allow_module_level=True)

import sfm_b200  # noqa: E402
from sfm_b200 import _lib, matcher, synth  # noqa: E402
from sfm_b200 import dist as sdist  # noqa: E402

ERR_ARG, ERR_STATE = -1, -4
PRM = dict(max_iters=256, seed=9, solver="8pt")
STAGES = dict(homography=True, intrinsics=synth.K_INTR)
ROW_KEYS = {"offsets", "matches", "inlier", "inlier_h", "in_front", "points3d"}
PAIR_KEYS = ("n_matches", "F", "n_inliers", "iters", "H", "n_inliers_h", "R", "t", "n_pose")


@pytest.fixture(scope="module")
def scene():
    sc = synth.make_scene(5, 2048, seed=8)
    bank = sfm_b200.DescriptorBank(5, 2048)
    bank.put(0, sc.desc, xy=sc.xy)
    return bank, synth.exhaustive_pairs(5)


def test_row_sink_on_one_gpu_equals_fetched_rows(scene):
    """Without a process group the sharded call pushes every row array into local arrays (five batches of two pairs: the
    three-set rotation of the sink path); summaries and rows equal what the pinned-host path returns."""
    bank, pairs = scene
    ref = sfm_b200.match_and_verify(bank, pairs, fetch=True, **STAGES, **PRM).to_host()
    out, res = sdist.match_and_verify_sharded(bank, pairs, pair_batch=2, **STAGES, **PRM)
    assert len(res.plan.sets) == 3
    for k in PAIR_KEYS:
        assert np.array_equal(out[k].cpu().numpy(), ref[k]), k
    start = out["row_start"].cpu().numpy()
    for name in ROW_KEYS - {"offsets"}:
        got = out[name].cpu().numpy()
        for p in range(len(pairs)):
            a, b = ref["offsets"][p], ref["offsets"][p + 1]
            assert np.array_equal(got[start[p]: start[p] + (b - a)], ref[name][a:b]), (name, p)
    assert len(ref["matches"]) > 0 and ref["inlier_h"].any() and ref["in_front"].any()


def test_one_stream_equals_two_streams(scene):
    """overlap=False (sweep and refinement on the caller's stream, one scratch set) returns what the two-stream pipeline returns."""
    bank, pairs = scene
    kw = dict(fetch=True, mutual=True, pair_batch=3, **STAGES, **PRM)
    two = sfm_b200.match_and_verify(bank, pairs, overlap=True, **kw)
    one = sfm_b200.match_and_verify(bank, pairs, overlap=False, **kw)
    assert two.plan.post_stream is not None and one.plan.post_stream is None
    a, b = two.to_host(), one.to_host()
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert one.d2h_bytes == two.d2h_bytes and len(a["matches"]) > 0


def test_empty_pair_list_with_every_stage(scene):
    """P == 0 returns the same keys, dtypes and trailing shapes as P > 0; without matches exactly the row keys are dropped."""
    bank, pairs = scene
    full = sfm_b200.match_and_verify(bank, pairs[:2], fetch=True, **STAGES, **PRM)
    empty = sfm_b200.match_and_verify(bank, np.zeros((0, 2), np.int32), fetch=True, **STAGES, **PRM)
    a, e = full.to_host(), empty.to_host()
    assert a.keys() == e.keys() and ROW_KEYS <= a.keys()
    for k in a:
        assert e[k].dtype == a[k].dtype and e[k].shape[1:] == a[k].shape[1:], k
        assert len(e[k]) == (1 if k == "offsets" else 0), k
    for k in PAIR_KEYS:
        assert getattr(empty, k).dtype == getattr(full, k).dtype and getattr(empty, k).shape == (0,) + getattr(full, k).shape[1:], k
    assert empty.to_host(with_matches=False).keys() == a.keys() - ROW_KEYS
    assert full.to_host(with_matches=False).keys() == a.keys() - ROW_KEYS


def test_d2h_byte_count_with_every_stage(scene):
    """One batch with both optional stages: offsets, 27 bytes per row (13 core + 1 homography + 13 pose) and 256 per pair
    (80 + 76 + 100); n_matches is never copied."""
    bank, pairs = scene
    r = sfm_b200.match_and_verify(bank, pairs, fetch=True, **STAGES, **PRM)
    P, rows = len(pairs), len(r.to_host()["matches"])
    assert r.d2h_bytes == 4 * (P + 1) + 27 * rows + 256 * P


def test_refine_filter_packed_checks_its_arguments(scene):
    """sfm_refine_filter_packed rejects an exact_int ratio outside 0 < num, den < 4096 and a bank with no images, like
    sfm_match_pairs_packed, before it launches anything."""
    bank, pairs = scene
    L, dev, cap = _lib.lib(), bank.device, bank.feat_stride
    st = _lib.current_stream_ptr(dev)
    pairs_t = torch.from_numpy(pairs[:1]).to(dev)
    scratch = sfm_b200.knn2(bank, pairs_t, sweep_only=4)                 # the candidate records of a sweep
    blk = torch.empty(cap // 256, dtype=torch.int32, device=dev)
    counts, offsets = torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(2, dtype=torch.int32, device=dev)
    matches = torch.empty((cap, 3), dtype=torch.int32, device=dev)
    corr = torch.empty((cap, 4), dtype=torch.float32, device=dev)
    prm = matcher.filter_params(0.75, "exact_int", False)

    def call(b, n_pairs):
        return L.sfm_refine_filter_packed(b.handle, _lib.ptr(pairs_t), n_pairs, C.byref(prm), None, _lib.ptr(scratch), _lib.ptr(blk),
                                          _lib.ptr(counts), _lib.ptr(offsets), _lib.ptr(matches), _lib.ptr(corr), st)

    assert call(bank, 1) == 0
    torch.cuda.synchronize()
    assert int(counts[0]) > 0
    prm.ratio_num = 5000
    assert call(bank, 1) == ERR_ARG
    assert "4096" in L.sfm_last_error().decode()
    prm.ratio_num = 3
    assert call(sfm_b200.DescriptorBank(2, 2048), 0) == ERR_STATE
    assert "empty" in L.sfm_last_error().decode()
