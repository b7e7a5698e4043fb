"""bench.py --dump-outputs: what the timed path returned, written as float32 / float64 .npy files within the size limit,
with a fixed sample of the rows of an array too large for its share, and a sharded result read in pair order.  CPU only."""
import os
import sys

import numpy as np
import pytest
import torch

import bench


def _sizes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_small_outputs_are_written_whole(tmp_path):
    arrays = {"n_matches": torch.tensor([3, 0, 7], dtype=torch.int32), "F": np.arange(18, dtype=np.float64).reshape(2, 3, 3),
              "xy": np.ones((4, 2), np.float32), "inlier": np.array([1, 0, 1], np.uint8)}
    bench.dump_outputs(str(tmp_path), arrays)
    assert sorted(os.listdir(tmp_path)) == ["F.npy", "inlier.npy", "n_matches.npy", "xy.npy"]
    n = np.load(tmp_path / "n_matches.npy")
    assert n.dtype == np.float64 and n.tolist() == [3, 0, 7]
    assert np.load(tmp_path / "xy.npy").dtype == np.float32
    assert np.array_equal(np.load(tmp_path / "F.npy"), arrays["F"])
    assert np.load(tmp_path / "inlier.npy").tolist() == [1, 0, 1]


def test_large_outputs_keep_a_fixed_sample_within_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    rng = np.random.default_rng(1)
    matches = rng.integers(0, 1 << 20, (50_000, 3)).astype(np.int32)
    for d, m in (("a", matches), ("b", torch.from_numpy(matches))):
        bench.dump_outputs(str(tmp_path / d), {"matches": m, "n_inliers": np.arange(10, dtype=np.int32)})
        assert _sizes(tmp_path / d) <= bench.DUMP_BYTES
    for f in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))      # the same sample every run
    rows = np.load(tmp_path / "a" / "matches.rows.npy")
    m = np.load(tmp_path / "a" / "matches.npy")
    assert m.dtype == np.float64 and 0 < len(rows) == len(m) < 50_000 and (np.diff(rows) > 0).all()
    assert np.array_equal(m, matches[rows.astype(np.int64)])
    assert not os.path.exists(tmp_path / "a" / "n_inliers.rows.npy")


def test_sharded_result_rows_are_read_in_pair_order():
    """Rank slices keep unwritten room after their rows (here -1): only rows row_start[p] : row_start[p] + n_matches[p] count."""
    full = torch.full((12, 3), -1, dtype=torch.int32)
    full[0:2] = torch.tensor([[0, 0, 0], [0, 1, 1]])                   # pair 0, rank 0
    full[6:9] = torch.tensor([[2, 0, 5], [2, 1, 6], [2, 2, 7]])        # pair 2, rank 1
    inl = torch.tensor([1, 0, 9, 9, 9, 9, 1, 1, 0, 9, 9, 9], dtype=torch.uint8)
    g = {"n_matches": torch.tensor([2, 0, 3], dtype=torch.int32), "F": torch.zeros((3, 3, 3), dtype=torch.float64),
         "row_start": torch.tensor([0, 2, 6]), "matches": full, "inlier": inl, "transport": "sendrecv"}
    out = bench.sharded_outputs(g, ("matches", "inlier", "in_front"))
    assert sorted(out) == ["F", "inlier", "matches", "n_matches"]
    assert out["matches"][:, 0].tolist() == [0, 0, 2, 2, 2] and out["inlier"].tolist() == [1, 0, 1, 1, 0]
    summaries = {k: v for k, v in g.items() if k in ("n_matches", "F")}
    assert sorted(bench.sharded_outputs(summaries, ("matches", "inlier"))) == ["F", "n_matches"]


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bad_arguments_are_refused(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.main()
