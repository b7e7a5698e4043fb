"""CPU checks of the feature tracks: the numpy oracle against scipy's connected components and on hand-made graphs, the
C-ABI argument checks of the four sfm_tracks_* entry points (all before any CUDA call) and the parameter struct's size."""
import ctypes as C

import numpy as np
import pytest

from oracle import track_oracle as to


def _scipy_partition(u, v, nodes):
    sp = pytest.importorskip("scipy.sparse")
    cg = pytest.importorskip("scipy.sparse.csgraph")
    n = int(max(u.max(), v.max())) + 1
    g = sp.csr_matrix((np.ones(len(u)), (u, v)), shape=(n, n))
    _, lab = cg.connected_components(g, directed=False)
    return lab[nodes]


@pytest.mark.parametrize("seed", range(8))
def test_oracle_components_equal_scipy(seed):
    """Random graphs with multi-edges and self-loops: the same partition as scipy, each label the component's smallest node."""
    rng = np.random.default_rng(seed)
    n, e = int(rng.integers(2, 3000)), int(rng.integers(1, 4000))
    u, v = rng.integers(0, n, e), rng.integers(0, n, e)
    u = np.concatenate([u, u[:50]])                          # multi-edges
    v = np.concatenate([v, v[:50]])
    u = np.concatenate([u, v[:20]])                          # self-loops
    v = np.concatenate([v, v[:20]])
    nodes, lab = to.components(u, v)
    assert np.array_equal(nodes, np.unique(np.concatenate([u, v])))
    ref = _scipy_partition(u, v, nodes)
    # the same partition: scipy's label determines ours and vice versa
    assert len(np.unique(np.stack([ref, lab]), axis=1)[0]) == len(np.unique(ref)) == len(np.unique(lab))
    for c in np.unique(lab):
        assert nodes[c] == nodes[lab == c].min()


def test_oracle_rows_to_tracks_equal_scipy():
    """Rows of random pairs, including i == j pairs and pairs without rows, through the whole oracle: every kept track is one
    scipy component, and keep_conflicts=True with min_length=2 keeps exactly the components of two or more nodes."""
    rng = np.random.default_rng(3)
    n_images, S, P = 6, 40, 30
    pairs = rng.integers(0, n_images, (P, 2))
    pairs[:4, 1] = pairs[:4, 0]                               # i == j pairs
    n_rows = rng.integers(0, 12, P)
    n_rows[4] = 0
    start = np.concatenate([[0], np.cumsum(n_rows)[:-1]])
    rows = rng.integers(0, S, (int(n_rows.sum()), 3)).astype(np.int32)
    out = to.build_tracks(pairs, start, n_rows, rows, None, None, n_images, S, keep_conflicts=True)
    u, v, bad = to.used_edges(pairs, start, n_rows, rows, None, None, n_images, S)
    assert bad == 0 and len(u) == n_rows.sum()
    nodes = np.unique(np.concatenate([u, v]))
    ref = _scipy_partition(u, v, nodes)
    sizes = np.bincount(ref)
    assert out["n_tracks"] == int((sizes[np.unique(ref)] >= 2).sum())
    assert out["n_short"] == int((sizes[np.unique(ref)] == 1).sum())
    flat = out["obs"][:, 0].astype(np.int64) * S + out["obs"][:, 1]
    for k in range(out["n_tracks"]):
        seg = flat[out["offsets"][k]: out["offsets"][k + 1]]
        assert np.all(np.diff(seg) > 0)
        comp = ref[np.searchsorted(nodes, seg)]
        assert np.all(comp == comp[0]) and len(seg) == sizes[comp[0]]
    empty = to.build_tracks(np.zeros((0, 2)), [], [], np.zeros((0, 3)), None, None, n_images, S)
    assert empty["n_tracks"] == 0 and empty["offsets"].tolist() == [0] and empty["obs"].shape == (0, 2)
    assert (empty["track_of"] == -1).all()


def test_oracle_drop_and_order_rules():
    """Hand-made graph, S = 10: conflicts are dropped first (and kept on request), then short candidates; tracks are numbered
    by smallest node, observations ascend by node."""
    S, n_images = 10, 4
    # a: 31-12-3 (three images), b: 5-25 (one pair), c: 6-7 (same image: conflicting), d: 14-34 plus self-loop 8-8
    edges = [(31, 12), (12, 3), (25, 5), (6, 7), (34, 14), (8, 8)]
    u, v = np.array(edges).T
    out = to.tracks_from_edges(u, v, n_images, S)
    assert out["n_tracks"] == 3 and out["n_conflicting"] == 1 and out["n_short"] == 1
    assert out["offsets"].tolist() == [0, 3, 5, 7]
    flat = (out["obs"][:, 0] * S + out["obs"][:, 1]).tolist()
    assert flat == [3, 12, 31, 5, 25, 14, 34]
    assert out["track_of"].reshape(-1)[[3, 12, 31, 5, 25, 14, 34, 6, 7, 8]].tolist() == [0, 0, 0, 1, 1, 2, 2, -1, -1, -1]
    kept = to.tracks_from_edges(u, v, n_images, S, keep_conflicts=True)
    assert kept["n_tracks"] == 4 and kept["n_conflicting"] == 1 and kept["n_short"] == 1
    assert (kept["obs"][:, 0] * S + kept["obs"][:, 1]).tolist() == [3, 12, 31, 5, 25, 6, 7, 14, 34]
    long3 = to.tracks_from_edges(u, v, n_images, S, min_length=3)
    assert long3["n_tracks"] == 1 and long3["n_short"] == 3 and long3["offsets"].tolist() == [0, 3]
    # rows: flags, the pair filter and invalid rows
    pairs = np.array([[0, 1], [1, 2]])
    rows = np.array([[1, 2, 0], [3, 4, 0], [12, 1, 0], [5, 6, 0]], np.int32)
    r = to.build_tracks(pairs, [0, 2], [2, 2], rows, np.array([1, 0, 1, 1], np.uint8), [20, 20], n_images, S)
    assert r["n_invalid_rows"] == 1 and (r["obs"][:, 0] * S + r["obs"][:, 1]).tolist() == [1, 12, 15, 26]
    r = to.build_tracks(pairs, [0, 2], [2, 2], rows, None, [20, 14], n_images, S)
    assert r["n_invalid_rows"] == 0 and r["n_tracks"] == 2


def test_track_params_size():
    from sfm_b200 import _lib

    assert C.sizeof(_lib.TrackParams) == 32
    assert [f[0] for f in _lib.TrackParams._fields_] == ["min_pair_inliers", "min_length", "keep_conflicts", "reserved"]


def test_track_entry_points_reject_bad_arguments_without_a_gpu():
    """Every rejection returns SFM_ERR_ARG with its message before any CUDA call (pointers are fake and never read)."""
    from sfm_b200 import _lib

    L = _lib.lib()
    err = lambda: L.sfm_last_error().decode()  # noqa: E731
    nb = C.c_size_t(0)
    assert L.sfm_tracks_workspace_bytes(3, 100, None) == -1 and "NULL" in err()
    assert L.sfm_tracks_workspace_bytes(0, 100, C.byref(nb)) == -1 and "positive" in err()
    assert L.sfm_tracks_workspace_bytes(3, -1, C.byref(nb)) == -1 and "positive" in err()
    assert L.sfm_tracks_workspace_bytes(65536, 32768, C.byref(nb)) == -1 and "2^31" in err()
    assert L.sfm_tracks_workspace_bytes(3, 100, C.byref(nb)) == 0 and nb.value >= 300 * 37
    need = nb.value
    ws = 0x100000
    assert L.sfm_tracks_init(3, 100, None, need, None) == -1 and "NULL workspace" in err()
    assert L.sfm_tracks_init(3, 100, ws + 16, need, None) == -1 and "256-byte aligned" in err()
    assert L.sfm_tracks_init(3, 100, ws, need - 1, None) == -1 and "needed" in err()
    assert L.sfm_tracks_init(65536, 32768, ws, need, None) == -1 and "2^31" in err()

    def hook(n_pairs=1, pairs=0x2000, prm=True, **fields):
        p = _lib.TrackParams(15, 2, 0)
        for k, v in fields.items():
            setattr(p, k, v)
        return L.sfm_tracks_hook(3, 100, pairs, n_pairs, 0x3000, 0x4000, 0x5000, None, None, C.byref(p) if prm else None, ws, need, None)

    assert hook(prm=False) == -1 and "NULL params" in err()
    assert hook(min_length=1) == -1 and "min_length must be at least 2, got 1" in err()
    assert hook(keep_conflicts=2) == -1 and "keep_conflicts" in err()
    assert hook(n_pairs=-1) == -1 and "negative pair count" in err()
    assert hook(pairs=None) == -1 and "sfm_tracks_hook: NULL argument" in err()
    assert hook(n_pairs=0) == 0                                  # nothing to add: no launch, no CUDA call

    def fin(out=0x6000, **fields):
        p = _lib.TrackParams(15, 2, 0)
        for k, v in fields.items():
            setattr(p, k, v)
        return L.sfm_tracks_finalize(3, 100, C.byref(p), ws, need, 0x7000, out, 0x8000, 0x9000, None)

    assert fin(min_length=0) == -1 and "sfm_tracks_finalize: min_length" in err()
    assert fin(out=None) == -1 and "sfm_tracks_finalize: NULL argument" in err()
    assert L.sfm_tracks_finalize(3, 100, None, ws, need, 0x7000, 0x6000, 0x8000, 0x9000, None) == -1 and "NULL params" in err()
    with pytest.raises(ValueError):
        from sfm_b200 import tracks as tr

        tr.TrackBuilder(3, 100, "cpu", min_length=1)
