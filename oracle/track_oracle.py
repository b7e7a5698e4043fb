"""numpy oracle of the feature tracks (csrc/tracks.cu), built with a different algorithm from the kernels.

The kernels run a lock-free union-find with link-by-index, then sort each component's slice.  Here the connected components
come from iterated min-label propagation over the edges (``np.minimum.at``, once onto the endpoints and once onto their
labels) plus pointer jumping until nothing changes; the dropping and ordering rules are applied with ``np.lexsort``.

The contract both follow: node ``n = image * S + feature``; the used rows of pair (i, j) give edges (i*S + q, j*S + t);
candidates are the components of those edges (nodes = their endpoints); a candidate holding two features of one image is
conflicting and dropped unless ``keep_conflicts``, then a candidate shorter than ``min_length`` is dropped; kept tracks are
numbered by ascending smallest node, observations ascend by node.
"""
from __future__ import annotations

import numpy as np


def used_edges(pairs, row_start, n_rows, rows, row_flag, n_inliers, n_images, S, *, min_pair_inliers=15):
    """(u, v, n_invalid_rows): the edges of the rows that are used, and the count of rows that would be used but name a
    feature outside [0, S) or an image outside [0, n_images)."""
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    P = len(pairs)
    start = np.asarray(row_start, np.int64).reshape(P)
    n = np.maximum(np.asarray(n_rows, np.int64).reshape(P), 0)
    if n_inliers is not None:
        n = np.where(np.asarray(n_inliers, np.int64).reshape(P) >= min_pair_inliers, n, 0)
    first = np.cumsum(n) - n
    idx = np.repeat(start, n) + (np.arange(int(n.sum())) - np.repeat(first, n))
    pid = np.repeat(np.arange(P), n)
    if row_flag is not None:
        sel = np.asarray(row_flag).reshape(-1)[idx] != 0
        idx, pid = idx[sel], pid[sel]
    rows = np.asarray(rows).reshape(-1, 3)
    q, t = rows[idx, 0].astype(np.int64), rows[idx, 1].astype(np.int64)
    i, j = pairs[pid, 0], pairs[pid, 1]
    ok = (q >= 0) & (q < S) & (t >= 0) & (t < S) & (i >= 0) & (i < n_images) & (j >= 0) & (j < n_images)
    return i[ok] * S + q[ok], j[ok] * S + t[ok], int((~ok).sum())


def components(u, v):
    """(nodes ascending, label): ``nodes[label[k]]`` is the smallest node of node k's component."""
    u, v = np.asarray(u, np.int64), np.asarray(v, np.int64)
    nodes, inv = np.unique(np.concatenate([u, v]), return_inverse=True)
    eu, ev = inv[: len(u)], inv[len(u):]
    lab = np.arange(len(nodes))
    while True:
        a, b = lab[eu], lab[ev]
        if np.array_equal(a, b):
            return nodes, lab
        np.minimum.at(lab, eu, b)
        np.minimum.at(lab, ev, a)
        np.minimum.at(lab, a, b)
        np.minimum.at(lab, b, a)
        while True:                                   # pointer jumping to the fixed point
            nxt = lab[lab]
            if np.array_equal(nxt, lab):
                break
            lab = nxt


def tracks_from_edges(u, v, n_images, S, *, min_length=2, keep_conflicts=False, n_invalid_rows=0) -> dict:
    """``offsets`` int64 [T+1], ``obs`` int32 [n_obs, 2], ``track_of`` int32 [n_images, S] and the counts."""
    nodes, lab = components(u, v)
    m = len(nodes)
    order = np.lexsort((np.arange(m), lab))          # by component (= smallest node), then by node
    lab_s, node_s = lab[order], nodes[order]
    head = np.ones(m, bool)
    head[1:] = lab_s[1:] != lab_s[:-1]
    seg = np.cumsum(head) - 1
    n_cand = int(head.sum())
    lens = np.bincount(seg, minlength=n_cand)
    img = node_s // S
    same_img = ~head[1:] & (img[1:] == img[:-1])
    conflict = np.zeros(n_cand, bool)
    conflict[seg[1:][same_img]] = True
    keep = np.ones(n_cand, bool) if keep_conflicts else ~conflict
    short = keep & (lens < min_length)
    keep &= ~short
    tid = np.cumsum(keep) - 1
    sel = keep[seg]
    kept = node_s[sel]
    track_of = np.full(n_images * S, -1, np.int32)
    track_of[kept] = tid[seg[sel]]
    offsets = np.zeros(int(keep.sum()) + 1, np.int64)
    np.cumsum(lens[keep], out=offsets[1:])
    return {"offsets": offsets, "obs": np.stack([kept // S, kept % S], axis=1).astype(np.int32).reshape(-1, 2),
            "track_of": track_of.reshape(n_images, S), "n_tracks": int(keep.sum()), "n_obs": len(kept),
            "n_conflicting": int(conflict.sum()), "n_short": int(short.sum()), "n_invalid_rows": int(n_invalid_rows)}


def build_tracks(pairs, row_start, n_rows, rows, row_flag, n_inliers, n_images, S, *, min_pair_inliers=15, min_length=2,
                 keep_conflicts=False) -> dict:
    """The tracks of packed rows: the same arguments as ``sfm_b200.build_tracks_device``, numpy in and out."""
    u, v, bad = used_edges(pairs, row_start, n_rows, rows, row_flag, n_inliers, n_images, S, min_pair_inliers=min_pair_inliers)
    return tracks_from_edges(u, v, n_images, S, min_length=min_length, keep_conflicts=keep_conflicts, n_invalid_rows=bad)


def build_tracks_host(host: dict, n_images, S, *, flags="inlier", **kw) -> dict:
    """The tracks of a ``VerifiedPairs.to_host()`` result."""
    off = np.asarray(host["offsets"], np.int64)
    return build_tracks(host["pairs"], off[:-1], np.diff(off), host["matches"], None if flags is None else host[flags],
                        host["n_inliers"], n_images, S, **kw)
