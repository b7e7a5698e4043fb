"""The serial per-pair reference of ``match_and_verify`` and the jobs it is run on, shared by
tests/test_gpu_pipeline_reference.py (one GPU) and tests/test_gpu_sharded_reference.py (``match_and_verify_sharded`` on 1 to 8
ranks).  Not a test module: it holds no tests.

The reference runs one pair at a time, with no plan, no streams and no batches, from the arrays a test gave ``bank.put``
(never read back from the bank): ``oracle.exact_match`` for the matches, the C RANSAC-F / RANSAC-H / pose oracles of
oracle/ransac_oracle.py with the pair's RANSAC stream id and its own two camera rows.  ``compare`` and ``compare_tracks`` hold
a result to it bit for bit and name the first pair that differs.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

from oracle import ransac_oracle as ro
from oracle.exact_match import filter_ref, knn2_ref
from sfm_b200 import _lib as slib
from sfm_b200 import synth
from sfm_b200.plan import OUTPUTS, intrinsics_rows
from sfm_b200.ransac import h_stop_target

RATIO = 0.75
RPRM = dict(thr=3.0, confidence=0.99, max_iters=300, solver="8pt", score="sym_epipolar", lo=False, seed=11, min_inliers=0)
BENCH_RANSAC = dict(thr=3.0, confidence=0.99, max_iters=2000, solver="8pt", score="sym_epipolar", lo=False, seed=1)   # bench.py
PAIR_KEYS = ("n_matches", "F", "n_inliers", "iters", "H", "n_inliers_h", "R", "t", "n_pose")
ROW_KEYS = ("matches", "inlier", "inlier_h", "in_front", "points3d")


# ====================================================================================================== the jobs

@dataclass
class Job:
    images: list                   # (desc uint8 [n,128], xy float32 [n,2]) per image, as given to bank.put (xy zeros when put without)
    puts: list                     # (first image, image ids, with xy) of each bank.put call
    pairs: np.ndarray              # int32 [P,2]
    K: np.ndarray                  # float64 [n_images,3,3] per-image intrinsics
    wide: tuple = (0, 0)           # the pair with more than 4,096 matches
    roles: dict = field(default_factory=dict)


def _image(desc, xy):
    return np.ascontiguousarray(desc, np.uint8).reshape(-1, 128), np.ascontiguousarray(xy, np.float32).reshape(-1, 2)


def ragged_job() -> Job:
    """Job (a); see the module docstring.  Image ids: 0-7 views of scene A (7 put without xy), 8, 9, 23 empty, 10-13 and 21
    the first 1, 4, 7, 8, 3 matches of pair (0, 1) taken out of view 0, 14-17 and 20 unrelated, 18-19 the wide views,
    22 a 300-feature subset of view 3."""
    sa = synth.make_scene(8, 2048, seed=4242)
    sizes = [2048, 2048, 1536, 1024, 2048, 1024, 768, 2048]
    imgs = [None] * 24
    for k, n in enumerate(sizes):
        imgs[k] = _image(sa.desc[k, :n], sa.xy[k, :n] if k != 7 else np.zeros((n, 2)))
    fwd = knn2_ref(imgs[0][0], imgs[1][0], device="cpu")
    q01 = filter_ref(fwd)[0]
    for k, m in ((10, 1), (11, 4), (12, 7), (13, 8), (21, 3)):
        imgs[k] = _image(imgs[0][0][q01[:m]], imgs[0][1][q01[:m]])
    for k in (8, 9, 23):
        imgs[k] = _image(np.zeros((0, 128)), np.zeros((0, 2)))
    rng = np.random.default_rng(np.random.PCG64(99))
    for k, n in ((14, 512), (15, 1024), (16, 256), (17, 768), (20, 128)):
        xy = np.stack([rng.uniform(0, synth.IMG_W, n), rng.uniform(0, synth.IMG_H, n)], 1)
        imgs[k] = _image(synth.sift_like(rng, n), xy)
    imgs[22] = _image(sa.desc[3, 1024:1324], sa.xy[3, 1024:1324])
    sw = synth.make_scene(2, 8192, seed=42, shared_frac=1.0)
    imgs[18], imgs[19] = _image(sw.desc[1], sw.xy[1]), _image(sw.desc[0], sw.xy[0])
    # several put calls: views with counts, the view without xy alone, the small images, the wide pair
    puts = [(0, list(range(7)), True), (7, [7], False), (8, list(range(8, 18)), True), (18, [18, 19], True),
            (20, list(range(20, 24)), True)]

    dense = list(range(8))
    narrow = [k for k in range(24) if k not in (18, 19)]
    empty_imgs = [8, 9, 23]
    tiny_imgs = [10, 11, 12, 13, 21]

    def rank(p):
        i, j = p
        if i in empty_imgs or j in empty_imgs:
            return 0
        if i == 22 or j == 22:
            return 1
        if i in (14, 15, 16, 17, 20) or j in (14, 15, 16, 17, 20):
            return 2
        if i in tiny_imgs or j in tiny_imgs:
            return 3
        return 4
    ordered = [(i, j) for i in narrow for j in narrow if i != j]
    sparse = sorted((p for p in ordered if rank(p) < 4), key=rank)          # stable: by kind, then (i, j)
    sparse.insert(len(sparse) - 40, (0, 1))                                # one dense pair among the tiny ones
    dense_pairs = [p for p in ordered if rank(p) == 4 and p != (0, 1)]
    extras = [(k, k) for k in dense] + [(13, 13), (8, 8), (21, 21), (9, 9)]
    extras += [dense_pairs[k] for k in rng.permutation(len(dense_pairs))[:55]]
    tail = dense_pairs + extras
    tail = [tail[k] for k in rng.permutation(len(tail))]
    pairs = sparse + tail
    # the wide pair twice, at stream ids where the RANSAC-F model makes pose choose the second rotation, then the first
    pairs.insert(491, (18, 19))
    pairs.insert(496, (18, 19))
    pairs = np.asarray(pairs, np.int32)

    K = np.broadcast_to(synth.K_INTR, (24, 3, 3)).copy()
    for k in range(24):
        if k not in (18, 19):                                               # the wide views keep the scene's own K
            K[k, 0, 0], K[k, 1, 1], K[k, 0, 2], K[k, 1, 2] = 900 + 13 * k, 880 + 11 * k, 950 - 3 * k, 530 + 2 * k
    return Job(imgs, puts, pairs, K, wide=(18, 19), roles=dict(empty=empty_imgs, no_xy=[7], tiny=tiny_imgs))


def put_job(bank, job: Job):
    """Fill ``bank`` the way the job says: one put per entry of ``job.puts``, counts and padding from the images."""
    for first, ids, with_xy in job.puts:
        n = max(max(len(job.images[k][0]) for k in ids), 1)
        desc = np.zeros((len(ids), n, 128), np.uint8)
        xy = np.zeros((len(ids), n, 2), np.float32)
        counts = np.zeros(len(ids), np.int32)
        for r, k in enumerate(ids):
            d, x = job.images[k]
            desc[r, : len(d)], xy[r, : len(d)], counts[r] = d, x, len(d)
        bank.put(first, desc, counts=counts, xy=xy if with_xy else None)


def padded(job: Job, n: int):
    """The job's images as the dense [n_images, n, 128] / [n_images, n, 2] arrays of match_and_verify_host (zero rows pad
    every image to n features), and the same images as reference inputs."""
    desc = np.zeros((len(job.images), n, 128), np.uint8)
    xy = np.zeros((len(job.images), n, 2), np.float32)
    for k, (d, x) in enumerate(job.images):
        desc[k, : len(d)], xy[k, : len(d)] = d, x
    return desc, xy, [(desc[k], xy[k]) for k in range(len(job.images))]


# ====================================================================================================== the reference

@dataclass(frozen=True)
class Cfg:
    """What the reference of one job depends on besides the images, the pair and its RANSAC stream id."""
    mutual: bool = False
    rprm: tuple = tuple(sorted(RPRM.items()))
    homography: bool = False
    h_ratio: float | None = 0.8
    pose: bool = False
    dist: float = 50.0


class Reference:
    """Serial per-pair reference over the images given to the bank.  kNN tables and per-pair results are cached; a
    ``replaced`` reference keeps the entries that do not involve the replaced image."""

    def __init__(self, images, K, device):
        self.images, self.device = list(images), device
        self.cam = intrinsics_rows(K, len(images))
        self._dev, self._knn, self._res = {}, {}, {}

    def replaced(self, k, image):
        r = Reference(self.images, self.cam, self.device)
        r.images[k] = image
        r._knn = {key: v for key, v in self._knn.items() if k not in key}
        r._res = {key: v for key, v in self._res.items() if k not in key[:2]}
        return r

    def _desc(self, k):
        if k not in self._dev:
            self._dev[k] = torch.from_numpy(self.images[k][0]).to(self.device)
        return self._dev[k]

    def knn(self, i, j):
        if (i, j) not in self._knn:
            self._knn[(i, j)] = knn2_ref(self._desc(i), self._desc(j))
        return self._knn[(i, j)]

    def matches(self, i, j, mutual=False):
        return filter_ref(self.knn(i, j), self.knn(j, i) if mutual else None, RATIO, "cv2_f32", mutual)

    def pair(self, i, j, pid, cfg: Cfg) -> dict:
        key = (i, j, int(pid), cfg)
        if key in self._res:
            return self._res[key]
        q, t, d = self.matches(i, j, cfg.mutual)
        p1, p2 = self.images[i][1][q], self.images[j][1][t]
        rp = dict(cfg.rprm)
        F, mask, ninl, iters = ro.ransac_f(p1, p2, pair_id=int(pid), solver=slib.SOLVERS[rp["solver"]], score=slib.SCORES[rp["score"]],
                                           thr=rp["thr"], max_iters=rp["max_iters"], confidence=rp["confidence"], seed=rp["seed"],
                                           lo=rp["lo"], min_inliers=rp["min_inliers"])
        F = np.zeros((3, 3)) if F is None else F
        r = dict(matches=np.stack([q, t, d], 1).astype(np.int32).reshape(-1, 3), F=F, n_inliers=ninl, iters=iters, inlier=mask)
        if cfg.homography:
            tgt = 0 if cfg.h_ratio is None else h_stop_target(ninl, cfg.h_ratio)
            H, hm, hn, _ = ro.ransac_h(p1, p2, pair_id=int(pid), thr=rp["thr"], max_iters=rp["max_iters"], confidence=rp["confidence"],
                                       seed=rp["seed"], lo=rp["lo"], stop_target=tgt)
            r.update(H=np.zeros((3, 3)) if H is None else H, n_inliers_h=hn, inlier_h=hm)
        if cfg.pose:
            cam = np.concatenate([self.cam[i], self.cam[j]])
            n, R, tv, _, pm, X = ro.two_view_pose(p1, p2, F, cam, mask=mask, distance_thresh=cfg.dist)
            r.update(R=R, t=tv, n_pose=n, in_front=pm, points3d=X, cam=cam)
        self._res[key] = r
        return r

    def job(self, pairs, ids, cfg: Cfg) -> dict:
        """The reference of a whole job in ``to_host()`` layout (plus per-pair extras under ``_pairs``)."""
        pairs = np.asarray(pairs, np.int32).reshape(-1, 2)
        per = [self.pair(int(i), int(j), pid, cfg) for (i, j), pid in zip(pairs, ids)]
        n = np.array([len(r["matches"]) for r in per], np.int32)
        off = np.zeros(len(per) + 1, np.int64)
        np.cumsum(n, out=off[1:])
        out = {"pairs": pairs, "n_matches": n, "offsets": off, "_pairs": per}
        names = ["F", "n_inliers", "iters"] + (["H", "n_inliers_h"] if cfg.homography else []) + (["R", "t", "n_pose"] if cfg.pose else [])
        dt = {"F": np.float64, "H": np.float64, "R": np.float64, "t": np.float64}
        for k in names:
            out[k] = np.array([r[k] for r in per], dt.get(k, np.int32)).reshape((len(per),) + np.shape(per[0][k])) if per else \
                OUTPUTS[k].empty(0).numpy()
        rows = ["matches", "inlier"] + (["inlier_h"] if cfg.homography else []) + (["in_front", "points3d"] if cfg.pose else [])
        for k in rows:
            out[k] = np.concatenate([r[k] for r in per]) if per else OUTPUTS[k].empty(0).numpy()    # (P = 0: the declared empties)
        return out


def _bits(a):
    """The bytes of each leading-axis entry of ``a``: [len(a), bytes per entry]."""
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(len(a), -1) if len(a) else np.zeros((0, 1), np.uint8)


def _batch_of(cuts, p):
    return next(b for b, (s, n) in enumerate(cuts) if s <= p < s + n)


def compare(label, got, want, cuts, P, *, rows=None, row_start=None, where=None):
    """Bit-for-bit comparison of per-pair arrays (``PAIR_KEYS``) and packed row arrays (``ROW_KEYS``) present in ``want``;
    ``row_start`` gives each pair's first row in ``got`` when it is not the reference's packing.  ``where(p)`` says where pair
    p ran (default: its batch among ``cuts``)."""
    pairs = want["pairs"]
    if where is None:
        def where(p):
            return f"of batch {_batch_of(cuts, p)}"

    def fail(name, p, extra=""):
        i, j = pairs[p]
        raise AssertionError(f"{label}: pair {p} ({i}, {j}) {where(p)}: {name} differs from the reference{extra}")

    for name in PAIR_KEYS:
        if name not in want:
            continue
        g = np.asarray(got[name])
        assert g.shape == want[name].shape and g.dtype == want[name].dtype, (label, name, g.shape, g.dtype)
        bad = np.nonzero((_bits(g) != _bits(want[name])).any(1))[0]
        if len(bad):
            fail(name, bad[0], f": got {g[bad[0]].ravel().tolist()}, want {want[name][bad[0]].ravel().tolist()}")
    if rows is None:
        return
    off = want["offsets"]
    start = off[:-1] if row_start is None else np.asarray(row_start, np.int64)
    if row_start is None:
        assert np.array_equal(got["offsets"], off), label
    for name in rows:
        g, w = np.asarray(got[name]), want[name]
        assert g.dtype == w.dtype and g.shape[1:] == w.shape[1:], (label, name)
        if row_start is None:
            assert len(g) == len(w), (label, name, len(g), len(w))
            idx = np.arange(len(w))
        else:
            idx = np.repeat(start - off[:-1], np.diff(off)) + np.arange(len(w))
        bad = np.nonzero((_bits(g[idx]) != _bits(w)).any(1))[0] if len(w) else []
        if len(bad):
            r = bad[0]
            p = int(np.searchsorted(off, r, side="right") - 1)
            fail(name, p, f" at row {r - off[p]}: got {g[idx[r]].ravel().tolist()}, want {w[r].ravel().tolist()}")


def compare_tracks(label, got, want):
    h = got.to_host() if hasattr(got, "to_host") else got
    for k in ("offsets", "obs", "track_of"):
        assert h[k].dtype == want[k].dtype and h[k].shape == want[k].shape and np.array_equal(h[k], want[k]), \
            f"{label}: tracks {k} differs from the reference"
    for k in ("n_tracks", "n_obs", "n_conflicting", "n_short", "n_invalid_rows"):
        assert h[k] == want[k], f"{label}: tracks {k} = {h[k]}, reference {want[k]}"
