"""match_and_verify end to end against a serial per-pair reference: every output of every pair of a ragged job and of the
bench job, through every batch size, stream mode, output path and optional stage.

The other tests of the plan (sfm_b200/plan.py, sfm_b200/pipeline.py) compare it mostly with itself (overlap against no
overlap, sink against fetch, host upload against a resident bank), which a slip that gives the same wrong answer twice
passes.  Here every job is held to a reference that runs one pair at a time, with no plan, no streams and no batches, built
from the arrays the test gave ``bank.put`` (never read back from the bank):

* matches: ``oracle.exact_match.knn2_ref`` + ``filter_ref`` (the exact integer matcher reference, with the mutual check);
* correspondences ``(xy_i[q], xy_j[t])`` from the input arrays (zeros for an image put without ``xy``);
* RANSAC-F, RANSAC-H (stop target ``h_stop_target(n_inliers_f, h_stop_ratio)``) and two-view pose with the pair's own two
  camera rows: the C oracles of oracle/ransac_oracle.py, themselves pinned to float64 references;
* tracks: ``oracle.track_oracle.build_tracks_host`` on the reference rows.

Every array of ``to_host()``, the device per-pair arrays of ``VerifiedPairs``, the rows of the device row sink,
``d2h_bytes`` and the tracks are compared bit for bit; a difference names the job, the array, the pair and its batch.

Job (a), ``ragged_job``: 24 images in several ``put`` calls -- eight views of one scene (768 to 2,048 features, one put
without ``xy``), two views of a second scene with 8,192 features whose pair has more than 4,096 verified matches and makes
pose choose the second rotation of the essential matrix, images with 0, 1, 3, 4, 7, 8 and 300 features, five unrelated
images -- and 531 pairs: the ordered pairs of the 22 narrow images (sparse pairs first, so that the first batch is almost
empty and the pinned row arrays must grow in the middle of the job), self pairs, duplicates and the wide pair.  Job (b) is
the bench job, configs[1], at bench.py's settings.  The ``gpu`` tests print, for each job, the pairs and rows compared and
which of these paths it reached:

1. the pinned row arrays growing while a job is in progress (``HotPathPlan._ensure_rows`` with rows already arrived);
2. pose on a pair with more than 4,096 correspondences that chooses the second rotation (points past the shared stash);
3. a pair with more than 4,096 matches through RANSAC-F, RANSAC-H, pose and the track hook on the same packed rows;
4. pairs with 0, 1-6 and m (the minimal sample) matches in one batch with dense pairs, a batch of empty pairs only, images
   with no features, self, duplicate and reversed pairs;
5. P = 1, P = pair_batch + 1, pair_batch = 1 and the halving of a one-batch job on a ragged pair list;
6. plan-cache eviction, growth of the pinned pair staging buffer, images put in several calls, an image put again with fewer
   features, images without ``xy``.
"""
from __future__ import annotations

import itertools
import time
from dataclasses import dataclass

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import track_oracle as to  # noqa: E402
from pipeline_reference import (BENCH_RANSAC, PAIR_KEYS, RATIO, ROW_KEYS, RPRM, Cfg, Job, Reference,  # noqa: E402
                                compare, compare_tracks, padded, put_job, ragged_job)
from sfm_b200 import synth  # noqa: E402

HAS_CUDA = torch.cuda.is_available()


def gpu_test(fn):
    """GPU tests are marked and skipped one by one: the CPU test of the job's claims must still run without one."""
    return pytest.mark.gpu(pytest.mark.skipif(not HAS_CUDA, reason="needs a GPU")(fn))


ROW_BYTES = {"matches": 12, "inlier": 1, "inlier_h": 1, "in_front": 1, "points3d": 12}
PAIR_BYTES = {"F": 72, "n_inliers": 4, "iters": 4, "H": 72, "n_inliers_h": 4, "R": 72, "t": 24, "n_pose": 4}
STASH = 4096                 # correspondences of pose_kernel's shared-memory stash
DENSE = 256                  # a pair with at least this many matches counts as dense


def decompose_essential(F, cam):
    """(R1, R2, t) of oracle/pose.c's decompose_essential restated in numpy: E = K2^T F K1 / |.|, eigenvectors of E^T E by
    the same cyclic Jacobi (8 sweeps, V from the identity), v0 / v1 the largest / middle, u0 = E v0 / |E v0|, u1 = E v1
    orthogonalised, R1 = U W V^T, R2 = U W^T V^T.  The order of the two rotations depends on the eigenvector signs."""
    K1 = np.array([[cam[0], 0, cam[2]], [0, cam[1], cam[3]], [0, 0, 1.0]])
    K2 = np.array([[cam[4], 0, cam[6]], [0, cam[5], cam[7]], [0, 0, 1.0]])
    E = K2.T @ np.asarray(F, np.float64) @ K1
    E = E / np.linalg.norm(E)
    A, V = E.T @ E, np.eye(3)
    with np.errstate(over="ignore"):
        for _ in range(8):
            for p, q in ((0, 1), (0, 2), (1, 2)):
                if A[p, q] == 0.0:
                    continue
                theta = (A[q, q] - A[p, p]) / (2.0 * A[p, q])
                tt = 1.0 / (abs(theta) + np.sqrt(theta * theta + 1.0))
                tt = -tt if theta < 0 else tt
                c = 1.0 / np.sqrt(tt * tt + 1.0)
                s = tt * c
                A[:, [p, q]] = A[:, [p, q]] @ np.array([[c, s], [-s, c]])
                A[[p, q], :] = np.array([[c, -s], [s, c]]) @ A[[p, q], :]
                V[:, [p, q]] = V[:, [p, q]] @ np.array([[c, s], [-s, c]])
    g = np.diag(A)
    i0, i2 = int(np.argmax(g)), int(np.argmin(g))
    v0, v1 = V[:, i0], V[:, 3 - i0 - i2]
    v2 = np.cross(v0, v1)
    u0 = E @ v0
    u0 = u0 / np.linalg.norm(u0)
    u1 = E @ v1
    u1 = u1 - (u1 @ u0) * u0
    u1 = u1 / np.linalg.norm(u1)
    u2 = np.cross(u0, u1)
    a, b = np.outer(u1, v0) - np.outer(u0, v1), np.outer(u2, v2)
    return b + a, b - a, u2


def pose_candidate(r) -> int:
    """Which rotation of decompose_essential the reference pose chose: 1, 2, or 0 (no pose)."""
    if r["n_pose"] == 0:
        return 0
    R1, R2, _ = decompose_essential(r["F"], r["cam"])
    return 1 if np.allclose(r["R"], R1, atol=1e-9) else 2 if np.allclose(r["R"], R2, atol=1e-9) else -1


# ====================================================================================================== scheduling, restated

def batch_cuts(P, pair_batch, overlap, segments=None):
    """(start, size) of every batch of match_and_verify: runs of <= pair_batch pairs that never cross a segment end; a
    one-batch job of 512 or more pairs is cut in two halves when overlap is on and there are no segments."""
    batch = min(pair_batch, P)
    if overlap and not segments and 512 <= P <= batch:
        batch = -(-P // 2)
    cuts, s0 = [], 0
    for end in (segments or [P]):
        while s0 < end:
            n = min(batch, end - s0)
            cuts.append((s0, n))
            s0 += n
    return cuts


def host_segments(pairs, n_images, n_chunks):
    """(order, segment ends) of match_and_verify_host: pairs stably re-ordered by the upload group of max(i, j)."""
    bounds = (n_images * np.linspace(0.0, 1.0, n_chunks + 1)).round().astype(int)
    bounds[-1] = n_images
    group = np.searchsorted(bounds[1:], pairs.max(axis=1), side="right")
    order = np.argsort(group, kind="stable")
    return order, list(np.cumsum([int((group == c).sum()) for c in range(n_chunks)]))


def rows_cap_trace(totals, P, cap):
    """The pinned row capacity along a job, restated from HotPathPlan.fetch_begin / _ensure_rows: [(rows already arrived,
    new capacity)] for every growth, starting from capacity ``cap``."""
    r0 = p0 = 0
    out = []
    for total, n in totals:
        per_pair = (r0 + total) / max(p0 + n, 1)
        expect = int(1.1 * per_pair * P) + 1024
        if r0 + total > cap:
            cap = max(r0 + total, expect, 2 * cap, 1 << 16)
            out.append((r0, cap))
        r0, p0 = r0 + total, p0 + n
    return out


def batch_totals(counts, cuts):
    return [(int(counts[s: s + n].sum()), n) for s, n in cuts]


# ====================================================================================================== the CPU claims

@pytest.fixture(scope="module")
def job_a():
    return ragged_job()


def pair_index(pairs, p):
    return [k for k, q in enumerate(pairs.tolist()) if tuple(q) == tuple(p)]


def test_job_builds_what_it_claims(job_a):
    """Job (a) has what the GPU tests rely on, from the reference alone (GEMMs on the CPU)."""
    job = job_a
    pairs, P = job.pairs, len(job.pairs)
    ref = Reference(job.images, job.K, "cpu")
    counts = np.array([len(ref.matches(int(i), int(j))[0]) for i, j in pairs])
    assert 512 < P <= 2048 and len(job.images) == 24
    assert max(len(d) for k, (d, _) in enumerate(job.images) if k not in job.wide) <= 2048
    # match counts: empty images, the planted 1 / 3 / 4 / 7 / 8 matches, self pairs of dense views, the wide pair
    for k in job.roles["empty"]:
        assert len(job.images[k][0]) == 0 and all(counts[p] == 0 for p in range(P) if k in pairs[p])
    for k, m in ((10, 1), (21, 3), (11, 4), (12, 7), (13, 8)):
        assert counts[pair_index(pairs, (k, 1))[0]] == m, k
    for k in range(8):
        assert counts[pair_index(pairs, (k, k))[0]] == len(job.images[k][0])
    assert set(counts[counts < 9]) >= {0, 1, 3, 4, 7, 8}
    assert not job.images[7][1].any() and counts[pair_index(pairs, (7, 0))[0]] >= DENSE
    assert len(pair_index(pairs, job.wide)) == 2 and pair_index(pairs, (3, 5)) and pair_index(pairs, (5, 3))
    assert len(set(map(tuple, pairs.tolist()))) < P                         # duplicates
    # which batches are empty, for each pair_batch the GPU tests use
    empty = {}
    for pb in (1, 2, 3, 7, P - 1, P, 2048):
        cuts = batch_cuts(P, pb, True)
        empty[pb] = [b for b, (s, n) in enumerate(cuts) if not counts[s: s + n].any()]
        assert empty[pb] or pb > 7, pb
    assert empty[7][0] == 0 and len(empty[1]) == int((counts == 0).sum())
    # the halves of the ragged job: the first is almost empty, the second is dense and mixes every size
    cuts = batch_cuts(P, 2048, True)
    assert cuts == [(0, -(-P // 2)), (-(-P // 2), P // 2)]
    (s0, n0), (s1, n1) = cuts
    assert 0 < counts[:n0].sum() < 0.05 * counts.sum() and counts.sum() > 1 << 16
    second = counts[s1:]
    assert (second == 0).any() and ((second >= 1) & (second <= 6)).any() and (second == 8).any() and (second >= DENSE).any()
    # the mid-job growth of the pinned rows, restated from fetch_begin: a fresh plan sizes them for 64 Ki rows after the
    # first half, the second half outgrows them with rows already arrived
    trace = rows_cap_trace(batch_totals(counts, cuts), P, 0)
    assert trace[0] == (0, 1 << 16) and len(trace) == 2 and trace[1][0] == counts[:n0].sum() > 0, trace
    # the wide pair: more than 4,096 verified matches, pose chooses the second rotation, in-front points past the stash
    # (which rotation comes second depends on the signs of Jacobi eigenvectors, so on the RANSAC stream: the pair is listed twice)
    wide = [ref.pair(*job.wide, p, Cfg(pose=True)) for p in pair_index(pairs, job.wide)]
    r = next(r for r in wide if pose_candidate(r) == 2)
    assert r["n_inliers"] > STASH and [pose_candidate(w) for w in wide] == [2, 1]
    assert (np.nonzero(r["in_front"])[0] >= STASH).sum() > 1000
    print(f"\njob (a): {P} pairs, {int(counts.sum())} rows; empty batches at pair_batch 1/2/3/7: "
          f"{[len(empty[pb]) for pb in (1, 2, 3, 7)]}; row capacity {trace}; wide pair {int(counts[pair_index(pairs, job.wide)[0]])} "
          f"matches, {r['n_inliers']} inliers, {r['n_pose']} in front, candidate {pose_candidate(r)}")


# ====================================================================================================== the GPU runs

PATHS: dict = {}             # path number -> set of what reached it


def reach(path, what):
    PATHS.setdefault(path, set()).add(what)



STAGES = {
    "F": dict(),
    "H": dict(homography=True),
    "pose": dict(homography=True, pose=True),
    "tracks_inlier": dict(homography=True, pose=True, tracks="inlier"),
    "tracks_inlier_h": dict(homography=True, pose=True, tracks="inlier_h"),
    "tracks_in_front": dict(homography=True, pose=True, tracks="in_front"),
}


@dataclass(frozen=True)
class Run:
    route: str = "fetch"         # fetch | view | summaries | sink | host1 | host3
    pb: int = 2048
    stage: str = "F"
    overlap: bool = True
    mutual: bool = False
    prefilter: bool = True
    ids: str = "default"         # default | custom
    seed: int = RPRM["seed"]
    solver: str = RPRM["solver"]


def custom_ids(P):
    return (np.arange(P, dtype=np.int64) * 2654435761 + 977) % (1 << 32)


class Env:
    """One bank (job (a)), its reference, the host-upload bank and its padded reference, and what every run reached."""

    def __init__(self, job: Job):
        import sfm_b200

        self.sfm = sfm_b200
        self.job = job
        self.bank = sfm_b200.DescriptorBank(len(job.images), 8192)
        put_job(self.bank, job)
        reach(6, "images put in several calls")
        reach(6, "images put without xy")
        self.ref = Reference(job.images, job.K, "cuda")
        self.desc_pad, self.xy_pad, pad_images = padded(job, 8192)
        self.host_bank = sfm_b200.DescriptorBank(len(job.images), 8192)
        self.host_ref = Reference(pad_images, job.K, "cuda")
        self.growth = []                                       # (id of the plan, rows arrived, old capacity, new capacity) of every _ensure_rows

    def params(self, run: Run):
        st = STAGES[run.stage]
        kw = dict(ratio=RATIO, mutual=run.mutual, prefilter=run.prefilter, pair_batch=run.pb, overlap=run.overlap,
                  **dict(RPRM, seed=run.seed, solver=run.solver), homography=st.get("homography", False))
        if st.get("pose"):
            kw["intrinsics"] = self.job.K
        if st.get("tracks"):
            kw.update(tracks=True, track_flags=st["tracks"])
        cfg = Cfg(mutual=run.mutual, rprm=tuple(sorted(dict(RPRM, seed=run.seed, solver=run.solver).items())),
                  homography=kw["homography"], pose=bool(st.get("pose")))
        return kw, cfg

    def run(self, run: Run, pairs=None, ids=None, label=None, ref=None):
        """Run one job, compare it with the reference, record the paths it reached; returns (res, reference)."""
        sfm = self.sfm
        pairs = self.job.pairs if pairs is None else pairs
        P = len(pairs)
        if ids is None:
            ids = custom_ids(P) if run.ids == "custom" else np.arange(P, dtype=np.int64)
        kw, cfg = self.params(run)
        label = label or f"{run}"
        host_route = run.route.startswith("host")
        bank = self.host_bank if host_route else self.bank
        plans_before = dict(bank.__dict__.get("_plans", {}))
        stage_before = bank.__dict__.get("_pair_stage")
        stage_before = 0 if stage_before is None else stage_before[0].shape[0]
        n_growth = len(self.growth)
        t0 = time.perf_counter()
        if host_route:
            n_chunks = int(run.route[4:])
            order, seg = host_segments(pairs, len(self.job.images), n_chunks)
            res, got_order = sfm.match_and_verify_host(self.desc_pad, self.xy_pad, pairs, bank=bank, n_chunks=n_chunks,
                                                       fetch=True if n_chunks == 1 else "view",
                                                       pair_ids=None if run.ids == "default" else ids, **kw)
            assert np.array_equal(got_order, order), label
            want = (ref or self.host_ref).job(pairs[order], ids[order], cfg)
            cuts = batch_cuts(P, run.pb, run.overlap, seg)
        else:
            want = (ref or self.ref).job(pairs, ids, cfg)
            cuts = batch_cuts(P, run.pb, run.overlap)
            pid = None if run.ids == "default" else ids
            if run.route == "sink":
                assert pid is None
                from sfm_b200 import dist as sdist

                out, res = sdist.match_and_verify_sharded(bank, pairs, **kw)
            else:
                fetch = {"fetch": True, "view": "view", "summaries": False}[run.route]
                res = sfm.match_and_verify(bank, pairs, pair_ids=pid, fetch=fetch, **kw)
        torch.cuda.synchronize()
        elapsed = time.perf_counter() - t0
        rows = [k for k in ROW_KEYS if k in want]
        # device per-pair arrays of VerifiedPairs
        dev = {k: getattr(res, k).cpu().numpy() for k in PAIR_KEYS if getattr(res, k) is not None}
        assert set(dev) == {k for k in PAIR_KEYS if k in want}, label
        compare(label + " [device]", dev, want, cuts, P)
        if run.route == "sink":
            got = {k: v.cpu().numpy() for k, v in out.items() if isinstance(v, torch.Tensor)}
            compare(label + " [sink]", got, want, cuts, P, rows=rows, row_start=got["row_start"])
            assert np.array_equal(out["pairs"], pairs), label
        elif run.route != "summaries":
            got = res.to_host()
            assert np.array_equal(got["pairs"], want["pairs"]), label
            assert set(got) == {"pairs", "offsets"} | {k for k in PAIR_KEYS if k in want} | set(rows), (label, sorted(got))
            compare(label + " [to_host]", got, want, cuts, P, rows=rows)
            d2h = 4 * (P + len(cuts)) + sum(ROW_BYTES[k] for k in rows) * len(want["matches"]) + \
                sum(PAIR_BYTES[k] for k in PAIR_KEYS if k in want and k != "n_matches") * P
            assert res.d2h_bytes == d2h, (label, res.d2h_bytes, d2h)
        st = STAGES[run.stage]
        if st.get("tracks"):
            b = self.host_bank if host_route else self.bank
            twant = to.build_tracks_host(want, b.n_images, b.max_feats, flags=st["tracks"])
            compare_tracks(label, out["tracks"] if run.route == "sink" else res.tracks, twant)
        self.record(run, label, want, cuts, P, res, plans_before, stage_before, n_growth, host_route, elapsed)
        return res, want

    def record(self, run, label, want, cuts, P, res, plans_before, stage_before, n_growth, host_route, elapsed):
        counts = want["n_matches"]
        reached = set()
        # 1: row arrays grown with rows already arrived, exactly as fetch_begin's arithmetic says
        ev = [e for e in self.growth[n_growth:] if e[0] == id(res.plan)]
        if ev:
            trace = rows_cap_trace(batch_totals(counts, cuts), P, ev[0][2])
            got = [(e[1], e[3]) for e in ev if e[3] != e[2]]
            assert got == trace, (label, got, trace)
            if any(r0 > 0 for r0, _ in trace):
                reached.add(1)
                reach(1, label)
        # 2 / 3: the wide pair
        wide = [p for p in range(P) if tuple(want["pairs"][p]) == self.job.wide]
        per = want["_pairs"]
        for p in wide:
            r = per[p]
            if "n_pose" in r and r["n_inliers"] > STASH and pose_candidate(r) == 2 and (np.nonzero(r["in_front"])[0] >= STASH).any():
                reached.add(2)
                reach(2, label)
            if len(r["matches"]) > STASH and run.stage.startswith("tracks") and "n_pose" in r and "n_inliers_h" in r:
                reached.add(3)
                reach(3, label)
        # 4: one batch with 0, 1-6 and m matches beside a dense pair; a batch of empty pairs only
        m = 7 if run.solver == "7pt" else 8
        for s, n in cuts:
            c = counts[s: s + n]
            if (c == 0).any() and ((c >= 1) & (c <= 6)).any() and (c == m).any() and (c >= DENSE).any():
                reached.add(4)
                reach(4, f"mixed batch, m = {m}")
            if len(cuts) > 1 and not c.any():
                reach(4, "batch of empty pairs")
        pl = want["pairs"].tolist()
        if any(i == j for i, j in pl):
            reach(4, "self pairs")
        if len(set(map(tuple, pl))) < P and any([j, i] in pl for i, j in pl if i != j):
            reach(4, "duplicate and reversed pairs")
        if any(len(self.job.images[k][0]) == 0 for k in set(np.ravel(pl))):
            reach(4, "images with no features")
        # 5: batch shapes
        if P == 1:
            reach(5, "P = 1")
        if P == run.pb + 1:
            reach(5, "P = pair_batch + 1")
        if run.pb == 1:
            reach(5, "pair_batch = 1")
        if run.overlap and not host_route and 512 <= P <= run.pb and counts.min() == 0 and counts.max() > STASH:
            reach(5, "halving of a ragged one-batch job")
        # 6: plan cache and staging buffer
        plans = res.plan.bank.__dict__.get("_plans", {})
        if len(plans_before) >= 4 and res.plan not in plans_before.values():
            assert len(plans) == 1 and res.plan in plans.values(), label
            reach(6, "plan cache eviction")
        stage = self.bank.__dict__.get("_pair_stage")
        if not host_route and stage_before and stage[0].shape[0] > stage_before:
            reach(6, "staging buffer growth")
        print(f"{label}: {P} pairs, {len(want['matches'])} rows, {len(cuts)} batches, {elapsed:.2f} s, paths {sorted(reached)}")


def covering_runs(P):
    """A pairwise covering set of runs: every value of every dimension appears, and every pair of values of two dimensions
    meets in some run (the sink has no pair_ids of its own, so it never meets custom ids)."""
    dims = dict(pb=[1, 2, 3, 7, P - 1, P, 2048], route=["fetch", "view", "summaries", "sink", "host1", "host3"],
                stage=list(STAGES), overlap=[True, False], mutual=[False, True], prefilter=[True, False], ids=["default", "custom"])
    names = list(dims)

    def ok(row):
        return not (row["route"] == "sink" and row["ids"] == "custom")

    need = set()
    for a, b in itertools.combinations(names, 2):
        for va in dims[a]:
            for vb in dims[b]:
                if ok({"route": None, "ids": None, a: va, b: vb}):
                    need.add((a, va, b, vb))
    rng = np.random.default_rng(7)
    runs = []
    while need:
        best, gain = None, -1
        first = sorted(need, key=repr)[0]
        for _ in range(200):
            row = {k: dims[k][rng.integers(len(dims[k]))] for k in names}
            row[first[0]], row[first[2]] = first[1], first[3]
            if not ok(row):
                continue
            g = sum((a, row[a], b, row[b]) in need for a, b in itertools.combinations(names, 2))
            if g > gain:
                best, gain = row, g
        for a, b in itertools.combinations(names, 2):
            need.discard((a, best[a], b, best[b]))
        runs.append(Run(**best))
    return runs


@pytest.fixture(scope="module")
def env(job_a):
    return Env(job_a)


@pytest.fixture
def spy(env, monkeypatch):
    from sfm_b200 import plan as plan_mod

    orig = plan_mod.HotPathPlan._ensure_rows

    def ensure_rows(self, rows, expect_total):
        cap = self._rows_cap
        orig(self, rows, expect_total)
        env.growth.append((id(self), self.job_rows, cap, self._rows_cap))

    monkeypatch.setattr(plan_mod.HotPathPlan, "_ensure_rows", ensure_rows)
    return env


@gpu_test
def test_ragged_job_on_a_fresh_bank_grows_its_rows(spy):
    """The first job on the bank: two halves, the first almost empty; the pinned rows grow after the first half has
    arrived, with every stage and tracks (paths 1, 2, 3, 5)."""
    env = spy
    env.run(Run(route="fetch", pb=2048, stage="tracks_in_front"), label="fresh bank, halves")
    assert 1 in PATHS and 2 in PATHS and 3 in PATHS


@gpu_test
def test_ragged_job_through_the_scheduling_matrix(spy):
    """Every run of a pairwise covering set of (pair_batch, output path, stages, overlap, mutual, prefilter, pair_ids)
    against the reference."""
    env = spy
    P = len(env.job.pairs)
    runs = covering_runs(P)
    for k, run in enumerate(runs):
        env.run(run, label=f"matrix {k + 1}/{len(runs)} {run}")


@gpu_test
def test_bank_and_plan_lifecycle(spy):
    """Five parameter sets (the plan cache is cleared), a one-pair job followed by a job of 4,644 pairs (the pair staging
    buffer grows), then an image put again with fewer features and the same job checked again."""
    env = spy
    job = env.job
    for k, (seed, solver) in enumerate([(21, "8pt"), (22, "7pt"), (23, "8pt"), (24, "7pt"), (25, "8pt")]):
        env.run(Run(route="fetch", pb=len(job.pairs), seed=seed, solver=solver), label=f"parameter set {k + 1}")
    wide = np.asarray([job.wide], np.int32)
    env.run(Run(route="fetch", stage="pose"), pairs=wide, label="one pair")
    long_pairs = np.tile(job.pairs, (9, 1))
    env.run(Run(route="summaries", ids="custom"), pairs=long_pairs, ids=np.tile(custom_ids(len(job.pairs)), 9), label="9 x the job")
    # view 0 again with its first 600 features: rows 600..2047 of the bank are stale and must never match
    d, x = job.images[0]
    env.bank.put(0, d[None, :600], xy=x[None, :600])
    ref2 = env.ref.replaced(0, (d[:600], x[:600]))
    _, want = env.run(Run(route="fetch", stage="tracks_inlier"), label="view 0 put again with 600 features", ref=ref2)
    q = np.concatenate([r["matches"][:, 0] for r, (i, _) in zip(want["_pairs"], want["pairs"]) if i == 0])
    t = np.concatenate([r["matches"][:, 1] for r, (_, j) in zip(want["_pairs"], want["pairs"]) if j == 0])
    assert len(q) and len(t) and q.max() < 600 and t.max() < 600
    reach(6, "image put again with fewer features")
    env.bank.put(0, d[None], xy=x[None])                       # (the bank as the job says, for any later test)


@gpu_test
def test_every_path_was_reached():
    """The runs above reached all six paths (the module's tests run in order)."""
    for p in sorted(PATHS):
        print(f"path {p}: {sorted(PATHS[p])[:8]}")
    assert sorted(PATHS) == [1, 2, 3, 4, 5, 6]
    assert {"batch of empty pairs", "self pairs", "duplicate and reversed pairs", "images with no features"} <= PATHS[4]
    assert any(w.startswith("mixed batch") for w in PATHS[4])
    assert {"P = 1", "P = pair_batch + 1", "pair_batch = 1", "halving of a ragged one-batch job"} <= PATHS[5]
    assert {"plan cache eviction", "staging buffer growth", "image put again with fewer features", "images put in several calls",
            "images put without xy"} <= PATHS[6]


@gpu_test
def test_bench_job_equals_the_reference():
    """configs[1] (50 x 8,192 features, 1,225 exhaustive pairs) at bench.py's settings: the resident path at its default
    pair_batch (two halves of 613 and 612 pairs) and the end-to-end host-upload path (n_chunks=3, pair_batch=512, views)."""
    import sfm_b200

    sc = synth.make_scene(50, 8192, seed=2001)
    pairs = synth.exhaustive_pairs(50)
    P = len(pairs)
    ref = Reference([(sc.desc[k], sc.xy[k]) for k in range(50)], synth.K_INTR, "cuda")
    cfg = Cfg(rprm=tuple(sorted(dict(BENCH_RANSAC, min_inliers=0).items())))
    t0 = time.perf_counter()
    want = ref.job(pairs, np.arange(P), cfg)
    print(f"\nbench reference: {time.perf_counter() - t0:.1f} s")
    bank = sfm_b200.DescriptorBank(50, 8192)
    bank.put(0, sc.desc, xy=sc.xy)
    res = sfm_b200.match_and_verify(bank, pairs, ratio=RATIO, pair_batch=2048, fetch=True, **BENCH_RANSAC)
    cuts = batch_cuts(P, 2048, True)
    assert cuts == [(0, 613), (613, 612)]
    got = res.to_host()
    compare("bench resident", got, want, cuts, P, rows=["matches", "inlier"])
    compare("bench resident [device]", {k: getattr(res, k).cpu().numpy() for k in ("n_matches", "F", "n_inliers", "iters")}, want, cuts, P)
    assert res.d2h_bytes == 4 * (P + 2) + 13 * len(want["matches"]) + 80 * P
    res, order = sfm_b200.match_and_verify_host(sc.desc, sc.xy, pairs, n_chunks=3, ratio=RATIO, pair_batch=512, fetch="view", **BENCH_RANSAC)
    order_r, seg = host_segments(pairs, 50, 3)
    assert np.array_equal(order, order_r)
    want_h = ref.job(pairs[order], order, cfg)
    cuts = batch_cuts(P, 512, True, seg)
    got = res.to_host()
    compare("bench host upload", got, want_h, cuts, P, rows=["matches", "inlier"])
    assert res.d2h_bytes == 4 * (P + len(cuts)) + 13 * len(want["matches"]) + 80 * P
    print(f"bench job: {P} pairs, {len(want['matches'])} rows, resident 2 batches, host upload {len(cuts)} batches")
