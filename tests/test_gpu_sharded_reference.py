"""match_and_verify_sharded (sfm_b200/dist.py) against the serial per-pair reference of tests/pipeline_reference.py, at 1 to
8 ranks.

RANSAC streams are keyed by the global pair index, so one reference per (job, ``Cfg``) serves every world size: every
gathered array is compared bit for bit with ``Reference.job(pairs, ids=global pair index, cfg)``.  A difference names the
world size, the run, the array, the global pair, the rank that owned it and its position in that rank's block.

* World sizes 2, 3, 4 and 8 on GPUs (as many as are visible): one spawned NCCL job per world size runs a list of runs in
  sequence.  After each job the workers copy what ``dst`` holds to the host and write it under ``tmp_path`` (the row arrays
  are views of a region that the job after next rewrites); the parent process builds the reference and does every
  comparison.  The runs: a pairwise covering set over transport, partition, gather, ``dst``, ``pair_batch``, overlap, the
  optional stages, mutual, tracks and a tight ``rows_per_pair_cap`` on the ragged job of tests/pipeline_reference.py; the
  same call three times (the region pair alternates, the third job waits on the reuse fence) and then a change of shape and
  of ``dst`` (cached regions evicted and closed collectively); P = 0, 1, ws - 1, ws + 1 and a list whose pairs on rank 1
  all have zero matches; ``upload_bank_sharded`` with an image count not divisible by the world size, fewer images than
  ranks and a bank with spare slots, followed by a sharded job and by bench.py's end-to-end arm on that bank; and, at the
  largest world size that runs, bench.py's sharded job (configs[2], 19,900 pairs).
* World size 1, in process: no process group; the sink's overflow (``SfmError("row sink overflow")``) is tested only here.
  At more than one rank the rank that raises leaves its peers waiting in ``dist.gather``.
* World sizes 2 to 8 on the CPU (gloo): ``gather_summaries``, ``GatherRegion`` (sendrecv) and ``row_starts`` with payloads
  whose per-pair row counts are those of the ragged job's reference.
"""
from __future__ import annotations

import itertools
import os
import queue as _queue
import time
from dataclasses import dataclass, replace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import bench  # noqa: E402
from oracle import track_oracle as to  # noqa: E402
from pipeline_reference import (PAIR_KEYS, RATIO, ROW_KEYS, RPRM, Cfg, Reference, _bits, compare,  # noqa: E402
                                compare_tracks, put_job, ragged_job)
from sfm_b200 import synth  # noqa: E402

HAS_CUDA = torch.cuda.is_available()
N_GPUS = torch.cuda.device_count() if HAS_CUDA else 0
WORLD_SIZES = (2, 3, 4, 8)
LARGEST = max([w for w in WORLD_SIZES if w <= N_GPUS], default=0)
A_FEATS = 8192                       # the ragged job's bank (its wide views have 8,192 features)
UP_FEATS = 1024                      # the images of the sharded-upload cases
BENCH_CFG = Cfg(rprm=tuple(sorted(dict(bench.RANSAC, min_inliers=0).items())))
PORT_BASE = 34000                    # test_dist_gloo.py uses 29500+, test_gpu_multi.py 29700+, test_gpu_tracks.py 31700+


def port(slot):
    return PORT_BASE + (os.getpid() % 800) * 32 + slot


def gpu_test(fn):
    return pytest.mark.gpu(pytest.mark.skipif(not HAS_CUDA, reason="needs a GPU")(fn))


# ====================================================================================================== the runs

STAGES = {
    "F": dict(),
    "pose": dict(homography=True, pose=True),
    "tracks_inlier": dict(homography=True, pose=True, tracks="inlier", min_length=3),
    "tracks_inlier_h": dict(homography=True, pose=True, tracks="inlier_h", keep_conflicts=True),
    "tracks_in_front": dict(homography=True, pose=True, tracks="in_front"),
    "tracks_all": dict(tracks=None, min_length=3, keep_conflicts=True),
}


@dataclass(frozen=True)
class Run:
    name: str
    kind: str = "sharded"        # sharded | upload (upload_bank_sharded, then a sharded job) | e2e (bench.py's end-to-end arm)
    job: str = "a"               # a (the ragged job) | bench | the name of an upload case
    transport: str = "auto"
    mode: str = "block"
    gather: str = "full"
    dst: int = 0
    pb: int = 2048
    overlap: bool = True
    stage: str = "F"
    mutual: bool = False
    tight_cap: bool = False      # rows_per_pair_cap = the largest n_matches of the job

    def cfg(self):
        if self.job != "a":
            return BENCH_CFG
        st = STAGES[self.stage]
        return Cfg(mutual=self.mutual, homography=st.get("homography", False), pose=bool(st.get("pose")))

    def kwargs(self, K, cap):
        """The keyword arguments of match_and_verify_sharded (``K``: the job's per-image intrinsics)."""
        if self.job != "a":
            return dict(mode=self.mode, dst=self.dst, gather=self.gather, transport=self.transport, ratio=bench.RATIO,
                        pair_batch=self.pb, overlap=self.overlap, **bench.RANSAC)
        st = STAGES[self.stage]
        kw = dict(mode=self.mode, dst=self.dst, gather=self.gather, transport=self.transport, rows_per_pair_cap=cap, ratio=RATIO,
                  mutual=self.mutual, pair_batch=self.pb, overlap=self.overlap, homography=st.get("homography", False), **RPRM)
        if st.get("pose"):
            kw["intrinsics"] = K
        if "tracks" in st:
            kw.update(tracks=True, track_flags=st["tracks"], min_length=st.get("min_length", 2),
                      keep_conflicts=st.get("keep_conflicts", False))
        return kw


def pairwise(dims, ok, seed=5):
    """A pairwise covering set: every pair of values of two dimensions meets in some row that ``ok`` accepts."""
    names = list(dims)
    need = {(a, va, b, vb) for a, b in itertools.combinations(names, 2) for va in dims[a] for vb in dims[b]
            if ok({**{k: dims[k][0] for k in names}, a: va, b: vb}) or ok({**{k: dims[k][-1] for k in names}, a: va, b: vb})}
    rng = np.random.default_rng(seed)
    rows = []
    while need:
        first = sorted(need, key=repr)[0]
        best, gain = None, -1
        for _ in range(300):
            row = {k: dims[k][rng.integers(len(dims[k]))] for k in names}
            row[first[0]], row[first[2]] = first[1], first[3]
            if not ok(row):
                continue
            g = sum((a, row[a], b, row[b]) in need for a, b in itertools.combinations(names, 2))
            if g > gain:
                best, gain = row, g
        if best is None:                                  # (no acceptable row holds this pair of values)
            need.discard(first)
            continue
        for a, b in itertools.combinations(names, 2):
            need.discard((a, best[a], b, best[b]))
        rows.append(best)
    return rows


def matrix_runs(ws):
    dims = dict(transport=["p2p", "sendrecv", "auto"], mode=["block", "cyclic"], gather=["full", "summaries"], dst=[0, ws - 1],
                pb=[1, 7, 2048], overlap=[True, False], stage=["F", "pose", "tracks_inlier", "tracks_inlier_h", "tracks_all"],
                mutual=[False, True], tight_cap=[False, True])

    def ok(row):
        return row["gather"] == "full" or (not row["stage"].startswith("tracks") and not row["tight_cap"])
    return [Run(f"matrix {k + 1}", **row) for k, row in enumerate(pairwise(dims, ok))]


def small_lists(job, ws):
    """Index arrays into the ragged job's pair list: P = 0, 1, ws - 1, ws + 1, and 3 ws pairs whose block on rank 1 (pairs
    3-5) holds pairs with an empty image only (zero matches) between pairs of dense views."""
    pl = job.pairs.tolist()
    dense = [k for k, (i, j) in enumerate(pl) if i != j and i < 7 and j < 7]
    zero = [k for k, (i, j) in enumerate(pl) if i in job.roles["empty"] or j in job.roles["empty"]]
    return {"P = 0": np.zeros(0, np.int64), "P = 1": np.array([dense[0]]), "P = ws - 1": np.array(dense[1: ws]),
            "P = ws + 1": np.array(dense[ws: 2 * ws + 1]),
            "zero rows on rank 1": np.array(dense[:3] + zero[:3] + dense[3: 3 * ws - 3])}


def upload_cases(ws):
    """name -> (n_img, max_images) of the sharded uploads: ceil(n_img / ws) images per rank."""
    per = lambda n: -(-n // ws)  # noqa: E731
    return {"upload, n_img % ws != 0": (2 * ws + 1, ws * per(2 * ws + 1)),
            "upload, fewer images than ranks": (ws - 1, ws),
            "upload, spare bank slots": (ws + 1, ws * per(ws + 1) + 5)}


def upload_scene(n_img):
    return synth.make_scene(n_img, UP_FEATS, seed=500 + n_img)


def upload_pairs(n_img):
    return synth.exhaustive_pairs(n_img) if n_img > 1 else np.zeros((1, 2), np.int32)


def plan_runs(ws, job):
    """(Run, index array into the job's pairs or None = the run's own pair list) in the order one spawn runs them."""
    first = Run("first", transport="auto", mode="block", dst=0, pb=7, stage="pose")
    small = small_lists(job, ws)
    every = np.arange(len(job.pairs))
    runs = [(replace(first, name=f"first, call {k + 1} of 3"), every) for k in range(3)]
    runs += [(replace(first, name="first, P = ws + 1 (regions evicted)"), small["P = ws + 1"]),
             (replace(first, name="first, dst = ws - 1 (regions evicted)", dst=ws - 1), every),
             (replace(first, name="first, again"), every)]
    runs += [(r, every) for r in matrix_runs(ws)]
    runs += [(Run("P = 0", dst=ws - 1, stage="tracks_inlier"), small["P = 0"]),
             (Run("P = 1", mode="cyclic", transport="sendrecv", stage="pose"), small["P = 1"]),
             (Run("P = ws - 1", transport="p2p", dst=ws - 1, stage="tracks_inlier_h"), small["P = ws - 1"]),
             (Run("P = ws + 1, summaries", gather="summaries", dst=ws - 1, stage="pose"), small["P = ws + 1"]),
             (Run("P = ws + 1", pb=1, stage="tracks_all"), small["P = ws + 1"]),
             (Run("zero rows on rank 1", transport="p2p", pb=1, stage="pose"), small["zero rows on rank 1"]),
             (Run("zero rows on rank 1, tight cap", transport="sendrecv", dst=ws - 1, tight_cap=True), small["zero rows on rank 1"])]
    for k, name in enumerate(upload_cases(ws)):
        runs.append((Run(name, kind="upload", job=name, dst=(ws - 1) * (k % 2), pb=7), None))
    runs.append((Run("end-to-end arm", kind="e2e", job="upload, n_img % ws != 0", pb=bench.E2E_PAIR_BATCH), None))
    if ws == LARGEST:
        runs.append((Run("bench job configs[2]", job="bench", pb=bench.SHARD_PAIR_BATCH), None))
    return runs


def bench_job():
    wl = bench.WORKLOADS["c3"]
    sc = synth.make_scene(wl["n_images"], bench.N_FEATS, seed=wl["seed"])
    return sc, synth_pairs_blocked(wl["n_images"])


def synth_pairs_blocked(n):
    from sfm_b200.pairs import blocked_exhaustive_pairs

    return blocked_exhaustive_pairs(n, bench.PAIR_BLOCK)


# ====================================================================================================== host copies

def host_result(out):
    """What ``dst`` holds after a job, on the host: per-pair arrays, ``row_start``, the row arrays compacted in pair order
    (pair p's rows read at row_start[p] : row_start[p] + n_matches[p], indices clipped to the region), the tracks."""
    h = {}
    for k, v in out.items():
        if k == "tracks":
            h.update({f"tracks.{kk}": np.asarray(vv) for kk, vv in v.to_host().items()})
        elif k in ROW_KEYS:
            continue
        elif isinstance(v, torch.Tensor):
            h[k] = v.cpu().numpy()
        else:
            h[k] = np.asarray(v)
    if "row_start" in h:
        n = np.maximum(h["n_matches"].astype(np.int64), 0)
        idx = np.repeat(h["row_start"], n) + np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n)
        for k in ROW_KEYS:
            if k in out:
                full = out[k]
                ix = torch.from_numpy(np.clip(idx, 0, len(full) - 1)).to(full.device)
                h[k] = full.index_select(0, ix).cpu().numpy()
    return h


def region_is_new(bank):
    """1 when the job that just ran created the bank's cached region pair (the previous one was evicted), 0 otherwise."""
    regs = list(bank.__dict__.get("_gather_regions", {}).values())
    if not regs:
        return 0
    new = not getattr(regs[0], "_seen_by_test", False)
    regs[0]._seen_by_test = True
    return int(new)


# ====================================================================================================== the comparison

class Where:
    """Names the owner of a global pair: the rank and the position in its block."""

    def __init__(self, lay, ids=None):
        self.rank = np.zeros(lay.n_total, np.int64)
        self.pos = np.zeros(lay.n_total, np.int64)
        for r, own in enumerate(lay.owned):
            self.rank[own], self.pos[own] = r, np.arange(len(own))
        self.ids = ids                   # global pair of each compared entry (None: the entries are the global pairs)

    def __call__(self, p):
        g = p if self.ids is None else int(self.ids[p])
        return f"= global pair {g}, owned by rank {self.rank[g]} at position {self.pos[g]} of its block"


def expected_row_start(lay, n_matches, cap):
    """Rank r's rows lie in its slice (slices of sizes[r] * cap rows back to back in rank order), in its processing order."""
    base = np.concatenate([[0], np.cumsum([n * cap for n in lay.sizes])]).astype(np.int64)
    start = np.zeros(lay.n_total, np.int64)
    for r, own in enumerate(lay.owned):
        n = np.asarray(n_matches, np.int64)[own]
        start[own] = base[r] + np.cumsum(n) - n
    return start


def check_gathered(label, got, want, lay, run, cap, where=None, ids=None):
    """``got`` (host_result of dst) against the reference ``want`` of the whole job; returns the rows compared."""
    where = where or Where(lay)
    P = lay.n_total
    assert np.array_equal(got["pairs"], want["pairs"]) if "pairs" in got else run.gather == "summaries", f"{label}: pairs"
    rows = [k for k in ROW_KEYS if k in want] if run.gather == "full" else []
    assert set(got) - {"pairs", "transport", "row_start"} - {k for k in got if k.startswith("tracks.")} == \
        {k for k in PAIR_KEYS if k in want} | set(rows), f"{label}: gathered arrays {sorted(got)}"
    got = dict(got)
    got["offsets"] = np.concatenate([[0], np.cumsum(got["n_matches"].astype(np.int64))])
    compare(label, got, want, None, P, rows=rows or None, where=where)
    if rows:
        exp = expected_row_start(lay, want["n_matches"], cap)
        bad = np.nonzero(got["row_start"] != exp)[0]
        if len(bad):
            p = int(bad[0])
            raise AssertionError(f"{label}: pair {p} {where(p)}: row_start {got['row_start'][p]}, its rank's slice puts it at {exp[p]}")
    return len(want["matches"]) if rows else 0


def check_tracks(label, got, want, run, n_images):
    st = STAGES[run.stage]
    if "tracks" not in st:
        return
    h = {k[len("tracks."):]: (v if v.ndim else v.item()) for k, v in got.items() if k.startswith("tracks.")}
    twant = to.build_tracks_host(want, n_images, A_FEATS, flags=st["tracks"], min_length=st.get("min_length", 2),
                                 keep_conflicts=st.get("keep_conflicts", False))
    compare_tracks(label, h, twant)


# ====================================================================================================== the spawned ranks

def spawn(target, ws, args, timeout):
    """Start ``ws`` processes ``target(rank, ws, *args, q)``; errors come back through ``q``.  On an error, a failed rank or
    the timeout every live rank is killed; every rank is joined.  Returns the error messages."""
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=target, args=(r, ws) + tuple(args) + (q,)) for r in range(ws)]
    for p in procs:
        p.start()
    errors, t0 = [], time.time()
    try:
        while any(p.is_alive() for p in procs) and time.time() - t0 < timeout:
            try:
                errors.append(q.get(timeout=1))
            except _queue.Empty:
                pass
            if errors or any(p.exitcode not in (None, 0) for p in procs):
                break
    finally:
        end = time.time() + 15                              # ranks whose peer failed usually fail too: let them report
        for p in procs:
            p.join(max(0.0, end - time.time()))
        for p in procs:                                     # (only ranks that hang are still alive)
            if p.is_alive():
                p.kill()
        for p in procs:
            p.join(60)
            if p.is_alive():
                p.kill()
                p.join()
    while True:
        try:
            errors.append(q.get_nowait())
        except _queue.Empty:
            break
    if not errors and any(p.exitcode != 0 for p in procs):
        errors.append(f"exit codes {[p.exitcode for p in procs]} (timeout {timeout} s)")
    return errors


def _nccl_worker(rank, ws, port_, job, specs, out_dir, q):
    import faulthandler
    import traceback

    faulthandler.dump_traceback_later(900, exit=True)                   # a hung collective shows where, and ends the rank
    try:
        _nccl_worker_body(rank, ws, port_, job, specs, out_dir)
    except Exception:
        q.put(f"rank {rank}: {traceback.format_exc()}")
        raise
    finally:
        faulthandler.cancel_dump_traceback_later()


def _nccl_worker_body(rank, ws, port_, job, specs, out_dir):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    import sfm_b200
    from sfm_b200 import dist as sdist

    banks = {}

    def broadcast_bank(name, n_img, feats, fill):
        if name not in banks:
            banks[name] = sfm_b200.DescriptorBank(n_img, feats, device=dev)
            if rank == 0:
                fill(banks[name])
            sdist.broadcast_bank(banks[name], src=0)
        return banks[name]

    def save(k, arrays):
        np.savez(os.path.join(out_dir, f"{k}_r{rank}.npz"), **arrays)

    for k, (run, pairs, cap) in enumerate(specs):
        if run.kind == "sharded":
            if run.job == "bench":
                sc, _ = bench_job()
                n_img = len(sc.desc)
                bank = broadcast_bank("bench", -(-n_img // ws) * ws, bench.N_FEATS, lambda b: b.put(0, sc.desc, xy=sc.xy))
                del sc
            else:
                bank = broadcast_bank("a", len(job.images), A_FEATS, lambda b: put_job(b, job))
            ev = {}
            out, _ = sdist.match_and_verify_sharded(bank, pairs, events=ev, **run.kwargs(job.K, cap))
            h = host_result(out) if out is not None else {}                 # before the next job: the rows are a region's view
            save(k, dict(h, _rows_pushed=np.int64(ev["rows_pushed"]), _region_new=np.int64(region_is_new(bank))))
        elif run.kind == "upload":
            n_img, max_images = upload_cases(ws)[run.job]
            sc = upload_scene(n_img)
            bank = sfm_b200.DescriptorBank(max_images, UP_FEATS, device=dev)
            sdist.upload_bank_sharded(bank, sc.desc, sc.xy)
            one = sfm_b200.DescriptorBank(max_images, UP_FEATS, device=dev)
            one.put(0, sc.desc, xy=sc.xy)
            torch.cuda.synchronize()
            same = {}
            for name in ("desc", "ext", "norm", "xy"):
                b = bank.section(name).numel() // max_images * n_img
                same[name] = bool(torch.equal(bank.section(name)[:b], one.section(name)[:b]))
            same["counts"] = bool(torch.equal(bank.counts[:n_img], one.counts[:n_img]))
            same["counts_host"] = np.array_equal(bank.counts_host(), one.counts_host()) and bank.n_images == n_img
            banks[run.job] = bank
            ev = {}
            out, _ = sdist.match_and_verify_sharded(bank, pairs, events=ev, **run.kwargs(None, None))
            h = host_result(out) if out is not None else {}
            save(k, dict(h, _rows_pushed=np.int64(ev["rows_pushed"]), _region_new=np.int64(region_is_new(bank)),
                         _same=np.array([same[n] for n in sorted(same)]), _same_names=np.array(sorted(same))))
        else:                                                              # bench.py's end-to-end arm on an uploaded bank
            n_img, _ = upload_cases(ws)[run.job]
            sc = upload_scene(n_img)
            bank = banks[run.job]
            sdist.upload_bank_sharded(bank, torch.from_numpy(sc.desc).pin_memory(), torch.from_numpy(sc.xy).pin_memory())
            mine = sdist.layout(len(pairs), ws, "block").owned[rank]
            res = sfm_b200.match_and_verify(bank, pairs[mine], ratio=bench.RATIO, pair_batch=run.pb, pair_ids=mine, fetch="view",
                                            **bench.RANSAC)
            save(k, {kk: np.array(v) for kk, v in res.to_host().items()})
    dist.barrier()
    for bank in banks.values():
        for reg in bank.__dict__.get("_gather_regions", {}).values():
            reg.close()
    dist.destroy_process_group()


# ====================================================================================================== reference side

@pytest.fixture(scope="module")
def job_a():
    return ragged_job()


@pytest.fixture(scope="module")
def ref_a(job_a):
    return Reference(job_a.images, job_a.K, "cuda")


REPORT: dict = {}            # world size -> {"runs", "pairs", "rows", "paths"}
PATHS: dict = {}             # path -> set of world sizes that reached it


def reach(ws, path):
    PATHS.setdefault(path, set()).add(ws)
    REPORT.setdefault(ws, {"runs": 0, "pairs": 0, "rows": 0, "paths": set()})["paths"].add(path)


def count(ws, pairs, rows):
    r = REPORT.setdefault(ws, {"runs": 0, "pairs": 0, "rows": 0, "paths": set()})
    r["runs"] += 1
    r["pairs"] += pairs
    r["rows"] += rows


def specs_for(ws, job, ref):
    """(Run, pairs, rows_per_pair_cap) of every run, and the reference of every run (None for the bench job)."""
    specs, wants = [], []
    for run, idx in plan_runs(ws, job):
        if run.kind in ("upload", "e2e"):
            n_img, _ = upload_cases(ws)[run.job]
            pairs, want = upload_pairs(n_img), None
        elif run.job == "bench":
            pairs, want = None, None
        else:
            pairs = job.pairs[idx]
            want = ref.job(pairs, np.arange(len(pairs)), run.cfg())
        cap = max(int(want["n_matches"].max()), 1) if run.tight_cap and len(pairs) else None
        specs.append((run, pairs if pairs is not None else synth_pairs_blocked(bench.WORKLOADS["c3"]["n_images"]), cap))
        wants.append(want)
    return specs, wants


def load(out_dir, k, rank):
    with np.load(os.path.join(out_dir, f"{k}_r{rank}.npz")) as z:
        return {n: z[n] for n in z.files}


def check_run(ws, k, run, pairs, cap, want, out_dir, ref_up, regions_used, job):
    """Every check of run k of world size ws.  ``regions_used``: the banks on which a job with gather="full" has run."""
    from sfm_b200.dist import layout

    label = f"world size {ws}, run {k} ({run.name})"
    P = len(pairs)
    mode = run.mode if run.kind != "e2e" else "block"
    lay = layout(P, ws, mode)
    if run.kind == "e2e":
        want = ref_up.job(pairs, np.arange(P), run.cfg())
        got = {n: np.zeros((P,) + want[n].shape[1:], want[n].dtype) for n in PAIR_KEYS if n in want}
        got.update(pairs=pairs, offsets=np.zeros(P + 1, np.int64))
        rows = {n: [] for n in ("matches", "inlier")}
        for r, own in enumerate(lay.owned):                   # assembled by partition: rank r's block is global pairs owned[r]
            h = load(out_dir, k, r)
            assert np.array_equal(h["pairs"], pairs[own]), (label, r)
            for n in got:
                if n in PAIR_KEYS:
                    got[n][own] = h[n]
            for n in rows:
                rows[n].append(h[n])
        for n in rows:                                        # block order is global order
            got[n] = np.concatenate(rows[n])
        got["offsets"][1:] = np.cumsum(got["n_matches"])
        compare(label, got, want, None, P, rows=["matches", "inlier"], where=Where(lay))
        count(ws, P, len(want["matches"]))
        return
    if run.kind == "upload":
        n_img, _ = upload_cases(ws)[run.job]
        per = -(-n_img // ws)
        for r in range(ws):
            h = load(out_dir, k, r)
            for name, ok in zip(h["_same_names"], h["_same"]):
                assert ok, f"{label}: rank {r}: the packed {name} differ from one put of the same images"
            if r * per >= n_img:
                reach(ws, "a rank that owned no images in the upload")
        want = ref_up.job(pairs, np.arange(P), run.cfg())
    got = load(out_dir, k, run.dst)
    rows_pushed = [int(load(out_dir, k, r)["_rows_pushed"]) for r in range(ws)]
    region_new = int(got["_region_new"])
    got = {n: v for n, v in got.items() if not n.startswith("_")}
    cap_rows = cap if cap is not None else (A_FEATS if run.job == "a" else UP_FEATS)
    if run.gather == "full":
        assert str(got["transport"]) == ("sendrecv" if run.transport == "sendrecv" else "p2p"), (label, got["transport"])
        if str(got["transport"]) == "p2p":
            reach(ws, "real p2p")
        for r, own in enumerate(lay.owned):
            assert rows_pushed[r] == int(want["n_matches"][own].sum()), f"{label}: rank {r} pushed {rows_pushed[r]} rows"
        if run.name.startswith("first, call") and not run.name.startswith("first, call 1"):
            assert not region_new, f"{label}: the same call did not reuse the cached region pair"
        if region_new and run.job in regions_used:
            reach(ws, "region eviction")
        regions_used.add(run.job)
    rows = check_gathered(label, got, want, lay, run, cap_rows)
    check_tracks(label, got, want, run, len(job.images))
    count(ws, P, rows)
    if run.dst != 0:
        reach(ws, "dst != 0")
    for r, own in enumerate(lay.owned):
        if len(own) == 0 and P:
            reach(ws, "an empty rank")
        elif len(own) and want["n_matches"][own].sum() == 0:
            reach(ws, "a rank with zero rows")
    if run.job == "a" and run.gather == "full":
        for p in np.nonzero((pairs == np.asarray(job.wide)).all(1))[0]:
            reach(ws, f"the wide pair in the block of rank {Where(lay).rank[p]}")


def check_bench(ws, k, run, pairs, out_dir):
    """configs[2] at the largest world size: the reference on the first and last 8 pairs of every rank's block and 400
    seeded pairs; all 19,900 pairs equal a world-size-1 run and lie in their rank's slice in processing order."""
    import sfm_b200
    from sfm_b200 import dist as sdist
    from sfm_b200.dist import layout

    label = f"world size {ws}, run {k} ({run.name})"
    P = len(pairs)
    lay = layout(P, ws, "block")
    where = Where(lay)
    got = {n: v for n, v in load(out_dir, k, 0).items() if not n.startswith("_")}
    sc, _ = bench_job()
    ref = Reference([(sc.desc[i], sc.xy[i]) for i in range(len(sc.desc))], synth.K_INTR, "cuda")
    sample = set(np.random.default_rng(2024).choice(P, 400, replace=False).tolist())
    for own in lay.owned:
        sample |= set(own[:8].tolist()) | set(own[-8:].tolist())
    sample = np.array(sorted(sample))
    want = ref.job(pairs[sample], sample, run.cfg())
    sub = {n: got[n][sample] for n in PAIR_KEYS if n in got}
    off = np.concatenate([[0], np.cumsum(got["n_matches"].astype(np.int64))])
    sel = np.concatenate([np.arange(off[p], off[p + 1]) for p in sample])
    sub.update(pairs=pairs[sample], matches=got["matches"][sel], inlier=got["inlier"][sel])
    sub["offsets"] = np.concatenate([[0], np.cumsum(sub["n_matches"].astype(np.int64))])
    compare(label + " [reference sample]", sub, want, None, len(sample), rows=["matches", "inlier"], where=Where(lay, sample))
    # all pairs: a world-size-1 run of the same call in this process (no process group)
    bank = sfm_b200.DescriptorBank(len(sc.desc), bench.N_FEATS)
    bank.put(0, sc.desc, xy=sc.xy)
    out1, _ = sdist.match_and_verify_sharded(bank, pairs, **run.kwargs(None, None))
    one = host_result(out1)
    del out1, bank
    for n in ("n_matches", "F", "n_inliers", "iters", "matches", "inlier"):
        if got[n].shape == one[n].shape and np.array_equal(_bits(got[n]), _bits(one[n])):
            continue
        assert len(got[n]) == len(one[n]), f"{label}: {n}: {len(got[n])} entries, the world-size-1 run has {len(one[n])}"
        bad = np.nonzero((_bits(got[n]) != _bits(one[n])).any(1))[0]
        if len(bad):
            r = int(bad[0])
            p = r if n not in ROW_KEYS else int(np.searchsorted(off, r, side="right") - 1)
            raise AssertionError(f"{label}: pair {p} {where(p)}: {n} differs from the world-size-1 run")
    exp = expected_row_start(lay, got["n_matches"], bench.N_FEATS)
    bad = np.nonzero(got["row_start"] != exp)[0]
    assert not len(bad), f"{label}: pair {bad[0]} {where(int(bad[0]))}: row_start {got['row_start'][bad[0]]}, its slice puts it at {exp[bad[0]]}"
    count(ws, len(sample), len(want["matches"]))
    print(f"{label}: reference on {len(sample)} pairs ({len(want['matches'])} rows); all {P} pairs and {len(got['matches'])} rows "
          f"equal the world-size-1 run")


RAN: list = []


@pytest.mark.gpu
@pytest.mark.parametrize("ws", WORLD_SIZES)
def test_sharded_equals_the_reference(ws, tmp_path, request):
    if N_GPUS < ws:
        pytest.skip(f"world size {ws} needs {ws} GPUs: {N_GPUS} visible, {ws - N_GPUS} missing")
    job_a, ref_a = request.getfixturevalue("job_a"), request.getfixturevalue("ref_a")
    t0 = time.perf_counter()
    specs, wants = specs_for(ws, job_a, ref_a)
    errors = spawn(_nccl_worker, ws, (port(ws), job_a, specs, str(tmp_path)), timeout=1200)
    assert not errors, "\n".join(map(str, errors))
    t1 = time.perf_counter()
    refs_up, regions_used = {}, set()
    for k, ((run, pairs, cap), want) in enumerate(zip(specs, wants)):
        if run.job == "bench":
            check_bench(ws, k, run, pairs, str(tmp_path))
            continue
        ref_up = None
        if run.kind != "sharded":
            if run.job not in refs_up:
                sc = upload_scene(upload_cases(ws)[run.job][0])
                refs_up[run.job] = Reference([(sc.desc[i], sc.xy[i]) for i in range(len(sc.desc))], synth.K_INTR, "cuda")
            ref_up = refs_up[run.job]
        check_run(ws, k, run, pairs, cap, want, str(tmp_path), ref_up, regions_used, job_a)
    RAN.append(ws)
    rep = REPORT[ws]
    print(f"\nworld size {ws}: {rep['runs']} runs, {rep['pairs']} pairs and {rep['rows']} rows compared; ranks {t1 - t0:.1f} s, "
          f"checks {time.perf_counter() - t1:.1f} s; paths {sorted(rep['paths'])}")


@gpu_test
def test_every_path_was_reached():
    """The world sizes that ran reached every path (the module's tests run in order)."""
    if not RAN:
        pytest.skip(f"no world size above 1 ran ({N_GPUS} GPU visible)")
    for p in sorted(PATHS):
        print(f"{p}: world sizes {sorted(PATHS[p])}")
    need = {"an empty rank", "a rank with zero rows", "dst != 0", "real p2p", "region eviction",
            "a rank that owned no images in the upload"}
    assert need <= set(PATHS), sorted(need - set(PATHS))
    assert any(p.startswith("the wide pair in the block of rank") for p in PATHS)


# ====================================================================================================== world size 1, in process

class Local:
    """The ragged job's bank in this process, with no process group: match_and_verify_sharded at world size 1."""

    def __init__(self, job, ref):
        import sfm_b200
        from sfm_b200 import dist as sdist

        self.sdist, self.job, self.ref = sdist, job, ref
        self.bank = sfm_b200.DescriptorBank(len(job.images), A_FEATS)
        put_job(self.bank, job)

    def run(self, run, pairs=None, cap=None, want=None):
        from sfm_b200.dist import layout

        pairs = self.job.pairs if pairs is None else pairs
        P = len(pairs)
        want = want or self.ref.job(pairs, np.arange(P), run.cfg())
        ev = {}
        out, _ = self.sdist.match_and_verify_sharded(self.bank, pairs, events=ev, **run.kwargs(self.job.K, cap))
        got = host_result(out)
        label = f"world size 1 ({run.name})"
        if run.gather == "full":
            assert str(got["transport"]) == "sendrecv", (label, got["transport"])
            assert ev["rows_pushed"] == int(want["n_matches"].sum()), label
        rows = check_gathered(label, got, want, layout(P, 1, run.mode), run, cap or A_FEATS)
        check_tracks(label, got, want, run, len(self.job.images))
        print(f"{label}: {P} pairs, {rows} rows")
        return want


@pytest.fixture(scope="module")
def local(job_a, ref_a):
    return Local(job_a, ref_a)


@gpu_test
def test_world_size_1_gathers_and_tracks(local):
    """Both gathers, ``transport="p2p"`` (sendrecv at one rank), both partitions and tracks with every flag."""
    local.run(Run("full, p2p", transport="p2p", stage="pose"))
    local.run(Run("summaries, cyclic", gather="summaries", mode="cyclic", stage="pose", dst=0))
    for stage in ("tracks_inlier", "tracks_inlier_h", "tracks_in_front", "tracks_all"):
        local.run(Run(f"{stage}, pair_batch 7", stage=stage, pb=7))
    local.run(Run("mutual, no overlap, tight cap", mutual=True, overlap=False, tight_cap=True),
              cap=int(local.ref.job(local.job.pairs, np.arange(len(local.job.pairs)), Cfg(mutual=True))["n_matches"].max()))
    for name, idx in small_lists(local.job, 2).items():
        local.run(Run(name, stage="tracks_inlier", pb=1), pairs=local.job.pairs[idx])


@gpu_test
def test_world_size_1_row_sink_overflow(local):
    """The sink holds P * rows_per_pair_cap rows per rank: ceil(total / P) is the smallest cap that holds the job, one less
    overflows with SfmError, and the next job on the same bank still equals the reference."""
    from sfm_b200._lib import SfmError

    job = local.job
    P = len(job.pairs)
    run = Run("cap = ceil(rows / P)", pb=7)
    want = local.ref.job(job.pairs, np.arange(P), run.cfg())
    cap = -(-int(want["n_matches"].sum()) // P)
    assert cap < int(want["n_matches"].max())                  # a per-pair cap this small would not hold the wide pair
    local.run(run, cap=cap, want=want)
    with pytest.raises(SfmError, match="row sink overflow"):
        local.run(replace(run, name="cap = ceil(rows / P) - 1"), cap=cap - 1, want=want)
    torch.cuda.synchronize()
    local.run(replace(run, name="after the overflow"), cap=cap, want=want)
    local.run(replace(run, name="after the overflow, default cap", stage="tracks_inlier"))


# ====================================================================================================== CPU, gloo

@pytest.fixture(scope="module")
def counts_a(job_a):
    """n_matches of the ragged job's reference (GEMMs on the CPU)."""
    ref = Reference(job_a.images, job_a.K, "cpu")
    return np.array([len(ref.matches(int(i), int(j))[0]) for i, j in job_a.pairs], np.int64)


def gloo_cases(ws, job, counts):
    small = small_lists(job, ws)
    cases = [("ragged job, block, dst 0", counts, "block", 0), ("ragged job, cyclic, dst ws - 1", counts, "cyclic", ws - 1),
             ("ragged job, block, dst ws - 1", counts, "block", ws - 1), ("ragged job, cyclic, dst 0", counts, "cyclic", 0)]
    for name, idx in small.items():
        for mode, dst in (("block", ws - 1), ("cyclic", 0)):
            cases.append((f"{name}, {mode}, dst {dst}", counts[idx], mode, dst))
    return cases


def _payload(p, n):
    """Rows of global pair p: matches[k] = (p, k, 1000 p + k), inlier[k] = (p + k) & 1."""
    k = np.arange(n)
    return np.stack([np.full(n, p), k, 1000 * p + k], 1).astype(np.int32), ((p + k) & 1).astype(np.uint8)


def _summaries(idx, counts, stages):
    from types import SimpleNamespace

    g = torch.as_tensor(np.asarray(idx, np.int64))
    n = len(idx)
    F = g.to(torch.float64).view(n, 1, 1) + torch.arange(9, dtype=torch.float64).view(1, 3, 3) / 16.0
    r = SimpleNamespace(n_matches=torch.as_tensor(np.asarray(counts, np.int64)[idx].astype(np.int32)),
                        n_inliers=(g % 3).to(torch.int32), iters=(g % 11).to(torch.int32), F=F)
    if stages:
        r.H, r.n_inliers_h = F + 0.5, (g % 2).to(torch.int32)
        r.R, r.t, r.n_pose = F * 2.0, torch.stack([g.to(torch.float64), -g.to(torch.float64), g.to(torch.float64) / 4], 1) \
            if n else torch.zeros((0, 3), dtype=torch.float64), (g % 4).to(torch.int32)
    return r


def _gloo_worker(rank, ws, port_, cases, q):
    import faulthandler
    import traceback

    faulthandler.dump_traceback_later(240, exit=True)
    try:
        _gloo_worker_body(rank, ws, port_, cases, q)
    except Exception:
        q.put(f"rank {rank}: {traceback.format_exc()}")
        raise
    finally:
        faulthandler.cancel_dump_traceback_later()


def _gloo_worker_body(rank, ws, port_, cases, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_)
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    from sfm_b200.dist import GatherRegion, gather_summaries, layout

    cpu = torch.device("cpu")
    for name, counts, mode, dst in cases:
        label = f"world size {ws}, {name}"
        P = len(counts)
        lay = layout(P, ws, mode)
        mine = lay.owned[rank]
        where = Where(lay)
        stages = "cyclic" in name
        summ = gather_summaries(_summaries(mine, counts, stages), mine, P, dst, mode=mode, homography=stages, pose=stages)
        cap = max(int(np.max(counts)) if P else 1, 1)
        reg = GatherRegion([n * cap for n in lay.sizes], ("matches", "inlier"), dst, cpu, "sendrecv")
        rows = 0
        for p in mine:
            m, f = _payload(int(p), int(counts[p]))
            reg.local["matches"][rows: rows + len(m)] = torch.from_numpy(m)
            reg.local["inlier"][rows: rows + len(m)] = torch.from_numpy(f)
            rows += len(m)
        if rank == dst:                                   # (before the exchange, which takes its sizes from n_matches)
            want = _summaries(np.arange(P), counts, stages)
            for k in ("n_matches", "n_inliers", "iters", "F") + (("H", "n_inliers_h", "R", "t", "n_pose") if stages else ()):
                g, w = summ[k].numpy(), getattr(want, k).numpy()
                assert g.shape == w.shape and g.dtype == w.dtype, (label, k, g.shape, g.dtype)
                bad = np.nonzero((_bits(g) != _bits(w)).any(1))[0]
                assert not len(bad), f"{label}: pair {bad[0]} {where(int(bad[0]))}: {k} = {g[bad[0]].tolist()}, sent {w[bad[0]].tolist()}"
        reg.exchange(rows, summ["n_matches"] if rank == dst else None, lay)
        if rank == dst:
            start = reg.row_starts(summ["n_matches"], lay).numpy()
            exp = expected_row_start(lay, counts, cap)
            bad = np.nonzero(start != exp)[0]
            assert not len(bad), f"{label}: pair {bad[0]} {where(int(bad[0]))}: row_start {start[bad[0]]}, its rank's slice puts it at {exp[bad[0]]}"
            for p in range(P):
                m, f = _payload(p, int(counts[p]))
                s = int(start[p])
                assert np.array_equal(reg.full["matches"][s: s + len(m)].numpy(), m) and \
                    np.array_equal(reg.full["inlier"][s: s + len(m)].numpy(), f), f"{label}: pair {p} {where(p)}: rows differ"
        else:
            assert summ is None, label
        reg.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("ws", [2, 3, 4, 5, 6, 7, 8])
def test_gloo_gather_with_the_ragged_jobs_row_counts(ws, job_a, counts_a):
    """gather_summaries, GatherRegion (sendrecv) and row_starts on world sizes 2 to 8, with the per-pair row counts of the
    ragged job's reference (many zeros, one pair with 5,498 rows), dst in {0, ws - 1}, empty ranks and a rank whose pairs
    all have zero rows."""
    cases = gloo_cases(ws, job_a, counts_a)
    errors = spawn(_gloo_worker, ws, (port(8 + ws), cases), timeout=300)
    assert not errors, "\n".join(map(str, errors))
