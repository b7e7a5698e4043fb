"""Pair-sharded multi-GPU execution (one process per GPU, torch.distributed).

The reference's pair loop (code/pipeline.py:38-47) is embarrassingly parallel by image pair, so the only communication
is (1) one NCCL broadcast of the packed descriptor bank from rank 0 and (2) the gather of every pair's results on rank 0
-- the distributed form of ``pair_matches.append(Pair(...))`` (code/pipeline.py:43-47; SURVEY.md §8e):

* per-pair summaries (n_matches, n_inliers, iters, F, optional H / R / t ...) travel as ONE fixed-size ``dist.gather``
  (the partition sizes are known on every rank, so there is no size exchange and no host synchronisation);
* the variable-length part (packed match rows, inlier flags) is PUSHED by each rank into its slice of a region of the
  gathering rank's HBM (``GatherRegion``): with the ``p2p`` transport the region is mapped into every process
  (``sfm_peer_open``) and each batch's rows go over NVLink with copy-engine copies while the SMs sweep the next batch;
  the summary gather that follows is also the completion signal.  The ``sendrecv`` transport (grouped send/recv with the
  exact sizes taken from the gathered n_matches) is the portable form: it runs under gloo on CPU tensors
  (tests/test_dist_gloo.py) and is the fallback when peer mapping is unavailable.

No collective runs inside the compute phase, so there is nothing to fuse with a kernel.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch
import torch.distributed as dist

from .plan import OUTPUTS, RowSink, outputs
from .tracks import build_tracks_from_rows


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def partition(n_items: int, rank: int, world_size: int, mode: str = "block"):
    """Index array of the items rank ``rank`` owns.

    block : contiguous ceil(P/R) slices of the (i,j)-sorted pair list (keeps image i hot in L2)
    cyclic: items rank, rank+R, ... (balances RANSAC cost when match counts vary along the list)
    """
    if mode == "block":
        per = -(-n_items // world_size) if n_items else 0
        return np.arange(min(rank * per, n_items), min((rank + 1) * per, n_items))
    if mode == "cyclic":
        return np.arange(rank, n_items, world_size)
    raise ValueError(f"unknown partition mode {mode!r}")


class Layout:
    """Who owns which pair, as index arrays every rank can compute on its own: ``owned[r]`` (global pair indices of rank
    r, in its processing order), ``perm`` = their concatenation (rank-major order -> global index) and the row of the
    gathered [world * per, W] summary table each entry comes from."""

    def __init__(self, n_total: int, world_size: int, mode: str = "block"):
        self.n_total, self.ws, self.mode = int(n_total), int(world_size), mode
        self.owned = [partition(self.n_total, r, self.ws, mode) for r in range(self.ws)]
        self.sizes = [len(o) for o in self.owned]
        self.per = max(max(self.sizes), 1)
        self.perm = np.concatenate(self.owned).astype(np.int64) if self.n_total else np.zeros(0, np.int64)
        self.src_rows = np.concatenate([r * self.per + np.arange(n) for r, n in enumerate(self.sizes)]).astype(np.int64)
        self.rank_of = np.concatenate([np.full(n, r, np.int64) for r, n in enumerate(self.sizes)])
        self.first = np.concatenate([[0], np.cumsum(self.sizes)])[:-1].astype(np.int64)     # rank-major index of each rank's first pair
        self._dev = {}

    def on(self, dev):
        """The same index arrays as device tensors (cached per device)."""
        t = self._dev.get(dev)
        if t is None:
            as_t = lambda a: torch.as_tensor(a, dtype=torch.int64, device=dev)  # noqa: E731
            t = self._dev[dev] = {"perm": as_t(self.perm), "src_rows": as_t(self.src_rows), "rank_of": as_t(self.rank_of),
                                  "first": as_t(self.first)}
        return t


_LAYOUTS = {}


def layout(n_total: int, world_size: int, mode: str = "block") -> Layout:
    key = (int(n_total), int(world_size), mode)
    if key not in _LAYOUTS:
        if len(_LAYOUTS) > 16:
            _LAYOUTS.clear()
        _LAYOUTS[key] = Layout(*key)
    return _LAYOUTS[key]


def broadcast_bank(bank, src: int = 0):
    """Broadcast the packed bank storage (descriptors, K-extension, norms, xy, counts) from ``src``.
    Non-source ranks end up with a ready bank without running the pack kernel."""
    rank, ws = world()
    meta = torch.tensor([bank.n_images if rank == src else 0], dtype=torch.int64, device=bank.storage.device)
    if ws > 1:
        dist.broadcast(bank.storage, src=src)
        dist.broadcast(meta, src=src)
    if rank != src:
        n = int(meta.item())
        bank.mark_filled(n, bank.counts[:n].cpu().numpy())
    return bank


def upload_bank_sharded(bank, desc, xy=None):
    """Fill the bank of EVERY rank from host arrays that every rank holds (``desc`` uint8 [n_images, n, 128], ``xy`` float32
    [n_images, n, 2]; pinned torch tensors avoid a staging copy): rank r uploads and packs only images [r * per, (r + 1) * per),
    then the packed sections are all-gathered over NVLink in place.  Replaces N full uploads over PCIe (N x 223 MB per job at
    200 images) by N slices plus one NCCL all-gather of the packed bank.  The bank must have room for ``world * per`` images."""
    rank, ws = world()
    desc_t = desc if isinstance(desc, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(desc, np.uint8))
    xy_t = None if xy is None else (xy if isinstance(xy, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(xy, np.float32)))
    n_img = int(desc_t.shape[0])
    if ws == 1:
        bank.put(0, desc_t, xy=xy_t)
        return bank
    per = -(-n_img // ws)
    if ws * per > bank.max_images:
        raise ValueError(f"sharded upload of {n_img} images over {ws} ranks needs a bank for {ws * per} images (has {bank.max_images})")
    a, b = min(rank * per, n_img), min((rank + 1) * per, n_img)
    if b > a:
        bank.put(a, desc_t[a:b], xy=None if xy_t is None else xy_t[a:b])
    fs = bank.feat_stride
    per_image = {"desc": fs * bank.dim, "ext": (fs // 128) * 4096 if bank.metric == "l2" else 0, "norm": fs * 4, "xy": fs * 8, "count": 4}
    for name, bpi in per_image.items():
        if bpi == 0:
            continue
        sec = bank.section(name)[: ws * per * bpi]
        if rank * per >= n_img and name == "count":
            sec[rank * per * bpi: (rank + 1) * per * bpi].zero_()    # a rank without images contributes zero counts
        dist.all_gather_into_tensor(sec, sec[rank * per * bpi: (rank + 1) * per * bpi])
    counts = np.full(n_img, int(desc_t.shape[1]), np.int32)
    bank.mark_filled(n_img, counts)
    return bank


# ------------------------------------------------------------------------------------ per-pair summaries
def summary_columns(homography: bool = False, pose: bool = False):
    """Column layout of the float64 summary table, from the CALL parameters (not from what a rank happened to produce: a
    rank whose block is empty must contribute a tile of the same width as everybody else).  name -> (first column, width,
    dtype, trailing shape); column 0 is reserved."""
    cols, w = {}, 1
    for o in outputs(homography, pose):
        if o.per == "pair":
            cols[o.name] = (w, math.prod(o.shape), o.dtype, o.shape)
            w += math.prod(o.shape)
    return cols, w


def gather_summaries(res, order: np.ndarray, n_total: int, dst: int = 0, *, mode: str = "block", homography=None, pose=None):
    """Per-pair summaries of every rank on ``dst`` in global pair order with ONE ``dist.gather`` of a fixed-size float64
    [ceil(P/R), W] tile per rank (integers are exact in float64) and no host synchronisation anywhere: which tile row is
    which pair follows from ``partition()``, which every rank can evaluate.  ``homography`` / ``pose`` say whether the
    optional stages were requested (default: whether ``res`` carries them).  Returns a dict of device tensors on ``dst``,
    None elsewhere."""
    rank, ws = world()
    dev = res.n_matches.device
    if homography is None:
        homography = getattr(res, "H", None) is not None
    if pose is None:
        pose = getattr(res, "R", None) is not None
    lay = layout(n_total, ws, mode)
    n = len(order)
    if n != lay.sizes[rank] or (n and not np.array_equal(np.asarray(order), lay.owned[rank])):
        raise ValueError("order must be this rank's partition(n_total, rank, world_size, mode)")
    cols, w = summary_columns(homography, pose)
    tile = torch.zeros((lay.per, w), dtype=torch.float64, device=dev)
    for name, (c0, width, _, _) in cols.items():
        v = getattr(res, name, None)
        if v is None:
            if n:
                raise ValueError(f"{name!r} was requested in the summary but this rank's result does not carry it")
            continue
        tile[:n, c0: c0 + width] = v.to(torch.float64).reshape(n, width)
    if ws == 1:
        full = tile
    else:
        recv = torch.empty((ws, lay.per, w), dtype=torch.float64, device=dev) if rank == dst else None
        dist.gather(tile, list(recv.unbind(0)) if rank == dst else None, dst=dst)
        full = recv.view(ws * lay.per, w) if rank == dst else None
    if rank != dst:
        return None
    ix = lay.on(dev)
    rows = full.index_select(0, ix["src_rows"])                      # rank-major order
    out = {}
    for name, (c0, width, dt, shape) in cols.items():
        o = torch.empty((n_total,) + shape, dtype=dt, device=dev)
        o[ix["perm"]] = rows[:, c0: c0 + width].to(dt).reshape((-1,) + shape)
        out[name] = o
    return out


# ------------------------------------------------------------------------------------ packed rows
class _DevArray:
    """Minimal ``__cuda_array_interface__`` carrier: lets torch view memory this process got from sfm_peer_alloc."""

    def __init__(self, ptr: int, shape, typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2, "strides": None}


class GatherRegion:
    """Receive buffers on ``dst`` for the packed rows of every rank's pair block, and each rank's way into its slice.

    ``caps[r]`` = row capacity of rank r's slice (slices are laid out back to back in rank order), ``fields`` = names of the
    row arrays (``plan.RowSink.ROW_BYTES``).  After a job, rank r's rows occupy ``[base[r], base[r] + rows_r)`` of every
    array on ``dst``; ``row_starts()`` turns the gathered ``n_matches`` into each pair's first row.

    transport ``p2p``     : the arrays live in memory from ``sfm_peer_alloc`` on ``dst`` and are mapped into every other
                            process (CUDA IPC, same box); ``sink()`` points straight into the slice, nothing is left to do
                            after the job but the completion signal (the summary gather).
    transport ``sendrecv``: every rank fills a local staging array; ``exchange()`` moves exactly ``rows_r`` rows per rank
                            with grouped send/recv.  Runs on any backend and any device (gloo/CPU in the tests).
    ``auto`` tries ``p2p`` on CUDA under NCCL and falls back -- on ALL ranks together -- when mapping fails."""

    def __init__(self, caps, fields=("matches", "inlier"), dst: int = 0, device=None, transport: str = "auto"):
        self.rank, self.ws = world()
        self.dst, self.fields = int(dst), tuple(fields)
        self.caps = [int(c) for c in caps]
        if len(self.caps) != self.ws:
            raise ValueError("one capacity per rank")
        self.base = np.concatenate([[0], np.cumsum(self.caps)]).astype(np.int64)
        self.total_cap = int(self.base[-1])
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._peer_ptrs, self._owned_ptrs = {}, {}
        self.full, self.local = {}, {}
        want = transport
        if want == "auto":
            want = "p2p" if (self.device.type == "cuda" and self.ws > 1 and dist.get_backend() == "nccl") else "sendrecv"
        if want == "p2p" and self.ws > 1:
            ok = self._setup_p2p()
            flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                self._teardown_p2p()
                if transport == "p2p":
                    raise RuntimeError("GatherRegion: peer mapping failed on at least one rank: " + getattr(self, "_p2p_error", ""))
                want = "sendrecv"
        elif want == "p2p":
            want = "sendrecv"                                          # one rank: plain local arrays
        self.transport = want
        if want == "sendrecv":
            my_cap = max(self.caps[self.rank], 1)
            for name in self.fields:
                if self.rank == self.dst:
                    self.full[name] = OUTPUTS[name].empty(max(self.total_cap, 1), device=self.device)
                    b = int(self.base[self.rank])
                    self.local[name] = self.full[name][b: b + my_cap]
                else:
                    self.local[name] = OUTPUTS[name].empty(my_cap, device=self.device)
        self._sink = None
        self._fence = None

    # ---- p2p plumbing
    def _setup_p2p(self) -> bool:
        from . import _lib

        L = _lib.lib()
        dev_index = self.device.index or 0
        handles = [None]
        try:
            if self.rank == self.dst:
                hs = {}
                for name in self.fields:
                    rb = RowSink.ROW_BYTES[name]
                    ptr, h = C.c_void_p(), (C.c_uint8 * 64)()
                    _lib.check(L.sfm_peer_alloc(dev_index, max(self.total_cap, 1) * rb, C.byref(ptr), h), "sfm_peer_alloc")
                    self._owned_ptrs[name] = int(ptr.value)
                    hs[name] = bytes(h)
                handles = [hs]
        except Exception as e:                                        # the broadcast below must still be entered by every rank
            self._p2p_error = repr(e)
            handles = [None]
        dist.broadcast_object_list(handles, src=self.dst)
        if handles[0] is None:
            return False
        try:
            if self.rank == self.dst:
                for name in self.fields:
                    o = OUTPUTS[name]
                    arr = _DevArray(self._owned_ptrs[name], (max(self.total_cap, 1),) + o.shape, o.empty(0).numpy().dtype.str)
                    self.full[name] = torch.as_tensor(arr, device=self.device)
                    self._peer_ptrs[name] = self._owned_ptrs[name]
            else:
                for name in self.fields:
                    ptr = C.c_void_p()
                    buf = (C.c_uint8 * 64).from_buffer_copy(handles[0][name])
                    _lib.check(L.sfm_peer_open(dev_index, buf, C.byref(ptr)), "sfm_peer_open")
                    self._peer_ptrs[name] = int(ptr.value)
        except Exception as e:
            self._p2p_error = repr(e)
            return False
        return True

    def _teardown_p2p(self) -> None:
        from . import _lib

        L = _lib.lib()
        dev_index = self.device.index or 0
        self.full = {}
        for name, p in list(self._peer_ptrs.items()):
            if name not in self._owned_ptrs:
                L.sfm_peer_close(dev_index, C.c_void_p(p))
        for p in self._owned_ptrs.values():
            L.sfm_peer_free(dev_index, C.c_void_p(p))
        self._peer_ptrs, self._owned_ptrs = {}, {}

    def close(self) -> None:
        """Collective: nobody unmaps or frees while another rank may still be copying."""
        if self.ws > 1 and dist.is_initialized():
            if self.device.type == "cuda":
                torch.cuda.synchronize(self.device)
            dist.barrier()
        if self._peer_ptrs or self._owned_ptrs:
            self._teardown_p2p()

    # ---- use
    def sink(self) -> RowSink:
        """This rank's slice as a ``RowSink`` for ``match_and_verify(..., sink=...)`` (one per region, reset per job)."""
        if self._sink is None:
            b = int(self.base[self.rank])
            if self.transport == "p2p":
                f = {n: self._peer_ptrs[n] + b * RowSink.ROW_BYTES[n] for n in self.fields}
            else:
                f = {n: self.local[n].data_ptr() for n in self.fields}
            self._sink = RowSink(f, self.caps[self.rank])
        self._sink.reset()
        return self._sink

    def fence_issue(self) -> None:
        """Region reuse fence (p2p transport): no rank may overwrite its slice before ``dst`` has finished the work it had
        enqueued on the rows of the job that used this region.  One tiny all-reduce on a SIDE stream that first waits for the
        caller's stream.  Regions come in pairs (``get_regions``): the fence of a region is issued at the START of the job that
        uses its twin, a whole job before the rows that wait for it -- issued at the start of the job that needs it, the
        all-reduce kernel has to find room beside that job's persistent sweep, and single steps were seen to lose 20-120 ms
        there (profiles/r02_n2_per_rank_diag.log)."""
        if self.transport != "p2p" or self.ws == 1:
            return
        if self._fence is None:
            self._fence = (torch.cuda.Stream(device=self.device, priority=-1), torch.zeros(1, dtype=torch.int32, device=self.device))
        s, flag = self._fence
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            t0 = torch.cuda.Event(enable_timing=True)
            t0.record(s)
            dist.all_reduce(flag)
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(s)
        self._pending = (t0, ev)

    def fence_wait(self, sink: RowSink) -> None:
        """The rows of the job that starts now wait for the fence issued one job ago (nothing to wait for on first use)."""
        pend = getattr(self, "_pending", None)
        self._pending = None
        sink.ready_event = None if pend is None else pend[1]
        self.last_fence = pend                        # diagnostics: how long the rows of this job waited for the region

    def exchange(self, rows_local: int, n_matches_global: torch.Tensor | None, lay: Layout) -> None:
        """``sendrecv`` transport: move every rank's ``rows_local`` staged rows into its slice on ``dst``.  ``dst`` takes the
        sizes from the gathered ``n_matches`` (one device->host read, after all of the job's work has been enqueued).
        ``p2p``: nothing to move."""
        if self.transport == "p2p" or self.ws == 1:
            return
        ops = []
        if self.rank == self.dst:
            nm = n_matches_global.to("cpu", torch.int64).numpy()
            for r in range(self.ws):
                if r == self.dst:
                    continue
                rows_r = int(nm[lay.owned[r]].sum())
                if rows_r > self.caps[r]:
                    raise RuntimeError(f"rank {r} reports {rows_r} rows for a slice of {self.caps[r]}")
                if rows_r:
                    b = int(self.base[r])
                    ops += [dist.P2POp(dist.irecv, self.full[name][b: b + rows_r], r) for name in self.fields]
        elif rows_local:
            ops = [dist.P2POp(dist.isend, self.local[name][:rows_local], self.dst) for name in self.fields]
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()

    def row_starts(self, n_matches_global: torch.Tensor, lay: Layout) -> torch.Tensor:
        """int64 [P]: first row of every pair (global pair order) inside the ``full`` arrays.  Device arithmetic only."""
        dev = n_matches_global.device
        if lay.n_total == 0:
            return torch.zeros(0, dtype=torch.int64, device=dev)
        ix = lay.on(dev)
        n_rm = n_matches_global.to(torch.int64).index_select(0, ix["perm"])          # rank-major order = storage order
        cs = torch.cumsum(n_rm, 0) - n_rm                                          # exclusive scan over all ranks
        seg0 = cs.index_select(0, ix["first"].clamp(max=max(len(n_rm) - 1, 0))) if len(n_rm) else cs
        base = torch.as_tensor(self.base[:-1], dtype=torch.int64, device=dev)
        start_rm = cs - seg0.index_select(0, ix["rank_of"]) + base.index_select(0, ix["rank_of"])
        out = torch.empty_like(start_rm)
        out[ix["perm"]] = start_rm
        return out


class RegionPair:
    """Two regions used in turn, so that the reuse fence of one is issued a whole job before it is needed."""

    def __init__(self, a: GatherRegion, b: GatherRegion):
        self.regions, self.turn = (a, b), 0

    def next(self):
        """(region of the job that starts now, its twin)."""
        cur, other = self.regions[self.turn % 2], self.regions[(self.turn + 1) % 2]
        self.turn += 1
        return cur, other

    def close(self) -> None:
        for r in self.regions:
            r.close()


def get_regions(bank, n_total: int, mode: str, fields, dst: int = 0, rows_per_pair_cap: int | None = None,
                transport: str = "auto") -> RegionPair:
    """Region pairs are cached on the bank (creation is collective: every rank asks for the same sequence of regions)."""
    rank, ws = world()
    cap = int(bank.feat_stride if rows_per_pair_cap is None else rows_per_pair_cap)
    key = (int(n_total), ws, mode, tuple(fields), int(dst), cap, transport)
    cache = bank.__dict__.setdefault("_gather_regions", {})
    reg = cache.get(key)
    if reg is None:
        for old in cache.values():
            old.close()
        cache.clear()
        lay = layout(n_total, ws, mode)
        caps = [n * cap for n in lay.sizes]
        a = GatherRegion(caps, fields, dst, bank.device, transport)
        b = GatherRegion(caps, fields, dst, bank.device, a.transport)              # (the transport the ranks agreed on for the first)
        reg = cache[key] = RegionPair(a, b)
    return reg


def match_and_verify_sharded(bank, pairs, *, mode: str = "block", dst: int = 0, gather: str = "full",
                             transport: str = "auto", rows_per_pair_cap: int | None = None, events: dict | None = None, **params):
    """Every rank holds the (broadcast) bank; the pair list is partitioned; results are gathered on ``dst`` in global pair
    order -- the distributed ``pair_matches`` of code/pipeline.py:43-47.

    gather="summaries": n_matches, n_inliers, iters, F (H / n_inliers_h, R / t / n_pose when those stages are requested).
    gather="full"     : additionally the packed rows of every pair: ``matches`` int32 [rows,3] = (queryIdx, trainIdx, squared
                        L2), ``inlier`` uint8 [rows] (``inlier_h`` / ``in_front`` / ``points3d`` with the optional stages) and
                        ``row_start`` int64 [P]: pair p owns rows ``row_start[p] : row_start[p] + n_matches[p]``; ``pairs``
                        (numpy int32 [P,2]) is the pair list.  ``tracks=True`` (with the options of ``match_and_verify``) then builds
                        the feature tracks of the whole list on ``dst`` from the gathered rows (``out["tracks"]``); the ranks
                        themselves hook nothing.
    All values are device tensors on ``dst`` except ``pairs`` (host) and ``transport`` (a string).  RANSAC streams are keyed by GLOBAL pair index, so every value equals what one
    GPU computes for the whole list.  ``events`` (a dict) receives timing events recorded on the current stream: "compute"
    after this rank's last kernel and row copy, "done" after the gather.  Returns (gathered dict or None, local VerifiedPairs)."""
    from .pipeline import match_and_verify

    if gather not in ("full", "summaries"):
        raise ValueError("gather must be 'full' or 'summaries'")
    track_opts = {k: params.pop(k) for k in ("track_flags", "min_pair_inliers", "min_length", "keep_conflicts") if k in params}
    tracks = bool(params.pop("tracks", False))
    if tracks and gather != "full":
        raise ValueError("tracks=True needs gather='full': the tracks are built from the gathered rows")
    rank, ws = world()
    pairs = np.asarray(pairs, np.int32).reshape(-1, 2)
    n_total = len(pairs)
    lay = layout(n_total, ws, mode)
    mine = lay.owned[rank]
    homography = bool(params.get("homography", False))
    pose = params.get("intrinsics") is not None
    region = sink = None
    if gather == "full":
        fields = tuple(o.name for o in outputs(homography, pose) if o.per == "row")
        region, twin = get_regions(bank, n_total, mode, fields, dst, rows_per_pair_cap, transport).next()
        sink = region.sink()
        region.fence_wait(sink)                       # issued one job ago
        twin.fence_issue()                            # for the next job: behind everything this stream has been asked to do so far
    # pair_id = global pair index, so the RANSAC sample streams (and hence the results) do not depend on the world size
    res = match_and_verify(bank, pairs[mine], pair_ids=mine, sink=sink, **params)
    if events is not None:
        events["compute"] = torch.cuda.Event(enable_timing=True)
        events["compute"].record()
        events["kernels"] = getattr(res.plan, "ev_kernels", None) if sink is not None else None
        events["fence"] = getattr(region, "last_fence", None) if region is not None else None
        events["rows_pushed"] = 0 if sink is None else sink.rows
        events["bytes_pushed"] = 0 if sink is None else sink.bytes
    out = gather_summaries(res, mine, n_total, dst, mode=mode, homography=homography, pose=pose)
    if region is not None:
        region.exchange(sink.rows, out["n_matches"] if rank == dst else None, lay)
        if rank == dst:
            for name in region.fields:
                out[name] = region.full[name]
            out["row_start"] = region.row_starts(out["n_matches"], lay)
            out["pairs"] = pairs                                         # (host: the caller's list, as passed)
            out["transport"] = region.transport
            if tracks:
                opts = dict(track_opts)
                flags = opts.pop("track_flags", "inlier")
                out["tracks"] = build_tracks_from_rows(out, max(bank.n_images, 1), bank.max_feats, flags=flags, **opts)
    if events is not None:
        events["done"] = torch.cuda.Event(enable_timing=True)
        events["done"].record()
        events["transport"] = None if region is None else region.transport
    return out, res
