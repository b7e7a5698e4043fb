"""Execution plan of the hot path for batches of image pairs: preallocated device and pinned-host buffers, a
fixed launch sequence on the caller's stream, and result copies on a side stream that overlap the RANSAC kernel.

    [reverse sweep -> refine: the full kNN table]                sfm_match_knn2                 (mutual=True)
    sweep (tcgen05): candidate records into the scratch          sfm_match_knn2, sweep_only = 4
    refine + ratio / mutual filter -> scan -> gather             sfm_refine_filter_packed       (on a second stream with overlap=True)
    RANSAC-F on the packed correspondences                       sfm_ransac_f_packed
    [RANSAC-H on the same correspondences]                       sfm_ransac_h_packed            (homography=True)
    [E, (R, t) by cheirality vote, triangulated inliers]         sfm_two_view_pose_packed       (intrinsics given)
    [union of the batch's used rows into the job's tracks]       sfm_tracks_hook                (tracks=True)

This is the batched body of the reference's pair loop (code/pipeline.py:38-47) plus the verification stage it left
empty (code/pipeline.py:60-65).  Nothing here computes: every array is produced by lib/libsfm_b200.so.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import NamedTuple

import numpy as np
import torch

from . import _lib
from .bank import DescriptorBank
from .matcher import filter_params
from .ransac import h_stop_target, ransac_params
from .tracks import FLAG_FIELDS, TrackBuilder


def intrinsics_rows(intrinsics, n_images: int) -> np.ndarray:
    """float64 [n_images, 4] = (fx, fy, cx, cy) per image from one 3x3 K, a [n,3,3] stack or ready [n,4] rows."""
    a = np.asarray(intrinsics, np.float64)
    if a.shape == (3, 3):
        a = np.broadcast_to(a, (n_images, 3, 3))
    if a.ndim == 3 and a.shape[1:] == (3, 3):
        if np.any(np.abs(a[:, 0, 1]) > 1e-12):
            raise ValueError("camera matrices with skew are not supported")
        a = np.stack([a[:, 0, 0], a[:, 1, 1], a[:, 0, 2], a[:, 1, 2]], axis=1)
    if a.ndim != 2 or a.shape[1] != 4 or a.shape[0] < n_images:
        raise ValueError(f"intrinsics must be [3,3], [n_images,3,3] or [n_images,4]; got {a.shape} for {n_images} images")
    if not np.all(a[:, :2] > 0):
        raise ValueError("focal lengths must be positive")
    return np.ascontiguousarray(a[:n_images])


class Output(NamedTuple):
    """One result array of the pipeline.  ``per`` is "pair" or "row" (one row per surviving match, packed: pair p owns rows
    [offsets[p], offsets[p+1])); ``shape`` is the trailing shape; ``stage`` is None (always), "homography" or "pose"; ``ready``
    says when a row array is complete: "filter" (written by the filter) or "done" (after the batch's last kernel)."""

    name: str
    per: str
    dtype: torch.dtype
    shape: tuple
    stage: str | None = None
    ready: str = "done"

    @property
    def nbytes(self) -> int:
        """Bytes per pair or per row."""
        return self.dtype.itemsize * math.prod(self.shape)

    def empty(self, n: int, **kw) -> torch.Tensor:
        return torch.empty((n,) + self.shape, dtype=self.dtype, **kw)


# Every result array, in the order results list them.  n_matches is never copied to the host: the host derives it from the offsets.
OUTPUTS = {o.name: o for o in (
    Output("n_matches", "pair", torch.int32, ()),
    Output("F", "pair", torch.float64, (3, 3)),                     # zeros when no model
    Output("n_inliers", "pair", torch.int32, ()),
    Output("iters", "pair", torch.int32, ()),                       # hypotheses evaluated
    Output("H", "pair", torch.float64, (3, 3), "homography"),       # x2 ~ H x1, H[2,2] == 1 (zeros when no model)
    Output("n_inliers_h", "pair", torch.int32, (), "homography"),
    Output("R", "pair", torch.float64, (3, 3), "pose"),             # x2 ~ R x1 + t
    Output("t", "pair", torch.float64, (3,), "pose"),               # |t| = 1
    Output("n_pose", "pair", torch.int32, (), "pose"),              # inliers in front of both cameras
    Output("matches", "row", torch.int32, (3,), ready="filter"),    # (queryIdx, trainIdx, squared L2)
    Output("inlier", "row", torch.uint8, ()),
    Output("inlier_h", "row", torch.uint8, (), "homography"),
    Output("in_front", "row", torch.uint8, (), "pose"),
    Output("points3d", "row", torch.float32, (3,), "pose"),         # in the first camera's frame
)}


def outputs(homography: bool = False, pose: bool = False) -> list[Output]:
    """The result arrays of a run with the given optional stages."""
    return [o for o in OUTPUTS.values() if o.stage is None or (o.stage == "homography" and homography) or (o.stage == "pose" and pose)]


# When bench.py sets this to a list, every sweep launch appends (start event, end event, pairs): the roofline's launch
# duration is then the one measured inside the timed steps, on the stream the kernel runs on.
SWEEP_EVENTS = None


class RowSink:
    """Where a job's packed per-match rows go when they stay on the GPU side instead of travelling to pinned host memory:
    raw device pointers, local or PEER memory (a region of the gathering rank's HBM mapped with sfm_peer_open, see
    dist.GatherRegion).  ``fields`` maps a row array name to (base pointer of this job's slice, bytes per row); the rows of
    consecutive batches land back to back, ``rows`` is the host-side cursor."""

    ROW_BYTES = {o.name: o.nbytes for o in OUTPUTS.values() if o.per == "row"}

    def __init__(self, fields: dict, cap_rows: int):
        for name in fields:
            if name not in self.ROW_BYTES:
                raise ValueError(f"unknown row array {name!r}")
        self.fields = {k: int(v) for k, v in fields.items()}
        self.cap_rows = int(cap_rows)
        self.rows = 0
        self.pairs = 0
        self.bytes = 0
        self.ready_event = None          # CUDA event the first copy of a job must wait for (the region's reuse fence)

    def reset(self) -> None:
        self.rows = self.pairs = self.bytes = 0
        self.ready_event = None


class _OutSet:
    """Device outputs of one batch, one attribute per result array of the plan (``OUTPUTS``) plus the packed offsets and
    correspondences.  Two sets alternate so that batch k + 1 can be enqueued before the host has read batch k's packed size
    and started its copies."""

    def __init__(self, B, cap, dev, outs):
        for o in outs:
            setattr(self, o.name, o.empty(B, device=dev).zero_() if o.per == "pair" else o.empty(B * cap, device=dev))
        self.offsets = torch.zeros(B + 1, dtype=torch.int32, device=dev)
        self.corr = torch.empty((B * cap, 4), dtype=torch.float32, device=dev)
        self.offsets_h = torch.zeros(B + 1, dtype=torch.int32).pin_memory()
        self.ev_filter, self.ev_done = torch.cuda.Event(), torch.cuda.Event()
        self.ev_offsets, self.ev_copied = torch.cuda.Event(), torch.cuda.Event()
        self.copy_pending = False
        self.P = 0
        self.pair_id = None

    @property
    def counts(self) -> torch.Tensor:
        return self.n_matches


class HotPathPlan:
    """Buffers + launch sequence for up to ``max_pairs`` pairs per batch on one bank.

    Packed result layout (device and host): pair p of a batch owns rows [offsets[p], offsets[p+1]) of every row array
    (``OUTPUTS``) and of ``corr`` float32 [total,4].  Host results of a whole job (any number of batches) land back to back
    in ONE set of pinned arrays.
    """

    def __init__(self, bank: DescriptorBank, max_pairs: int, *, ratio=0.75, ratio_mode="cv2_f32", mutual=False,
                 thr=3.0, confidence=0.99, max_iters=2000, solver="7pt", score="sym_epipolar", lo=False, seed=0,
                 min_inliers=0, prefilter=True, homography=False, intrinsics=None, distance_thresh=50.0, h_stop_ratio=0.8, overlap=True,
                 tracks=False, track_flags="inlier", min_pair_inliers=15, min_length=2, keep_conflicts=False):
        if bank.metric != "l2":
            raise ValueError("the verification path needs an L2 bank")
        self.bank, self.B, self.cap, self.dev = bank, int(max_pairs), bank.feat_stride, bank.device
        if self.B < 1:
            raise ValueError("max_pairs must be positive")
        if self.B * self.cap >= 2 ** 31:
            raise ValueError("max_pairs * feat_stride must stay below 2^31 (int32 offsets); use smaller batches")
        self.mutual = bool(mutual)
        self.fprm = filter_params(ratio, ratio_mode, mutual)
        self.rprm = ransac_params(thr=thr, confidence=confidence, max_iters=max_iters, solver=solver, score=score, lo=lo,
                                  seed=seed, min_inliers=min_inliers)
        # The sweep alone: candidate records into the scratch, refined and filtered by sfm_refine_filter_packed.  With the
        # prefilter it marks rows that cannot pass the ratio test; the refinement skips them (they read as "no match").
        self.mprm = _lib.MatchParams()
        self.mprm.sweep_only = 4
        if prefilter:
            self.mprm.prefilter_mode, self.mprm.prefilter_ratio = self.fprm.ratio_mode, self.fprm.ratio
            self.mprm.prefilter_num, self.mprm.prefilter_den = int(self.fprm.ratio_num), int(self.fprm.ratio_den)
        # (mutual matching: the forward direction keeps the prefilter -- a row that fails the ratio test is dropped whatever its
        #  reverse neighbour is; the reverse direction needs every row's exact nearest neighbour: a full kNN table without it)
        self.rev_prm = _lib.MatchParams()
        B, cap, dev = self.B, self.cap, self.dev
        self.knn = torch.empty((B, cap, 4), dtype=torch.int32, device=dev)       # sweep records, then the compacted rows per block
        self.blk_count = torch.empty(B * (cap // 256), dtype=torch.int32, device=dev)
        self.knn_rev = torch.empty((B, cap, 4), dtype=torch.int32, device=dev) if self.mutual else None
        # Two-stream pipeline: the sweep of batch k + 1 runs on the caller's stream while batch k is refined, filtered and
        # verified on ``post_stream``.  The sweep is one persistent 352-thread CTA per SM and leaves registers / shared memory / issue slots
        # for one refinement CTA beside it, so the L1-bound refinement hides under the tensor-bound sweep (4.9 % on a four-batch job,
        # profiles/r02_overlap_proto.log).  Scratch and reverse tables are double-buffered for it (second copies made on first use).
        self.overlap = bool(overlap)
        self.post_stream = torch.cuda.Stream(device=dev) if self.overlap else None
        self._scratch = [(self.knn, self.blk_count, self.knn_rev)]
        self._consumed = [None, None]                                            # event: the post stage has finished with scratch[i]
        # optional stages after RANSAC-F (SURVEY.md 8f ranks 2 and 4)
        self.homography = bool(homography)
        self.h_ratio = None if h_stop_ratio is None else float(h_stop_ratio)
        self.hprm = ransac_params(thr=thr, confidence=confidence, max_iters=max_iters, solver="8pt", lo=lo, seed=seed) if self.homography else None
        self.intr = None
        if intrinsics is not None:
            self.intr = torch.as_tensor(intrinsics_rows(intrinsics, bank.max_images)).to(dev)
        self.dist = float(distance_thresh)
        self.outputs = outputs(self.homography, self.intr is not None)
        # feature tracks of a job (per job, not per pair or row: no entry in OUTPUTS): every batch's rows are hooked on the
        # stream that verified them, before its output set can be reused; match_and_verify begins and finalizes
        self.tracks = None
        if tracks:
            if track_flags not in FLAG_FIELDS or (track_flags is not None and track_flags not in [o.name for o in self.outputs]):
                raise ValueError(f"track_flags {track_flags!r} is not a row array of this plan ({[o.name for o in self.outputs if o.per == 'row']})")
            self.track_flags = track_flags
            self.tracks = TrackBuilder(bank.max_images, bank.max_feats, dev, min_pair_inliers=min_pair_inliers, min_length=min_length,
                                       keep_conflicts=keep_conflicts)
        self.sets = [_OutSet(B, cap, dev, self.outputs)]                        # the second set is created on the first multi-batch job
        self.cur = self.sets[0]
        self._n_launched = 0
        self.copy_stream = torch.cuda.Stream(device=dev)
        # pinned host results of a job: every row array, every per-pair array but n_matches (the host has it from the offsets)
        self._host_rows = [o for o in self.outputs if o.per == "row"]
        self._host_pairs = [o for o in self.outputs if o.per == "pair" and o.name != "n_matches"]
        self._row_bytes = sum(o.nbytes for o in self._host_rows)
        self._pair_bytes = sum(o.nbytes for o in self._host_pairs)
        self.host = {}
        self._rows_cap = self._pairs_cap = 0
        self.job_rows = self.job_pairs = self.job_d2h = 0
        self.job_counts = []

    # ------------------------------------------------------------------ launches (no host synchronisation)
    def launch(self, pairs_d: torch.Tensor, pair_id_d: torch.Tensor, pairs_rev_d: torch.Tensor | None = None) -> _OutSet:
        """Enqueue match -> filter -> verify on the current stream for ``pairs_d`` int32 [P,2] (device, image ids already
        validated by the caller), ``pair_id_d`` int32 [P] (RANSAC stream ids) and, for mutual matching, the swapped pair
        list.  Returns the output set the batch writes (also ``self.cur``)."""
        P = int(pairs_d.shape[0])
        if P > self.B:
            raise ValueError(f"{P} pairs exceed the plan's batch size {self.B}")
        o = self.cur = self.sets[self._n_launched % len(self.sets)]
        self._n_launched += 1
        o.P, o.pair_id = P, pair_id_d
        if P == 0:
            return o
        L, st, bank = _lib.lib(), _lib.current_stream_ptr(self.dev), self.bank
        cur = torch.cuda.current_stream(self.dev)
        slot = (self._n_launched - 1) % 2 if self.overlap else 0
        if slot >= len(self._scratch):                # second scratch set of the two-stream pipeline, on first use
            B, cap = self.B, self.cap
            self._scratch.append((torch.empty((B, cap, 4), dtype=torch.int32, device=self.dev),
                                  torch.empty(B * (cap // 256), dtype=torch.int32, device=self.dev),
                                  torch.empty((B, cap, 4), dtype=torch.int32, device=self.dev) if self.mutual else None))
        knn, blk_count, knn_rev = self._scratch[slot]
        if self._consumed[slot] is not None:
            cur.wait_event(self._consumed[slot])      # the batch that used this scratch two launches ago has been refined and gathered
        if self.mutual:
            if pairs_rev_d is None:
                pairs_rev_d = pairs_d.flip(1).contiguous()
            _lib.check(L.sfm_match_knn2(bank.handle, _lib.ptr(pairs_rev_d), P, C.byref(self.rev_prm), _lib.ptr(knn_rev), st),
                       "sfm_match_knn2 (reverse)")
        timing = SWEEP_EVENTS is not None                                                  # bench.py: in-situ duration of the sweep launches
        if timing:
            t0 = torch.cuda.Event(enable_timing=True)
            t0.record(cur)
        _lib.check(L.sfm_match_knn2(bank.handle, _lib.ptr(pairs_d), P, C.byref(self.mprm), _lib.ptr(knn), st), "sfm_match_knn2 (sweep)")
        ev_sweep = torch.cuda.Event(enable_timing=timing)
        ev_sweep.record(cur)
        if timing:
            SWEEP_EVENTS.append((t0, ev_sweep, P))
        if self.overlap:
            cur = self.post_stream                    # everything below is enqueued behind the sweep on the second stream
            cur.wait_event(ev_sweep)
            st = C.c_void_p(cur.cuda_stream)
        with torch.cuda.stream(cur):
            self._launch_post(o, pairs_d, pair_id_d, P, knn, blk_count, knn_rev, cur, st, slot)
        return o

    def _launch_post(self, o, pairs_d, pair_id_d, P, knn, blk_count, knn_rev, cur, st, slot):
        """Refinement + filter, RANSAC-F and the optional stages of one batch on ``cur``."""
        L, bank = _lib.lib(), self.bank
        if o.copy_pending:                            # result copies of the batch that used this set last
            cur.wait_event(o.ev_copied)
            o.copy_pending = False
        # refinement + ratio / mutual filter in one pass -> offsets -> gather (the kNN table is never written)
        _lib.check(L.sfm_refine_filter_packed(bank.handle, _lib.ptr(pairs_d), P, C.byref(self.fprm), _lib.ptr(knn_rev), _lib.ptr(knn),
                                              _lib.ptr(blk_count), _lib.ptr(o.n_matches), _lib.ptr(o.offsets), _lib.ptr(o.matches),
                                              _lib.ptr(o.corr), st), "sfm_refine_filter_packed")
        if self.overlap:
            ev = torch.cuda.Event()
            ev.record(cur)
            self._consumed[slot] = ev
        o.ev_filter.record(cur)
        self._ransac_f(o, st)
        if self.homography:
            # the scene graph only asks whether H explains more than h_ratio of what F explains: sampling may stop once a
            # homography with that support would have been found (general pairs: 32 hypotheses instead of max_iters)
            tgt = None if self.h_ratio is None else h_stop_target(o.n_inliers[:P], self.h_ratio)
            _lib.check(L.sfm_ransac_h_packed(_lib.ptr(o.corr), _lib.ptr(o.offsets), P, self.cap, _lib.ptr(pair_id_d), None, _lib.ptr(tgt),
                                             C.byref(self.hprm), _lib.ptr(o.H), _lib.ptr(o.n_inliers_h), _lib.ptr(o.inlier_h), None, st),
                       "sfm_ransac_h_packed")
        if self.intr is not None:
            pl = pairs_d.long()
            cam = torch.cat([self.intr[pl[:, 0]], self.intr[pl[:, 1]]], dim=1).contiguous()      # [P, 8] per-pair camera rows
            _lib.check(L.sfm_two_view_pose_packed(_lib.ptr(o.corr), _lib.ptr(o.offsets), P, _lib.ptr(o.inlier), _lib.ptr(o.F),
                                                  _lib.ptr(cam), self.dist, _lib.ptr(o.R), _lib.ptr(o.t), None, _lib.ptr(o.n_pose),
                                                  _lib.ptr(o.in_front), _lib.ptr(o.points3d), st), "sfm_two_view_pose_packed")
        if self.tracks is not None:
            self.tracks.hook(pairs_d, o.offsets, o.n_matches, o.matches,
                             None if self.track_flags is None else getattr(o, self.track_flags), o.n_inliers)
        o.ev_done.record(cur)

    def result_stream(self):
        """Stream on which a launched batch's outputs become valid (the caller's stream, or the pipeline's second stream)."""
        return self.post_stream if self.overlap else torch.cuda.current_stream(self.dev)

    def ensure_sets(self, n: int) -> None:
        """Multi-batch jobs rotate over two output sets, three when the rows go to a sink (created on first use)."""
        while len(self.sets) < n:
            self.sets.append(_OutSet(self.B, self.cap, self.dev, self.outputs))

    def rerun_ransac(self) -> None:
        """Verification stage alone on the packed correspondences of the last batch (bench.py times it in isolation)."""
        if self.cur.P:
            self._ransac_f(self.cur, _lib.current_stream_ptr(self.dev))

    def _ransac_f(self, o, st) -> None:
        """RANSAC-F on the packed correspondences of output set ``o`` (its ``P`` pairs), enqueued on stream ``st``."""
        _lib.check(_lib.lib().sfm_ransac_f_packed(_lib.ptr(o.corr), _lib.ptr(o.offsets), o.P, self.cap, _lib.ptr(o.pair_id), None,
                                                  C.byref(self.rprm), _lib.ptr(o.F), _lib.ptr(o.n_inliers), _lib.ptr(o.inlier),
                                                  _lib.ptr(o.iters), st), "sfm_ransac_f_packed")

    # ------------------------------------------------------------------ host results of a job
    def job_begin(self, n_pairs: int) -> None:
        """Start collecting host results for a job of ``n_pairs`` pairs (any number of batches)."""
        if n_pairs > self._pairs_cap:
            self._pairs_cap = n_pairs
            self.host.update({o.name: o.empty(n_pairs, pin_memory=True) for o in self._host_pairs})
        self.job_rows = self.job_pairs = self.job_d2h = 0
        self.job_counts = []

    def _ensure_rows(self, rows: int, expect_total: int) -> None:
        if rows <= self._rows_cap:
            return
        new_cap = max(rows, expect_total, 2 * self._rows_cap, 1 << 16)
        grown = {o.name: o.empty(new_cap, pin_memory=True) for o in self._host_rows}
        if self.job_rows:                             # a job in progress outgrew the buffer: keep what has arrived
            self.copy_stream.synchronize()
            for name, h in grown.items():
                h[: self.job_rows] = self.host[name][: self.job_rows]
        self.host.update(grown)
        self._rows_cap = new_cap

    def _offsets(self, out: _OutSet) -> np.ndarray:
        """Batch ``out``'s packed offsets on the host: the only host wait, until its filter has finished (RANSAC keeps the GPU
        busy meanwhile)."""
        P, cs = out.P, self.copy_stream
        with torch.cuda.stream(cs):
            cs.wait_event(out.ev_filter)
            out.offsets_h[: P + 1].copy_(out.offsets[: P + 1], non_blocking=True)
            out.ev_offsets.record(cs)
        out.ev_offsets.synchronize()
        return out.offsets_h[: P + 1].numpy()

    def fetch_begin(self, out: _OutSet, pairs_left_after: int = 0) -> None:
        """Enqueue the device -> pinned-host copies of batch ``out`` on the side stream, appending to the job's arrays.
        Blocks the host only until that batch's filter has finished (to learn the packed size); the match rows then
        travel while its RANSAC kernel is running."""
        P = out.P
        if P == 0:
            return
        off = self._offsets(out)
        total = int(off[P])
        r0, p0 = self.job_rows, self.job_pairs
        per_pair = (r0 + total) / max(p0 + P, 1)
        self._ensure_rows(r0 + total, int(1.1 * per_pair * (p0 + P + pairs_left_after)) + 1024)
        cs = self.copy_stream
        with torch.cuda.stream(cs):
            for ready, ev in (("filter", None), ("done", out.ev_done)):
                if ev is not None:
                    cs.wait_event(ev)
                for o in self._host_rows:
                    if o.ready == ready and total:
                        self.host[o.name][r0: r0 + total].copy_(getattr(out, o.name)[:total], non_blocking=True)
            for o in self._host_pairs:
                self.host[o.name][p0: p0 + P].copy_(getattr(out, o.name)[:P], non_blocking=True)
            out.ev_copied.record(cs)
        out.copy_pending = True
        self.job_counts.append(np.diff(off).astype(np.int32))
        self.job_rows, self.job_pairs = r0 + total, p0 + P
        self.job_d2h += 4 * (P + 1) + total * self._row_bytes + P * self._pair_bytes

    def push_begin(self, out: _OutSet, sink: RowSink) -> None:
        """Device-side twin of ``fetch_begin``: append batch ``out``'s packed rows to ``sink`` (local or peer memory) with
        plain device-to-device copies on the side stream -- copy engines over NVLink when the sink is a peer region, so the
        SMs go on with the next batch's sweep.  The host waits only for the batch's filter (to learn the packed size); the
        match rows travel while the batch's RANSAC kernel runs, the inlier flags follow it."""
        P = out.P
        if P == 0:
            return
        total = int(self._offsets(out)[P])
        r0 = sink.rows
        if r0 + total > sink.cap_rows:
            raise _lib.SfmError(f"row sink overflow: {r0 + total} rows exceed the region's capacity {sink.cap_rows}")
        L, cs = _lib.lib(), self.copy_stream
        st = C.c_void_p(cs.cuda_stream)
        if sink.ready_event is not None:              # the consumer of the previous job's rows has finished with the region
            cs.wait_event(sink.ready_event)
            sink.ready_event = None
        for ready, ev in (("filter", None), ("done", out.ev_done)):
            if ev is not None:
                cs.wait_event(ev)
            for name in sink.fields:
                if OUTPUTS[name].ready != ready:
                    continue
                src = getattr(out, name, None)
                if src is None:
                    raise ValueError(f"the plan does not produce {name!r} (request the stage that does)")
                rb = RowSink.ROW_BYTES[name]
                if total:
                    _lib.check(L.sfm_copy_async(C.c_void_p(sink.fields[name] + r0 * rb), _lib.ptr(src), total * rb, st),
                               "sfm_copy_async")
                    sink.bytes += total * rb
        out.ev_copied.record(cs)
        out.copy_pending = True
        sink.rows, sink.pairs = r0 + total, sink.pairs + P

    def job_end(self) -> dict:
        """Wait for the job's copies and return numpy VIEWS of the pinned arrays (valid until the next job on this plan)."""
        self.copy_stream.synchronize()
        P, rows = self.job_pairs, self.job_rows
        n_matches = np.concatenate(self.job_counts) if self.job_counts else np.zeros(0, np.int32)
        offsets = np.zeros(P + 1, np.int64)
        np.cumsum(n_matches, out=offsets[1:])
        out = {"n_matches": n_matches, "offsets": offsets}
        for o in self._host_rows + self._host_pairs:
            n = rows if o.per == "row" else P
            out[o.name] = self.host[o.name][:n].numpy() if n else o.empty(0).numpy()
        return out
