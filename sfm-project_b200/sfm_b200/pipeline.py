"""The throughput path: match a pair list from the bank, then verify every pair (K2 -> K5 -> K4).

This is the batched counterpart of the reference's serial double loop (code/pipeline.py:36-49) plus the
geometric-verification stage the reference left empty (code/pipeline.py:60-65).  ``pipeline.py`` itself is
left untouched; this driver sits beside it.
"""
from __future__ import annotations

import os
import time

from dataclasses import dataclass, field

import numpy as np
import torch

from .bank import DescriptorBank
from .plan import OUTPUTS, HotPathPlan, RowSink, outputs
from .tracks import Tracks, build_tracks_device


@dataclass
class VerifiedPairs:
    """Per-pair summaries stay on the device; the variable-length part (matches, inlier flags) is streamed to the
    host batch by batch when ``fetch=True`` and is then available through ``to_host``."""

    pairs: torch.Tensor          # int32 [P,2]
    n_matches: torch.Tensor      # int32 [P]
    F: torch.Tensor              # float64 [P,3,3]  (zeros when no model)
    n_inliers: torch.Tensor      # int32 [P]
    iters: torch.Tensor          # int32 [P]        hypotheses evaluated
    host: dict | None = field(default=None, repr=False)
    d2h_bytes: int = 0
    # optional stages (None unless requested): homography model and two-view initialisation
    H: torch.Tensor | None = None            # float64 [P,3,3]  x2 ~ H x1, H[2,2] == 1 (zeros when no model)
    n_inliers_h: torch.Tensor | None = None  # int32 [P]
    R: torch.Tensor | None = None            # float64 [P,3,3]  x2 ~ R x1 + t
    t: torch.Tensor | None = None            # float64 [P,3]    |t| = 1
    n_pose: torch.Tensor | None = None       # int32 [P]        inliers in front of both cameras
    plan: HotPathPlan | None = field(default=None, repr=False)     # the plan that ran the job (its buffers hold the last batch)
    tracks: Tracks | None = None             # feature tracks of the job (tracks=True)

    def to_host(self, with_matches: bool = True) -> dict:
        """``pairs, n_matches, F, n_inliers, iters`` and, with ``with_matches``, the packed rows
        ``matches`` int32 [sum n_matches, 3] = (queryIdx, trainIdx, squared L2), ``inlier`` uint8 [sum n_matches],
        ``offsets`` int64 [P+1] (pair p owns rows offsets[p]:offsets[p+1])."""
        if self.host is not None:
            out = dict(self.host)
            if not with_matches:
                for k in ["offsets"] + [o.name for o in OUTPUTS.values() if o.per == "row"]:
                    out.pop(k, None)
            return out
        if with_matches:
            raise ValueError("matches were not fetched: call match_and_verify(..., fetch=True)")
        out = {"pairs": self.pairs.cpu().numpy()}
        for o in OUTPUTS.values():
            if o.per == "pair" and getattr(self, o.name) is not None:
                out[o.name] = getattr(self, o.name).cpu().numpy()
        return out


_PLAN_KEYS = ("ratio", "ratio_mode", "mutual", "thr", "confidence", "max_iters", "solver", "score", "lo", "seed",
              "min_inliers", "prefilter", "homography", "distance_thresh", "h_stop_ratio", "overlap",
              "tracks", "track_flags", "min_pair_inliers", "min_length", "keep_conflicts")


def get_plan(bank: DescriptorBank, batch: int, **params) -> HotPathPlan:
    """Plans (device + pinned buffers) are cached on the bank, one per (batch size, parameter set)."""
    params.setdefault("homography", False)
    params.setdefault("distance_thresh", 50.0)
    params.setdefault("h_stop_ratio", 0.8)
    params.setdefault("overlap", True)
    if not params.get("tracks"):                    # the track options only matter to a plan that builds tracks
        for k in ("tracks", "track_flags", "min_pair_inliers", "min_length", "keep_conflicts"):
            params.pop(k, None)
    intr = params.get("intrinsics")
    key = (int(batch),) + tuple(params.get(k) for k in _PLAN_KEYS) + (None if intr is None else np.asarray(intr, np.float64).tobytes(),)
    cache = bank.__dict__.setdefault("_plans", {})
    plan = cache.get(key)
    if plan is None:
        if len(cache) >= 4:
            cache.clear()
        plan = cache[key] = HotPathPlan(bank, batch, **params)
    return plan


def match_and_verify(bank: DescriptorBank, pairs, *, ratio=0.75, ratio_mode="cv2_f32", mutual=False,
                     thr=3.0, confidence=0.99, max_iters=2000, solver="7pt", score="sym_epipolar", lo=False, seed=0,
                     min_inliers=0, pair_batch: int = 2048, pair_ids=None, fetch=False,
                     prefilter: bool = True, homography: bool = False, intrinsics=None, distance_thresh: float = 50.0,
                     h_stop_ratio: float | None = 0.8, sink: RowSink | None = None, overlap: bool = True, tracks: bool = False,
                     track_flags: str | None = "inlier", min_pair_inliers: int = 15, min_length: int = 2, keep_conflicts: bool = False,
                     _segments=None) -> VerifiedPairs:
    """Match and verify every pair of ``pairs`` (int32 [P,2], image ids in the bank).

    ``pair_ids`` (default 0..P-1) name the RANSAC sample stream of each pair, so a sharded run that passes global
    pair indices reproduces the single-GPU result exactly.  ``fetch=True`` also streams every batch's matches and
    inlier flags to the host (pinned buffers, copies overlapped with the RANSAC kernel of the same batch and the
    sweep of the next one); ``fetch="view"`` hands out the pinned result arrays themselves
    (zero host copies; valid until the next call with the same parameters on this bank).  ``prefilter`` lets the sweep drop rows that provably fail the ratio test before the
    exact refinement (results are identical with or without it).  ``overlap`` runs the sweep of batch k + 1 on the caller's
    stream while batch k is refined, filtered and verified on a second stream (a job that fits one batch is cut in two for it); on return the
    caller's stream has waited for everything.

    Two optional stages run on the same packed correspondences right after RANSAC-F (SURVEY.md §8f ranks 2 and 4):
    ``homography=True`` also fits a RANSAC homography per pair (``H``, ``n_inliers_h``; host rows ``inlier_h``), the
    second model a scene graph needs to tell planar / panoramic pairs from general ones (see
    ``geometric_verification.classify_pairs``; its sampling stops once a homography explaining ``h_stop_ratio`` of the pair's
    F inliers would have been found -- pass ``None`` for the plain stop rule); ``intrinsics`` (one 3x3 K, ``[n_images,3,3]`` or ``[n_images,4]`` rows
    fx fy cx cy) recovers the relative pose of every pair from its F and inliers (``R``, ``t``, ``n_pose``; host rows
    ``in_front`` and ``points3d`` float32 [rows,3] in the first camera's frame).

    ``tracks=True`` also builds the job's feature tracks (``VerifiedPairs.tracks``, see ``sfm_b200.tracks``) on the GPU: each
    batch's rows are hooked right after its last kernel, so tracks exist with ``fetch=False`` too and no row is kept or moved.
    A row is used when its ``track_flags`` row array (``"inlier"``, ``"inlier_h"``, ``"in_front"`` or None = every row) is
    set and its pair has ``n_inliers >= min_pair_inliers``; candidates holding two features of one image are dropped unless
    ``keep_conflicts``, then those shorter than ``min_length``.  Node numbering uses the bank's ``max_feats`` features per
    image and its ``n_images`` images."""
    pairs_host = np.ascontiguousarray(np.asarray(pairs.cpu() if isinstance(pairs, torch.Tensor) else pairs, np.int32).reshape(-1, 2))
    P = pairs_host.shape[0]
    if P and (pairs_host.min() < 0 or pairs_host.max() >= bank.n_images):
        raise ValueError(f"pair list refers to images outside [0, {bank.n_images})")
    ids_host = np.arange(P, dtype=np.int64) if pair_ids is None else np.asarray(pair_ids, np.int64).reshape(P)
    dev = bank.device
    if sink is not None and fetch:
        raise ValueError("fetch and sink are alternatives: rows go either to pinned host memory or to a device sink")
    if P == 0:
        # the arrays of every requested stage exist (empty), so that callers never have to special-case P == 0
        outs = outputs(homography, intrinsics is not None)
        host = None
        if fetch:
            host = {"pairs": pairs_host, "offsets": np.zeros(1, np.int64), **{o.name: o.empty(0).numpy() for o in outs}}
        trk = None
        if tracks:
            none = np.zeros(0, np.int32)
            trk = build_tracks_device(none, none, none, none, None, None, max(bank.n_images, 1), bank.max_feats,
                                      min_pair_inliers=min_pair_inliers, min_length=min_length, keep_conflicts=keep_conflicts, device=dev)
        return VerifiedPairs(pairs=torch.zeros((0, 2), dtype=torch.int32, device=dev), host=host, tracks=trk,
                             **{o.name: o.empty(0, device=dev) for o in outs if o.per == "pair"})
    batch = int(min(pair_batch, P))
    if overlap and not _segments and 512 <= P <= batch:
        batch = -(-P // 2)                          # one-batch job: two halves, so that the first half's refinement hides under the second sweep
    plan = get_plan(bank, batch, ratio=ratio, ratio_mode=ratio_mode, mutual=mutual, thr=thr, confidence=confidence,
                    max_iters=max_iters, solver=solver, score=score, lo=lo, seed=seed, min_inliers=min_inliers, prefilter=prefilter,
                    homography=homography, intrinsics=intrinsics, distance_thresh=distance_thresh, h_stop_ratio=h_stop_ratio, overlap=overlap,
                    tracks=tracks, track_flags=track_flags, min_pair_inliers=min_pair_inliers, min_length=min_length,
                    keep_conflicts=keep_conflicts)
    # one upload of the whole pair list and its RANSAC stream ids through a pinned staging buffer kept on the bank
    # (allocating pinned memory per call costs ~0.2 ms of idle GPU at the head of every job)
    stage = bank.__dict__.get("_pair_stage")
    if stage is None or stage[0].shape[0] < 3 * P:
        n = max(3 * P, 3 * 4096)
        stage = (torch.empty(n, dtype=torch.int32).pin_memory(), torch.empty(n, dtype=torch.int32, device=dev), torch.cuda.Event())
        bank.__dict__["_pair_stage"] = stage
    else:
        stage[2].synchronize()                        # the previous job's upload has left the staging buffer
    stage_h, stage_d, stage_ev = stage
    stage_h[: 2 * P].view(P, 2).numpy()[...] = pairs_host
    stage_h[2 * P: 3 * P].numpy()[...] = ids_host.astype(np.uint32).view(np.int32)
    stage_d[: 3 * P].copy_(stage_h[: 3 * P], non_blocking=True)
    stage_ev.record(torch.cuda.current_stream(dev))
    pairs_d = stage_d[: 2 * P].view(P, 2)
    ids_d = stage_d[2 * P: 3 * P]
    rev_d = pairs_d.flip(1).contiguous() if mutual else None
    if plan.tracks is not None:
        plan.tracks.begin(bank.n_images)              # ordered before every hook: the first sweep follows it on this stream
    # (the full-length result arrays are allocated after the first batch has been enqueued: every host microsecond before
    #  the first kernel is GPU idle time, everything after it hides behind the sweep)
    results = {}

    # batches: consecutive runs of <= batch pairs; with _segments (streamed upload) a batch never crosses a segment end and
    # first waits for the event that says the segment's images are in the bank
    cuts, waits = [], {}
    seg_ends = [(P, None)] if not _segments else list(_segments)
    s0 = 0
    for end, ev in seg_ends:
        first = True
        while s0 < end:
            n = min(batch, end - s0)
            cuts.append((s0, n))
            if first and ev is not None:
                waits[s0] = ev
            first = False
            s0 += n
    # Output sets: two alternate (batch k's rows are copied out while batch k+1 runs).  With a sink the host must read batch k's
    # packed size before it can enqueue the copy: with THREE sets it reads the size of batch k-1 after enqueuing batch k+1, a wait
    # that is normally over already, so a late host thread or a slow peer copy no longer stalls the kernels of the next batch.
    push_lag = 2 if (sink is not None and len(cuts) > 2) else 1
    plan.ensure_sets(min(len(cuts), push_lag + 1))
    pending = []
    if fetch:
        plan.job_begin(P)
    prev = None                                      # (output set, pairs remaining after it) of the batch still to be fetched
    trace = [] if os.environ.get("SFM_HOST_TRACE") else None          # diagnostics: host time per batch (enqueue, blocking waits)
    plan.host_trace = trace
    for s, n in cuts:
        if s in waits:
            torch.cuda.current_stream(dev).wait_event(waits[s])
        if trace is not None:
            trace.append(time.perf_counter())
        o = plan.launch(pairs_d[s: s + n], ids_d[s: s + n], None if rev_d is None else rev_d[s: s + n])
        if trace is not None:
            trace.append(time.perf_counter())
        if not results:
            results = {a.name: a.empty(P, device=dev) for a in plan.outputs if a.per == "pair"}
            if plan.overlap:                         # the result arrays were allocated on the caller's stream and are written on the second one
                plan.post_stream.wait_stream(torch.cuda.current_stream(dev))
        # per-pair summaries of this batch into the full-length device arrays (tiny device copies, ordered behind the batch's kernels)
        with torch.cuda.stream(plan.result_stream()):
            for name, full in results.items():
                full[s: s + n].copy_(getattr(o, name)[:n])
        if fetch:
            # the host learns batch k's packed size only after batch k + 1 has been enqueued: the GPU never waits for it
            if prev is not None:
                plan.fetch_begin(*prev)
            prev = (o, P - (s + n))
        elif sink is not None:
            pending.append(o)
            if len(pending) > push_lag:
                plan.push_begin(pending.pop(0), sink)
        if trace is not None:
            trace.append(time.perf_counter())
    if plan.overlap:
        torch.cuda.current_stream(dev).wait_stream(plan.post_stream)     # the caller's stream sees every batch's results
    trk = plan.tracks.finalize() if plan.tracks is not None else None
    host, d2h = None, 0
    if sink is not None:
        plan.ev_kernels = torch.cuda.Event(enable_timing=True)           # diagnostics: the job's last kernel, before its last row copies
        plan.ev_kernels.record()
        for o in pending:
            plan.push_begin(o, sink)
        torch.cuda.current_stream(dev).wait_stream(plan.copy_stream)      # later work on this stream sees the rows in place
    if fetch:
        plan.fetch_begin(*prev)
        h = plan.job_end()
        d2h = plan.job_d2h
        if fetch != "view":                          # the pinned arrays are reused by the next job on this bank: copy out
            h = {k: v.copy() for k, v in h.items()}
        host = dict(h)
        host["pairs"] = pairs_host
    return VerifiedPairs(pairs=pairs_d.clone(), host=host, d2h_bytes=d2h, plan=plan, tracks=trk, **results)      # (pairs_d is a view of the staging buffer)


def match_and_verify_host(desc, xy, pairs, *, bank: DescriptorBank | None = None, n_chunks: int = 3, fetch=True, pair_ids=None, chunk_growth: float = 1.0, **params):
    """The whole job from HOST descriptors: upload, pack, match, verify, results back -- with the upload overlapped.

    ``desc`` uint8 [n_images, n_feats, 128] and ``xy`` float32 [n_images, n_feats, 2] (pinned torch tensors avoid a staging
    copy).  The images travel in ``n_chunks`` groups on a side stream; the pair list is stably re-ordered by the group of
    max(i, j), so matching of the pairs inside the first groups runs while the later images are still on the bus.
    RANSAC streams are keyed by the CALLER's pair index (or ``pair_ids[k]`` for the caller's pair k), so per-pair results equal
    ``match_and_verify`` on a resident bank.

    Returns ``(VerifiedPairs, pair_index)``: everything in PROCESSING order; ``pair_index[k]`` is the caller's index of
    processed pair k (``res.to_host()['pairs']`` holds the pairs in that order)."""
    desc_t = desc if isinstance(desc, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(desc, np.uint8))
    xy_t = None if xy is None else (xy if isinstance(xy, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(xy, np.float32)))
    n_img, n = int(desc_t.shape[0]), int(desc_t.shape[1])
    if bank is None:
        bank = DescriptorBank(n_img, n)
    pairs_host = np.ascontiguousarray(np.asarray(pairs, np.int32).reshape(-1, 2))
    if len(pairs_host) and (pairs_host.min() < 0 or pairs_host.max() >= n_img):
        raise ValueError(f"pair list refers to images outside [0, {n_img})")
    n_chunks = max(1, min(int(n_chunks), n_img))
    # chunk_growth > 1 makes the first groups smaller (the GPU starts earlier); measured on the bench scene equal groups win:
    # 10.06 ms against 10.17 (1.5) and 10.46 (2.0) -- every extra small batch costs more than the upload gap it hides
    bounds = (n_img * np.linspace(0.0, 1.0, n_chunks + 1) ** float(chunk_growth)).round().astype(int)
    bounds[-1] = n_img
    group = np.searchsorted(bounds[1:], pairs_host.max(axis=1), side="right") if len(pairs_host) else np.zeros(0, int)
    order = np.argsort(group, kind="stable")
    cs = bank.__dict__.setdefault("_upload_stream", torch.cuda.Stream(device=bank.device))
    cur = torch.cuda.current_stream(bank.device)
    cs.wait_stream(cur)                                        # earlier work on the bank (a previous job) must be finished
    segments, done = [], 0
    with torch.cuda.stream(cs):
        for c in range(n_chunks):
            a, b = int(bounds[c]), int(bounds[c + 1])
            if b > a:
                bank.put(a, desc_t[a:b], xy=None if xy_t is None else xy_t[a:b])
            ev = torch.cuda.Event()
            ev.record(cs)
            done += int((group == c).sum())
            segments.append((done, ev))
    bank.n_images = n_img
    ids = order if pair_ids is None else np.asarray(pair_ids, np.int64).reshape(len(pairs_host))[order]
    res = match_and_verify(bank, pairs_host[order], pair_ids=ids, fetch=fetch, _segments=segments, **params)
    return res, order
