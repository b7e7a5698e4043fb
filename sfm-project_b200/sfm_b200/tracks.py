"""Feature tracks from the verified matches: host plumbing of csrc/tracks.cu (include/sfm_b200.h, "feature tracks").

A track is the set of (image, feature) observations of one scene point, joined through the used match rows -- what the
reference's empty ``code/3d_reconstruction.py`` (imported at ``code/pipeline.py:4``) would build from the ``pair_matches``
of ``code/pipeline.py:43-47``.  Node ``n = image * S + feature``; kept tracks are numbered in ascending order of their
smallest node and list their observations in ascending node order, so the result depends only on the set of used rows.
Nothing here computes: init, hook and finalize are kernels of lib/libsfm_b200.so, and the workspace is allocated here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib

# row arrays that can select the used rows (None: every row)
FLAG_FIELDS = (None, "inlier", "inlier_h", "in_front")
COUNT_NAMES = ("n_tracks", "n_obs", "n_conflicting", "n_short", "n_invalid_rows")
FINALIZE_LAUNCHES = 14          # kernels sfm_tracks_finalize launches (init and every non-empty hook launch one each)


@dataclass
class Tracks:
    """Tracks on the device.  The output buffers are sized for the worst case (the kernels never wait for the host); the
    first look at a count or at ``offsets`` / ``obs`` / ``track_of`` reads the five counts back -- the one host wait -- raises
    when a used row was invalid, and trims the views.

    ``offsets`` int64 [T+1]: track k owns ``obs[offsets[k]:offsets[k+1]]``; ``obs`` int32 [n_obs, 2] = (image, feature);
    ``track_of`` int32 [n_images, S]: track id of every feature, -1 = none.  ``n_conflicting`` counts the candidates that
    hold two features of one image (dropped unless ``keep_conflicts``), ``n_short`` the candidates dropped for having fewer
    than ``min_length`` observations."""

    offsets_buf: torch.Tensor
    obs_buf: torch.Tensor
    track_of_buf: torch.Tensor
    counts_dev: torch.Tensor                       # int64 [5], COUNT_NAMES order
    _counts: dict | None = field(default=None, repr=False)

    @property
    def counts(self) -> dict:
        if self._counts is None:
            c = dict(zip(COUNT_NAMES, (int(v) for v in self.counts_dev.cpu().tolist())))
            if c["n_invalid_rows"]:
                raise _lib.SfmError(f"{c['n_invalid_rows']} used match rows name a feature outside [0, S) or an image outside "
                                    f"[0, n_images): the row data does not belong to this image / feature numbering")
            self._counts = c
        return self._counts

    @property
    def n_tracks(self) -> int:
        return self.counts["n_tracks"]

    @property
    def n_obs(self) -> int:
        return self.counts["n_obs"]

    @property
    def offsets(self) -> torch.Tensor:
        return self.offsets_buf[: self.n_tracks + 1]

    @property
    def obs(self) -> torch.Tensor:
        return self.obs_buf[: self.n_obs]

    @property
    def track_of(self) -> torch.Tensor:
        self.counts                                  # (raises on invalid rows, like every other view)
        return self.track_of_buf

    def to_host(self) -> dict:
        """numpy ``offsets``, ``obs``, ``track_of`` and the counts."""
        out = {"offsets": self.offsets.cpu().numpy(), "obs": self.obs.cpu().numpy(), "track_of": self.track_of.cpu().numpy()}
        out.update(self.counts)
        return out


class TrackBuilder:
    """Caller-owned workspace for up to ``max_images`` x ``S`` nodes and the three entry points, enqueued on the current
    stream: ``begin`` (init), ``hook`` (any number of batches), ``finalize`` (-> ``Tracks``)."""

    def __init__(self, max_images: int, S: int, device, *, min_pair_inliers: int = 15, min_length: int = 2,
                 keep_conflicts: bool = False):
        if int(min_length) < 2:
            raise ValueError(f"min_length must be at least 2, got {min_length}")
        self.max_images, self.S, self.device = int(max_images), int(S), torch.device(device)
        self.prm = _lib.TrackParams(int(min_pair_inliers), int(min_length), int(bool(keep_conflicts)))
        nbytes = C.c_size_t(0)
        _lib.check(_lib.lib().sfm_tracks_workspace_bytes(self.max_images, self.S, C.byref(nbytes)), "sfm_tracks_workspace_bytes")
        self.ws = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)
        self.n_images = self.max_images
        self._row_start = torch.empty(0, dtype=torch.int64, device=self.device)

    def begin(self, n_images: int | None = None) -> None:
        n = self.max_images if n_images is None else int(n_images)
        if not 0 < n <= self.max_images:
            raise ValueError(f"n_images must lie in [1, {self.max_images}], got {n}")
        self.n_images = n
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().sfm_tracks_init(n, self.S, _lib.ptr(self.ws), self.ws.numel(), _lib.current_stream_ptr(self.device)),
                       "sfm_tracks_init")

    def hook(self, pairs, row_start, n_rows, rows, row_flag=None, n_inliers=None) -> None:
        """Add the used rows of a batch: ``pairs`` int32 [P,2], ``row_start`` int64 [P] (int32 offsets, as the plan's
        output sets hold them, are first widened into a buffer kept here: one torch copy on the same stream, which
        ``sfm_launch_count`` does not count), ``n_rows`` int32 [P], ``rows`` int32 [.,3], ``row_flag`` uint8 [.] or None, ``n_inliers`` int32
        [P] or None -- device tensors."""
        P = int(pairs.shape[0])
        if P == 0:
            return
        if row_start.dtype != torch.int64:
            if self._row_start.numel() < P:
                self._row_start = torch.empty(max(P, 2 * self._row_start.numel()), dtype=torch.int64, device=self.device)
            self._row_start[:P].copy_(row_start[:P])
            row_start = self._row_start
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().sfm_tracks_hook(self.n_images, self.S, _lib.ptr(pairs), P, _lib.ptr(row_start), _lib.ptr(n_rows),
                                                  _lib.ptr(rows), _lib.ptr(row_flag), _lib.ptr(n_inliers), C.byref(self.prm),
                                                  _lib.ptr(self.ws), self.ws.numel(), _lib.current_stream_ptr(self.device)),
                       "sfm_tracks_hook")

    def finalize(self) -> Tracks:
        n_nodes = self.n_images * self.S
        dev = self.device
        t = Tracks(offsets_buf=torch.empty(n_nodes // 2 + 1, dtype=torch.int64, device=dev),
                   obs_buf=torch.empty((n_nodes, 2), dtype=torch.int32, device=dev),
                   track_of_buf=torch.empty((self.n_images, self.S), dtype=torch.int32, device=dev),
                   counts_dev=torch.empty(len(COUNT_NAMES), dtype=torch.int64, device=dev))
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().sfm_tracks_finalize(self.n_images, self.S, C.byref(self.prm), _lib.ptr(self.ws), self.ws.numel(),
                                                      _lib.ptr(t.track_of_buf), _lib.ptr(t.offsets_buf), _lib.ptr(t.obs_buf),
                                                      _lib.ptr(t.counts_dev), _lib.current_stream_ptr(dev)), "sfm_tracks_finalize")
        return t


def _dev(x, dtype, device, shape=None):
    if x is None:
        return None
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    t = t.to(device=device, dtype=dtype)
    return (t if shape is None else t.reshape(shape)).contiguous()


def build_tracks_device(pairs, row_start, n_rows, rows, row_flag, n_inliers, n_images: int, S: int, *, min_pair_inliers: int = 15,
                        min_length: int = 2, keep_conflicts: bool = False, device=None) -> Tracks:
    """Tracks of one set of packed rows, on ``device`` (default: that of ``rows`` when it is a CUDA tensor, else the current
    device): pair p = ``pairs[p]`` owns rows ``row_start[p] : row_start[p] + n_rows[p]`` of ``rows`` (int32 [.,3] =
    (queryIdx, trainIdx, d2)) and ``row_flag``.  Arrays may be host or device; device ones of the right dtype are used in place."""
    if device is None:
        device = rows.device if isinstance(rows, torch.Tensor) and rows.is_cuda else torch.device("cuda", torch.cuda.current_device())
    dev = torch.device(device)
    pairs_t = _dev(pairs, torch.int32, dev, (-1, 2))
    P = int(pairs_t.shape[0])
    b = TrackBuilder(n_images, S, dev, min_pair_inliers=min_pair_inliers, min_length=min_length, keep_conflicts=keep_conflicts)
    with torch.cuda.device(dev):
        b.begin()
        b.hook(pairs_t, _dev(row_start, torch.int64, dev, (P,)), _dev(n_rows, torch.int32, dev, (P,)), _dev(rows, torch.int32, dev, (-1, 3)),
               _dev(row_flag, torch.uint8, dev, (-1,)), _dev(n_inliers, torch.int32, dev, (P,)))
        return b.finalize()


def flag_rows(result: dict, flags: str | None):
    """The row array of ``result`` that selects the used rows (None: every row)."""
    if flags not in FLAG_FIELDS:
        raise ValueError(f"flags must be one of {FLAG_FIELDS}, got {flags!r}")
    if flags is not None and flags not in result:
        raise ValueError(f"the result carries no {flags!r} rows (request the stage that produces them)")
    return None if flags is None else result[flags]


def build_tracks_from_rows(out: dict, n_images: int, S: int, *, flags: str | None = "inlier", min_pair_inliers: int = 15,
                           min_length: int = 2, keep_conflicts: bool = False) -> Tracks:
    """Tracks of a gathered result dict (``dist.match_and_verify_sharded(gather="full")`` on the destination rank: ``pairs``,
    ``row_start``, ``n_matches``, ``n_inliers``, ``matches`` and the flag row array), device tensors used in place."""
    return build_tracks_device(out["pairs"], out["row_start"], out["n_matches"], out["matches"], flag_rows(out, flags),
                               out["n_inliers"], n_images, S, min_pair_inliers=min_pair_inliers, min_length=min_length,
                               keep_conflicts=keep_conflicts, device=out["matches"].device)
