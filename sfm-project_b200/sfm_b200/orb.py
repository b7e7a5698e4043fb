"""ORB extraction on the GPU (C ABI: sfm_orb_resize, sfm_orb_blur, sfm_orb_describe, sfm_orb_fast_detect, sfm_orb_retain_best,
sfm_orb_harris_angle).

The reference extracts with ``cv2.ORB_create().detectAndCompute(gray, None)`` (code/feature_matching.py:42-45), which is 91 % of
its per-pair time (SURVEY.md §8 a1).  Both halves run here, bit for bit what cv2 computes (csrc/orb.cu; tests/test_gpu_orb.py):

* descriptors (``OrbDescriber``): pyramid, per-level Gaussian blur, 256 rotated intensity tests per keypoint;
* detection (``OrbExtractor``): per level FAST-9/16 with corner score, non-maximum suppression, border rule, row-major
  compaction on the device; ``retainBest`` (libstdc++'s nth_element + partition, whose permutation IS cv2's keypoint order) on
  the host on a few thousand floats; Harris response and intensity-centroid orientation on the device.

The host side only prepares integers and float32 scalars: level sizes, 8.8 fixed-point resize tables, features per level, each
keypoint's rounded position in its level and (cos, sin).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

F32, F64 = np.float32, np.float64
N_LEVELS = 8
SCALE_FACTOR = F64(F32(1.2))           # cv2.ORB_create() default, a float argument widened to double


def level_scale(level: int) -> np.float32:
    """float32(1.2f ** level): the factor between level-0 and level-``level`` coordinates."""
    return F32(np.power(SCALE_FACTOR, F64(level)))


def level_sizes(width: int, height: int, n_levels: int = N_LEVELS):
    """(w, h) of every pyramid level as cv2 sizes them: round-half-even of the float32 product w * float32(1 / scale).  Dividing
    by the scale instead rounds differently on 281 (width, level) pairs below 8192, e.g. 525 / 1.2 = 437.49997 but
    525 * float32(1 / 1.2) = 437.5 -> 438."""
    out = [(int(width), int(height))]
    for k in range(1, n_levels):
        inv = F32(F32(1.0) / level_scale(k))
        out.append((int(np.rint(F32(F32(width) * inv))), int(np.rint(F32(F32(height) * inv)))))
    return out


_TABLES = {}


def resize_table(src_n: int, dst_n: int) -> np.ndarray:
    """int32 [dst_n, 2] = (source index, weight of the next source pixel in 1/256) of INTER_LINEAR_EXACT along one axis:
    source coordinate (d + 1/2) src/dst - 1/2 in exact integer arithmetic, clamped to the image, fraction rounded half-even to 8 bits."""
    key = (int(src_n), int(dst_n))
    t = _TABLES.get(key)
    if t is None:
        d = np.arange(dst_n, dtype=np.int64)
        num, den = (2 * d + 1) * src_n - dst_n, 2 * dst_n            # coordinate = num / den
        fl = np.floor_divide(num, den)
        fr = num - fl * den
        q, r = np.divmod(fr * 256, den)
        c1 = q + ((2 * r > den) | ((2 * r == den) & (q & 1 == 1)))
        lo, hi = fl < 0, fl >= src_n - 1
        fl = np.where(lo, 0, np.where(hi, src_n - 1, fl))
        c1 = np.where(lo | hi, 0, c1)
        t = np.ascontiguousarray(np.stack([fl, c1], axis=1).astype(np.int32))
        if len(_TABLES) > 256:
            _TABLES.clear()
        _TABLES[key] = t
    return t


def keypoint_records(kps, n_levels: int = N_LEVELS):
    """(int32 [n, 4] = x, y in the level image, level, 0;  float32 [n, 2] = cos, sin) from cv2 keypoints (or float32 [n, 4] rows
    pt.x, pt.y, angle in degrees, octave): the roundings cv2 applies before it samples."""
    if isinstance(kps, np.ndarray):
        a = np.ascontiguousarray(kps, F32).reshape(-1, 4)
    else:
        a = np.array([[k.pt[0], k.pt[1], k.angle, k.octave] for k in kps], F32).reshape(-1, 4)
    lv = a[:, 3].astype(np.int32)
    if len(lv) and (lv.min() < 0 or lv.max() >= n_levels):
        raise ValueError(f"keypoint octaves must lie in [0, {n_levels})")
    inv = np.array([F32(1.0) / level_scale(k) for k in range(n_levels)], F32)[lv]
    rec = np.zeros((len(a), 4), np.int32)
    rec[:, 0] = np.rint(a[:, 0] * inv)
    rec[:, 1] = np.rint(a[:, 1] * inv)
    rec[:, 2] = lv
    rad = (a[:, 2] * F32(np.pi / 180.0)).astype(F32)
    rot = np.stack([np.cos(rad.astype(F64)).astype(F32), np.sin(rad.astype(F64)).astype(F32)], axis=1)
    return rec, np.ascontiguousarray(rot)


class OrbDescriber:
    """Device buffers for one image size (pyramid, blurred pyramid, resize tables) and the launch sequence:
    7 resizes, 8 blurs, 1 descriptor kernel per image."""

    EDGE = 31                      # cv2.ORB_create() edgeThreshold: no keypoint lies closer to a level's border

    def __init__(self, width: int, height: int, device=None, n_levels: int = N_LEVELS):
        if not torch.cuda.is_available():
            raise _lib.SfmError("OrbDescriber needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n_levels = int(n_levels)
        self.sizes = level_sizes(width, height, self.n_levels)
        if min(self.sizes[-1]) < 1:
            raise ValueError(f"image {width} x {height} is too small for {n_levels} pyramid levels")
        dev = self.device
        self.raw = [torch.empty((h, w), dtype=torch.uint8, device=dev) for w, h in self.sizes]
        self.blur = [torch.empty((h, w), dtype=torch.uint8, device=dev) for w, h in self.sizes]
        self.tabs = []
        for k in range(1, self.n_levels):
            (sw, sh), (dw, dh) = self.sizes[k - 1], self.sizes[k]
            self.tabs.append((torch.from_numpy(resize_table(sw, dw)).to(dev), torch.from_numpy(resize_table(sh, dh)).to(dev)))
        self._ptrs = (C.c_void_p * self.n_levels)(*[t.data_ptr() for t in self.blur])
        self._pitch = (C.c_int32 * self.n_levels)(*[w for w, _ in self.sizes])
        self._stage = torch.empty((height, width), dtype=torch.uint8).pin_memory()

    def pyramid(self, gray) -> None:
        """Upload ``gray`` (uint8 [H, W] numpy / torch, host or device) and build the raw and blurred levels."""
        L, st = _lib.lib(), _lib.current_stream_ptr(self.device)
        w0, h0 = self.sizes[0]
        if isinstance(gray, torch.Tensor) and gray.is_cuda:
            self.raw[0].copy_(gray)
        else:
            g = gray if isinstance(gray, np.ndarray) else gray.numpy()
            if g.shape != (h0, w0) or g.dtype != np.uint8:
                raise ValueError(f"expected a uint8 image of {h0} x {w0}, got {g.dtype} {g.shape}")
            self._stage.numpy()[...] = g
            self.raw[0].copy_(self._stage, non_blocking=True)
        for k in range(1, self.n_levels):
            (sw, sh), (dw, dh) = self.sizes[k - 1], self.sizes[k]
            xt, yt = self.tabs[k - 1]
            _lib.check(L.sfm_orb_resize(_lib.ptr(self.raw[k - 1]), sw, sh, sw, _lib.ptr(self.raw[k]), dw, dh, dw, _lib.ptr(xt), _lib.ptr(yt), st),
                       "sfm_orb_resize")
        for k in range(self.n_levels):
            w, h = self.sizes[k]
            _lib.check(L.sfm_orb_blur(_lib.ptr(self.raw[k]), w, h, w, _lib.ptr(self.blur[k]), w, st), "sfm_orb_blur")

    def describe(self, gray, kps, out: torch.Tensor | None = None) -> torch.Tensor:
        """uint8 [n, 32] descriptors (device) of cv2 keypoints on ``gray``; ``out`` may be rows of a Hamming bank."""
        rec, rot = keypoint_records(kps, self.n_levels)
        n = len(rec)
        if n:
            # cv2 never returns a keypoint whose 31-pixel patch leaves its level; a caller-made one must not read out of bounds
            w = np.array([s[0] for s in self.sizes])[rec[:, 2]]
            h = np.array([s[1] for s in self.sizes])[rec[:, 2]]
            if (rec[:, 0] < 22).any() or (rec[:, 1] < 22).any() or (rec[:, 0] >= w - 22).any() or (rec[:, 1] >= h - 22).any():
                raise ValueError("a keypoint lies closer than 22 pixels to the border of its pyramid level")
        if out is None:
            out = torch.empty((n, 32), dtype=torch.uint8, device=self.device)
        elif out.dtype != torch.uint8 or out.dim() != 2 or out.shape[0] < n or out.shape[1] != 32 or not out.is_contiguous():
            raise ValueError("out must be a contiguous uint8 [>= n, 32] CUDA tensor")
        self.pyramid(gray)
        if n:
            rec_d = torch.from_numpy(rec).to(self.device)
            rot_d = torch.from_numpy(rot).to(self.device)
            _lib.check(_lib.lib().sfm_orb_describe(self._ptrs, self._pitch, self.n_levels, _lib.ptr(rec_d), _lib.ptr(rot_d), n, _lib.ptr(out), 32,
                                                   _lib.current_stream_ptr(self.device)), "sfm_orb_describe")
            self._keep = (rec_d, rot_d)
        return out[:n]


_DESCRIBERS = {}


def describe(gray, kps, device=None, out=None) -> torch.Tensor:
    """Descriptors of cv2 keypoints on ``gray`` with a describer cached per image size."""
    h, w = gray.shape
    if not torch.cuda.is_available():
        raise _lib.SfmError("ORB extraction needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    key = (w, h, str(dev))
    d = _DESCRIBERS.get(key)
    if d is None:
        if len(_DESCRIBERS) >= 8:
            _DESCRIBERS.clear()
        d = _DESCRIBERS[key] = OrbDescriber(w, h, dev)
    return d.describe(gray, kps, out)


# ------------------------------------------------------------------------------------ detection (stage 2)
N_FEATURES, EDGE, PATCH, FAST_THRESHOLD = 500, 31, 31, 20           # cv2.ORB_create() defaults


def features_per_level(nfeatures: int = N_FEATURES, n_levels: int = N_LEVELS) -> list:
    """cv2's geometric split of ``nfeatures`` over the levels (float32 arithmetic, round-half-even, remainder to the last)."""
    factor = F32(1.0 / SCALE_FACTOR)
    nd = F32(nfeatures) * (F32(1) - factor) / (F32(1) - F32(np.power(F64(factor), F64(n_levels))))
    out, total = [], 0
    for _ in range(n_levels - 1):
        out.append(int(np.rint(nd)))
        total += out[-1]
        nd = F32(nd * factor)
    out.append(max(nfeatures - total, 0))
    return out


def retain_best(response: np.ndarray, n_points: int) -> np.ndarray:
    """KeyPointsFilter::retainBest: indices of the survivors in cv2's order (host; sfm_orb_retain_best)."""
    r = np.ascontiguousarray(response, F32)
    out = np.empty(max(len(r), 1), np.int32)
    n = _lib.lib().sfm_orb_retain_best(r.ctypes.data_as(C.c_void_p), len(r), int(n_points), out.ctypes.data_as(C.c_void_p))
    if n < 0:
        _lib.check(n, "sfm_orb_retain_best")
    return out[:n]


class OrbExtractor(OrbDescriber):
    """``cv2.ORB_create().detectAndCompute(gray, None)`` on the GPU: keypoints as float32 [n, 6] rows
    (pt.x, pt.y, size, angle, response, octave) in cv2's order, descriptors uint8 [n, 32] on the device.

    Host side of one image: two waits for the device (FAST counts, then the FAST scores of every level in one pinned
    buffer), ``retainBest`` of the eight levels on eight host threads (libstdc++'s nth_element on ~10^5 keypoints of a
    textured 1080p level 0 is the longest single item of the whole extraction; ctypes releases the GIL), the Harris /
    orientation kernels launched level by level as the selections arrive, one copy back of all candidates."""

    def __init__(self, width: int, height: int, device=None, n_levels: int = N_LEVELS, nfeatures: int = N_FEATURES):
        super().__init__(width, height, device, n_levels)
        dev = self.device
        self.per_level = features_per_level(nfeatures, self.n_levels)
        self.score = [torch.empty((h, w), dtype=torch.uint8, device=dev) for w, h in self.sizes]
        self.row_count = [torch.zeros(max(h, 1), dtype=torch.int32, device=dev) for _, h in self.sizes]
        self.totals = torch.zeros(self.n_levels, dtype=torch.int32, device=dev)
        self.totals_h = torch.zeros(self.n_levels, dtype=torch.int32).pin_memory()
        self.cap = [w * h // 4 + 1 for w, h in self.sizes]               # 3 x 3 suppression leaves at most one keypoint per 2 x 2
        self.xy = [torch.empty((c, 2), dtype=torch.int32, device=dev) for c in self.cap]
        self.resp = [torch.empty(c, dtype=torch.float32, device=dev) for c in self.cap]
        self.resp_h = [torch.empty(c, dtype=torch.float32).pin_memory() for c in self.cap]
        self._alloc_candidates(2 * max(self.per_level) + 64)
        self._pool = None

    def _alloc_candidates(self, m: int) -> None:
        """Per level, ``m`` candidate slots: selection indices in, (x, y) / Harris response / angle out -- one device buffer and
        one pinned twin each way, so that every level travels in the same copy."""
        dev, nl = self.device, self.n_levels
        self.m = int(m)
        self.sel_h = torch.zeros((nl, self.m), dtype=torch.int32).pin_memory()
        self.sel_d = torch.zeros((nl, self.m), dtype=torch.int32, device=dev)
        self.cand_d = torch.zeros((nl, 4, self.m), dtype=torch.int32, device=dev)       # rows: x, y (as [m, 2] over two rows), response, angle
        self.cand_h = torch.zeros((nl, 4, self.m), dtype=torch.int32).pin_memory()

    def _executor(self):
        if self._pool is None:
            from concurrent.futures import ThreadPoolExecutor

            self._pool = ThreadPoolExecutor(max_workers=self.n_levels, thread_name_prefix="orb-select")
        return self._pool

    def detect(self, gray, _pyramid_done: bool = False) -> np.ndarray:
        L, st = _lib.lib(), _lib.current_stream_ptr(self.device)
        if not _pyramid_done:
            self.pyramid(gray)
        for k, (w, h) in enumerate(self.sizes):
            _lib.check(L.sfm_orb_fast_detect(_lib.ptr(self.raw[k]), w, h, w, FAST_THRESHOLD, EDGE, _lib.ptr(self.score[k]), _lib.ptr(self.row_count[k]),
                                             C.c_void_p(self.totals.data_ptr() + 4 * k), _lib.ptr(self.xy[k]), _lib.ptr(self.resp[k]), st),
                       "sfm_orb_fast_detect")
        stream = torch.cuda.current_stream(self.device)
        self.totals_h.copy_(self.totals, non_blocking=True)
        stream.synchronize()                                            # host wait 1: how many FAST keypoints per level
        totals = [int(t) for t in self.totals_h.numpy()]
        for k in range(self.n_levels):
            if totals[k]:
                self.resp_h[k][: totals[k]].copy_(self.resp[k][: totals[k]], non_blocking=True)
        stream.synchronize()                                            # host wait 2: their FAST scores, all levels
        # retainBest(2 n_level) by FAST score: every level on its own host thread, the small ones first to the device
        pool = self._executor()
        jobs = {k: pool.submit(retain_best, self.resp_h[k][: totals[k]].numpy(), 2 * self.per_level[k]) for k in range(self.n_levels)}
        sels = [None] * self.n_levels
        need = 0
        for k in range(self.n_levels):
            sels[k] = jobs[k].result() if totals[k] else np.zeros(0, np.int32)
            need = max(need, len(sels[k]))
        if need > self.m:                                               # ties at the threshold can keep more than 2 n
            self._alloc_candidates(need + 64)
        for k in reversed(range(self.n_levels)):
            n = len(sels[k])
            if n == 0:
                continue
            w, h = self.sizes[k]
            self.sel_h[k, :n] = torch.from_numpy(sels[k])
            self.sel_d[k, :n].copy_(self.sel_h[k, :n], non_blocking=True)
            base = self.cand_d[k]
            _lib.check(L.sfm_orb_harris_angle(_lib.ptr(self.raw[k]), w, h, w, _lib.ptr(self.xy[k]), _lib.ptr(self.sel_d[k]), n, _lib.ptr(base[0]),
                                              _lib.ptr(base[2]), _lib.ptr(base[3]), st), "sfm_orb_harris_angle")
        self.cand_h.copy_(self.cand_d, non_blocking=True)
        stream.synchronize()                                            # host wait 3: positions, responses and angles of the candidates
        cand = self.cand_h.numpy()
        rows = []
        for k in range(self.n_levels):
            n = len(sels[k])
            if n == 0:
                continue
            xy = cand[k, 0:2].reshape(-1)[: 2 * n].reshape(n, 2)          # the kernel writes [n, 2] pairs from the start of row 0
            hr = cand[k, 2, :n].view(F32)
            ang = cand[k, 3, :n].view(F32)
            keep = retain_best(hr, self.per_level[k])
            sf = level_scale(k)
            out = np.empty((len(keep), 6), F32)
            x, y = xy[keep, 0].astype(F32), xy[keep, 1].astype(F32)
            out[:, 0] = x * sf if k else x
            out[:, 1] = y * sf if k else y
            out[:, 2] = F32(PATCH) * sf
            out[:, 3] = ang[keep]
            out[:, 4] = hr[keep]
            out[:, 5] = k
            rows.append(out)
        return np.concatenate(rows) if rows else np.zeros((0, 6), F32)

    def detect_and_compute(self, gray, out: torch.Tensor | None = None):
        """(keypoints float32 [n, 6], descriptors uint8 [n, 32] on the device) == cv2.ORB_create().detectAndCompute(gray, None)."""
        self.pyramid(gray)
        kp = self.detect(gray, _pyramid_done=True)
        rec, rot = keypoint_records(np.ascontiguousarray(kp[:, [0, 1, 3, 5]]), self.n_levels)
        n = len(rec)
        if out is None:
            out = torch.empty((n, 32), dtype=torch.uint8, device=self.device)
        if n:
            rec_d, rot_d = torch.from_numpy(rec).to(self.device), torch.from_numpy(rot).to(self.device)
            _lib.check(_lib.lib().sfm_orb_describe(self._ptrs, self._pitch, self.n_levels, _lib.ptr(rec_d), _lib.ptr(rot_d), n, _lib.ptr(out), 32,
                                                   _lib.current_stream_ptr(self.device)), "sfm_orb_describe")
            self._keep = (rec_d, rot_d)
        return kp, out[:n]


_EXTRACTORS = {}


def detect_and_compute(gray, device=None):
    """``cv2.ORB_create().detectAndCompute(gray, None)`` on the GPU with an extractor cached per image size."""
    h, w = gray.shape
    if not torch.cuda.is_available():
        raise _lib.SfmError("ORB extraction needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    key = (w, h, str(dev))
    e = _EXTRACTORS.get(key)
    if e is None:
        if len(_EXTRACTORS) >= 4:
            _EXTRACTORS.clear()
        e = _EXTRACTORS[key] = OrbExtractor(w, h, dev)
    return e.detect_and_compute(gray)


def to_cv2_keypoints(kp: np.ndarray):
    """list[cv2.KeyPoint] from float32 [n, 6] rows (what cv2.drawMatches wants)."""
    import cv2

    return [cv2.KeyPoint(float(r[0]), float(r[1]), float(r[2]), float(r[3]), float(r[4]), int(r[5]), -1) for r in kp]
