"""Bundle adjustment: registered cameras and triangulated points refined together, host plumbing of csrc/bundle.cu
(include/sfm_b200.h, "bundle adjustment").

Levenberg-Marquardt in fp64 on the squared pixel residuals of the used observations (track point status 0, observation an
inlier of its point, image registered), the normal equations reduced to the variable cameras by the Schur complement and
solved by a dense blocked Cholesky.  The call is a fixed launch sequence that never waits for the host: ``BundleResult``
reads its summary back on first look.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import torch

from . import _lib
from .tracks import Tracks
from .triangulate import TrackPoints

STATUS_NAMES = ("function_tolerance", "parameter_tolerance", "max_iterations", "no_progress", "nothing_to_adjust", "invalid")
BUNDLE_LAUNCHES_FIXED = 4        # kernels sfm_bundle_adjust launches besides the iterations: three of set-up, one of output
BUNDLE_LAUNCHES_PER_ITER = 5     # kernels per Levenberg-Marquardt iteration (all of them, whether or not the solve has stopped)
MAX_IMAGES = 1024


def bundle_launches(max_iters: int) -> int:
    """Kernels one ``sfm_bundle_adjust`` call launches."""
    return BUNDLE_LAUNCHES_FIXED + BUNDLE_LAUNCHES_PER_ITER * int(max_iters)


@dataclass
class BundleResult:
    """The adjusted reconstruction on the device.  ``pose`` float64 [n_images, 12] = R (row-major), t (drops into
    ``cams[:, 4:]``); ``X_buf`` float64 [max_tracks, 3] and ``obs_error_buf`` float32 [max_obs] (pixel error of every
    observation after the adjustment, as ``TrackPoints.obs_error``).  The first look at ``summary`` reads it back."""

    tracks: Tracks
    pose: torch.Tensor
    X_buf: torch.Tensor
    obs_error_buf: torch.Tensor
    summary_dev: torch.Tensor                       # uint8 [64]: sfm_bundle_summary
    _summary: dict | None = field(default=None, repr=False)

    @property
    def summary(self) -> dict:
        """``status`` (a ``STATUS_NAMES`` entry), ``status_code``, ``iterations``, ``accepted``, ``used_obs``, ``variable_cameras``,
        ``adjusted_points``, ``initial_cost``, ``final_cost``."""
        if self._summary is None:
            s = _lib.BundleSummary.from_buffer_copy(bytes(self.summary_dev.cpu().numpy()))
            self._summary = {name: getattr(s, name) for name, _ in s._fields_}
            self._summary["status_code"] = int(s.status)
            self._summary["status"] = STATUS_NAMES[int(s.status)]
        return self._summary

    @property
    def R(self) -> torch.Tensor:
        return self.pose[:, :9].reshape(-1, 3, 3)

    @property
    def t(self) -> torch.Tensor:
        return self.pose[:, 9:]

    @property
    def X(self) -> torch.Tensor:
        return self.X_buf[: self.tracks.n_tracks]

    @property
    def obs_error(self) -> torch.Tensor:
        return self.obs_error_buf[: self.tracks.n_obs]

    def to_host(self) -> dict:
        """numpy ``pose``, ``R``, ``t``, ``X``, ``obs_error`` and the summary."""
        out = {k: getattr(self, k).cpu().numpy() for k in ("pose", "R", "t", "X", "obs_error")}
        out.update(self.summary)
        return out


def bundle_params(*, max_iters=50, function_tolerance=1e-6, parameter_tolerance=1e-8):
    if not 1 <= int(max_iters) <= 10000:
        raise ValueError(f"max_iters must lie in [1, 10000], got {max_iters}")
    for name, v in (("function_tolerance", function_tolerance), ("parameter_tolerance", parameter_tolerance)):
        if not 0 <= float(v) < 1e300:
            raise ValueError(f"{name} must be non-negative and finite, got {v}")
    return _lib.BundleParams(float(function_tolerance), float(parameter_tolerance), int(max_iters))


def _mask(m, n, dev, name):
    if m is None:
        return None
    t = torch.as_tensor(m).to(device=dev).reshape(-1)
    if t.numel() != n:
        raise ValueError(f"{name} must have {n} entries, got {t.numel()}")
    return (t != 0).to(torch.uint8).contiguous()


def bundle_adjust_device(tracks: Tracks, points: TrackPoints, xy: torch.Tensor, cams: torch.Tensor, registered=None, *, fixed=None,
                         update: bool = False, S: int | None = None, workspace: torch.Tensor | None = None, **params) -> BundleResult:
    """Refine every variable camera and every adjusted point of ``points`` together, enqueued on the current stream without a
    host wait.

    ``xy`` float32 [n_images, xy_stride, 2] (a bank's ``DescriptorBank.xy``), ``cams`` float64 [n_images, 16] (the table
    ``triangulate_tracks_device`` reads), ``registered`` / ``fixed`` bool or uint8 [n_images] or None (None: every image
    registered; the lowest-index registered image fixed).  n_images is at most 1024.  With ``update=True`` the poses are written
    into ``cams[:, 4:]`` and the points and errors into ``points.X_buf`` / ``points.obs_error_buf`` by torch copies on the same
    stream; ``cams`` must then be a contiguous float64 tensor on the tracks' device.  ``workspace`` (uint8, at least
    ``workspace_bytes`` long) may be passed to reuse one across calls.  ``params``: see ``bundle_params``."""
    dev = tracks.obs_buf.device
    prm = bundle_params(**params)
    if xy.dtype != torch.float32 or xy.dim() != 3 or xy.shape[2] != 2 or xy.device != dev or not xy.is_contiguous():
        raise ValueError("xy must be a contiguous float32 tensor [n_images, stride, 2] on the tracks' device")
    n_images, stride = int(xy.shape[0]), int(xy.shape[1])
    if not 0 < n_images <= MAX_IMAGES:
        raise ValueError(f"bundle adjustment takes 1 to {MAX_IMAGES} images, got {n_images}")
    if update and not (isinstance(cams, torch.Tensor) and cams.dtype == torch.float64 and cams.device == dev and cams.is_contiguous()):
        raise ValueError("update=True writes the poses into cams: it must be a contiguous float64 tensor on the tracks' device")
    cams_t = torch.as_tensor(cams).to(device=dev, dtype=torch.float64).contiguous()
    if tuple(cams_t.shape) != (n_images, 16):
        raise ValueError(f"cams must be [{n_images}, 16], got {tuple(cams_t.shape)}")
    reg = _mask(registered, n_images, dev, "registered")
    fix = _mask(fixed, n_images, dev, "fixed")
    max_tracks, max_obs = int(points.X_buf.shape[0]), int(points.obs_inlier_buf.numel())
    ws = workspace_bytes(n_images, max_tracks, max_obs)
    if workspace is None:
        workspace = torch.empty(ws, dtype=torch.uint8, device=dev)
    elif workspace.dtype != torch.uint8 or workspace.numel() < ws or workspace.device != dev:
        raise ValueError(f"workspace must be a uint8 tensor of at least {ws} bytes on {dev}")
    out = BundleResult(tracks=tracks, pose=torch.empty((n_images, 12), dtype=torch.float64, device=dev),
                       X_buf=torch.empty((max_tracks, 3), dtype=torch.float64, device=dev),
                       obs_error_buf=torch.empty(max_obs, dtype=torch.float32, device=dev),
                       summary_dev=torch.empty(C.sizeof(_lib.BundleSummary), dtype=torch.uint8, device=dev))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sfm_bundle_adjust(
            n_images, stride if S is None else int(S), _lib.ptr(tracks.offsets_buf), _lib.ptr(tracks.obs_buf), _lib.ptr(tracks.counts_dev),
            max_tracks, max_obs, _lib.ptr(points.status_buf), _lib.ptr(points.obs_inlier_buf), _lib.ptr(points.X_buf), _lib.ptr(xy), stride,
            _lib.ptr(cams_t), _lib.ptr(reg), _lib.ptr(fix), C.byref(prm), _lib.ptr(workspace), workspace.numel(), _lib.ptr(out.pose),
            _lib.ptr(out.X_buf), _lib.ptr(out.obs_error_buf), _lib.ptr(out.summary_dev), _lib.current_stream_ptr(dev)), "sfm_bundle_adjust")
        if update:
            cams_t[:, 4:] = out.pose
            points.X_buf.copy_(out.X_buf)
            points.obs_error_buf.copy_(out.obs_error_buf)
    return out


def workspace_bytes(n_images: int, max_tracks: int, max_obs: int) -> int:
    """Bytes of device workspace ``sfm_bundle_adjust`` needs; the reduced camera system alone is (6 n_images)^2 doubles."""
    n = C.c_size_t(0)
    _lib.check(_lib.lib().sfm_bundle_workspace_bytes(int(n_images), int(max_tracks), int(max_obs), C.byref(n)), "sfm_bundle_workspace_bytes")
    return int(n.value)
