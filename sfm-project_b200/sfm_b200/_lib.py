"""ctypes binding of lib/libsfm_b200.so (C ABI: include/sfm_b200.h).

There is deliberately no fallback: if the shared library is missing or a call
fails, this module raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C sfm-project_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG_DIR, "lib", "libsfm_b200.so")

METRIC_L2, METRIC_HAMMING = 0, 1
RATIO_NONE, RATIO_CV2_F32, RATIO_EXACT_INT = 0, 1, 2
MATCH_AUTO, MATCH_TCGEN05, MATCH_SIMT = 0, 1, 2
SCORE_SYM_EPIPOLAR, SCORE_SAMPSON = 0, 1

RATIO_MODES = {None: RATIO_NONE, "none": RATIO_NONE, "cv2_f32": RATIO_CV2_F32, "exact_int": RATIO_EXACT_INT}
MATCH_IMPLS = {"auto": MATCH_AUTO, "tcgen05": MATCH_TCGEN05, "simt": MATCH_SIMT}
SCORES = {"sym_epipolar": SCORE_SYM_EPIPOLAR, "sampson": SCORE_SAMPSON}
SOLVERS = {"7pt": 7, "8pt": 8, 7: 7, 8: 8}

# every symbol include/sfm_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "sfm_last_error", "sfm_abi_version", "sfm_device_info",
    "sfm_bank_storage_bytes", "sfm_bank_create", "sfm_bank_destroy", "sfm_bank_layout",
    "sfm_bank_put_batch", "sfm_bank_mark_filled",
    "sfm_match_knn2", "sfm_filter_matches", "sfm_filter_matches_packed", "sfm_match_pairs_packed", "sfm_refine_filter_packed", "sfm_match_hamming",
    "sfm_ransac_f_batch", "sfm_ransac_f_packed", "sfm_ransac_h_batch", "sfm_ransac_h_packed",
    "sfm_two_view_pose_batch", "sfm_two_view_pose_packed",
    "sfm_orb_resize", "sfm_orb_blur", "sfm_orb_describe", "sfm_orb_fast_detect", "sfm_orb_retain_best", "sfm_orb_harris_angle",
    "sfm_tracks_workspace_bytes", "sfm_tracks_init", "sfm_tracks_hook", "sfm_tracks_finalize", "sfm_triangulate_tracks",
    "sfm_pnp_gather", "sfm_pnp_ransac", "sfm_bundle_workspace_bytes", "sfm_bundle_adjust", "sfm_next_images", "sfm_filter_points",
    "sfm_peer_alloc", "sfm_peer_open", "sfm_peer_close", "sfm_peer_free", "sfm_copy_async", "sfm_probe_int8_mma", "sfm_debug_tc_tile", "sfm_debug_refine_stats", "sfm_launch_count",
]


class MatchParams(C.Structure):
    _fields_ = [("impl", C.c_int32), ("grid", C.c_int32), ("prefilter_mode", C.c_int32), ("sweep_only", C.c_int32),
                ("prefilter_ratio", C.c_double), ("prefilter_num", C.c_int32), ("prefilter_den", C.c_int32)]


class FilterParams(C.Structure):
    _fields_ = [
        ("ratio_mode", C.c_int32), ("mutual", C.c_int32), ("ratio", C.c_double),
        ("ratio_num", C.c_int64), ("ratio_den", C.c_int64),
        ("max_distance_sq", C.c_int32), ("reserved", C.c_int32 * 3),
    ]


class RansacParams(C.Structure):
    _fields_ = [
        ("solver", C.c_int32), ("score", C.c_int32), ("threshold", C.c_float), ("max_iters", C.c_int32),
        ("confidence", C.c_double), ("seed", C.c_uint64), ("lo_refit", C.c_int32), ("min_inliers", C.c_int32),
        ("reserved", C.c_int32 * 4),
    ]


class TrackParams(C.Structure):
    _fields_ = [("min_pair_inliers", C.c_int32), ("min_length", C.c_int32), ("keep_conflicts", C.c_int32),
                ("reserved", C.c_int32 * 5)]


class TriangulateParams(C.Structure):
    _fields_ = [("max_error", C.c_double), ("min_angle", C.c_double), ("confidence", C.c_double), ("seed", C.c_uint64),
                ("max_iters", C.c_int32), ("min_inliers", C.c_int32), ("reserved", C.c_int32 * 6)]


class PnpParams(C.Structure):
    _fields_ = [("max_error", C.c_double), ("confidence", C.c_double), ("seed", C.c_uint64), ("max_iters", C.c_int32),
                ("min_inliers", C.c_int32), ("min_inlier_ratio", C.c_double), ("refine_iters", C.c_int32), ("reserved", C.c_int32 * 5)]


class BundleParams(C.Structure):
    _fields_ = [("function_tolerance", C.c_double), ("parameter_tolerance", C.c_double), ("max_iters", C.c_int32),
                ("reserved", C.c_int32 * 11)]


class BundleSummary(C.Structure):
    _fields_ = [("status", C.c_int64), ("iterations", C.c_int64), ("accepted", C.c_int64), ("used_obs", C.c_int64),
                ("variable_cameras", C.c_int64), ("adjusted_points", C.c_int64), ("initial_cost", C.c_double), ("final_cost", C.c_double)]


class NextImagesParams(C.Structure):
    _fields_ = [("min_visible", C.c_int32), ("max_trials", C.c_int32), ("max_select", C.c_int32), ("levels", C.c_int32),
                ("reserved", C.c_int32 * 12)]


class FilterPointsParams(C.Structure):
    _fields_ = [("max_error", C.c_double), ("min_angle", C.c_double), ("min_inliers", C.c_int32), ("reserved", C.c_int32 * 11)]


class SfmError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded library.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SfmError(
            f"{LIB_PATH} not found: the CUDA library has not been built. "
            "Run __graft_entry__.build() (or make -C sfm-project_b200/csrc). There is no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    vp, i32, u64, sz = C.c_void_p, C.c_int, C.c_uint64, C.c_size_t
    L.sfm_last_error.restype = C.c_char_p
    L.sfm_abi_version.restype = C.c_int
    L.sfm_launch_count.restype = C.c_int64
    L.sfm_device_info.argtypes = [i32, vp]
    L.sfm_bank_storage_bytes.argtypes = [i32, i32, i32, C.POINTER(sz)]
    L.sfm_bank_create.argtypes = [i32, i32, i32, i32, vp, sz, C.POINTER(vp)]
    L.sfm_bank_destroy.argtypes = [vp]
    L.sfm_bank_layout.argtypes = [vp, vp]
    L.sfm_bank_put_batch.argtypes = [vp, i32, i32, vp, i32, vp, vp, vp]
    L.sfm_bank_mark_filled.argtypes = [vp, i32]
    L.sfm_match_knn2.argtypes = [vp, vp, i32, C.POINTER(MatchParams), vp, vp]
    L.sfm_filter_matches.argtypes = [vp, vp, i32, vp, vp, C.POINTER(FilterParams), vp, vp, vp, vp]
    L.sfm_filter_matches_packed.argtypes = [vp, vp, i32, vp, vp, C.POINTER(FilterParams), vp, vp, vp, vp, vp]
    L.sfm_match_pairs_packed.argtypes = [vp, vp, i32, C.POINTER(MatchParams), C.POINTER(FilterParams), vp, vp, vp, vp, vp, vp, vp, vp]
    L.sfm_refine_filter_packed.argtypes = [vp, vp, i32, C.POINTER(FilterParams), vp, vp, vp, vp, vp, vp, vp, vp]
    L.sfm_ransac_f_packed.argtypes = [vp, vp, i32, i32, vp, vp, C.POINTER(RansacParams), vp, vp, vp, vp, vp]
    L.sfm_match_hamming.argtypes = [vp, vp, i32, i32, vp, vp, vp, sz, vp]
    L.sfm_ransac_f_batch.argtypes = [vp, i32, vp, i32, vp, vp, C.POINTER(RansacParams), vp, vp, vp, vp, vp]
    L.sfm_ransac_h_batch.argtypes = [vp, i32, vp, i32, vp, vp, vp, C.POINTER(RansacParams), vp, vp, vp, vp, vp]
    L.sfm_ransac_h_packed.argtypes = [vp, vp, i32, i32, vp, vp, vp, C.POINTER(RansacParams), vp, vp, vp, vp, vp]
    L.sfm_two_view_pose_batch.argtypes = [vp, i32, vp, i32, vp, vp, vp, C.c_double, vp, vp, vp, vp, vp, vp, vp]
    L.sfm_two_view_pose_packed.argtypes = [vp, vp, i32, vp, vp, vp, C.c_double, vp, vp, vp, vp, vp, vp, vp]
    L.sfm_orb_resize.argtypes = [vp, i32, i32, i32, vp, i32, i32, i32, vp, vp, vp]
    L.sfm_orb_blur.argtypes = [vp, i32, i32, i32, vp, i32, vp]
    L.sfm_orb_describe.argtypes = [vp, vp, i32, vp, vp, i32, vp, i32, vp]
    L.sfm_orb_fast_detect.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.sfm_orb_retain_best.argtypes = [vp, i32, i32, vp]
    L.sfm_orb_harris_angle.argtypes = [vp, i32, i32, i32, vp, vp, i32, vp, vp, vp, vp]
    L.sfm_tracks_workspace_bytes.argtypes = [i32, i32, C.POINTER(sz)]
    L.sfm_tracks_init.argtypes = [i32, i32, vp, sz, vp]
    L.sfm_tracks_hook.argtypes = [i32, i32, vp, i32, vp, vp, vp, vp, vp, C.POINTER(TrackParams), vp, sz, vp]
    L.sfm_tracks_finalize.argtypes = [i32, i32, C.POINTER(TrackParams), vp, sz, vp, vp, vp, vp, vp]
    L.sfm_triangulate_tracks.argtypes = [i32, i32, vp, vp, vp, C.c_int64, vp, i32, vp, vp, C.POINTER(TriangulateParams), vp, vp, vp, vp,
                                         vp, vp, vp]
    L.sfm_pnp_gather.argtypes = [i32, i32, vp, vp, C.c_int64, vp, vp, vp, i32, vp, i32, vp, vp, vp, vp, vp]
    L.sfm_pnp_ransac.argtypes = [i32, vp, vp, i32, vp, vp, i32, vp, C.POINTER(PnpParams), vp, vp, vp, vp, vp, vp, vp]
    L.sfm_bundle_workspace_bytes.argtypes = [i32, C.c_int64, C.c_int64, C.POINTER(sz)]
    L.sfm_bundle_adjust.argtypes = [i32, i32, vp, vp, vp, C.c_int64, C.c_int64, vp, vp, vp, vp, i32, vp, vp, vp, C.POINTER(BundleParams),
                                    vp, sz, vp, vp, vp, vp, vp]
    L.sfm_next_images.argtypes = [i32, i32, vp, vp, C.c_int64, vp, vp, i32, vp, vp, vp, C.POINTER(NextImagesParams), vp, vp, vp, vp, vp]
    L.sfm_filter_points.argtypes = [i32, vp, vp, vp, C.c_int64, vp, vp, vp, C.POINTER(FilterPointsParams), vp, vp, vp, vp, vp, vp]
    L.sfm_peer_alloc.argtypes = [i32, sz, C.POINTER(vp), vp]
    L.sfm_peer_open.argtypes = [i32, vp, C.POINTER(vp)]
    L.sfm_peer_close.argtypes = [i32, vp]
    L.sfm_peer_free.argtypes = [i32, vp]
    L.sfm_copy_async.argtypes = [vp, vp, sz, vp]
    L.sfm_probe_int8_mma.argtypes = [i32, i32, C.POINTER(C.c_float), C.POINTER(C.c_double)]
    L.sfm_debug_tc_tile.argtypes = [vp, vp, i32, vp, vp, vp]
    L.sfm_debug_refine_stats.argtypes = [i32, vp]
    for name in EXPORTS:
        if name not in ("sfm_last_error", "sfm_launch_count"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().sfm_last_error().decode("utf-8", "replace")
        raise SfmError(f"{what or 'libsfm_b200'} failed (code {rc}): {msg}")


def ptr(t):
    """data_ptr of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream_ptr(device=None):
    import torch

    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def launch_count() -> int:
    return int(lib().sfm_launch_count())
