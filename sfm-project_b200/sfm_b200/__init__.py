"""sfm_b200 -- host side of the B200-native matching + verification hot path.

Python here is plumbing only (device memory, streams, torch.distributed); all computation is in
lib/libsfm_b200.so (hand-written sm_100a CUDA behind the C ABI of include/sfm_b200.h).
"""
from . import _lib  # noqa: F401
from . import orb  # noqa: F401
from ._lib import SfmError, launch_count  # noqa: F401
from .bank import DescriptorBank, build_bank  # noqa: F401
from .matcher import MatchBatch, knn2, match_pairs, match_pairs_hamming, probe_int8_peak  # noqa: F401
from .pipeline import VerifiedPairs, get_plan, match_and_verify, match_and_verify_host  # noqa: F401
from .plan import HotPathPlan  # noqa: F401
from .ransac import VerifyBatch, verify_corr  # noqa: F401
from .tracks import Tracks, build_tracks_device  # noqa: F401
from .triangulate import TrackPoints, triangulate_tracks_device  # noqa: F401
from .pnp import AbsolutePoses, pnp_ransac_device, register_images_device  # noqa: F401
from .bundle import BundleResult, bundle_adjust_device  # noqa: F401
from .pairs import Pair, blocked_exhaustive_pairs, exhaustive_pairs, ordered_pairs, to_reference_pairs, windowed_pairs  # noqa: F401
