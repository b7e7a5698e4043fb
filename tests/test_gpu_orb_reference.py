"""GPU ORB extraction against cv2 on adversarial images: extreme contrast, tie storms, threshold steps, exact-axis angles,
edge sizes and feature budgets.

``tests/test_gpu_orb.py`` compares ``sfm_b200.orb`` with cv2 on the golden images and on cubic-upsampled noise at
``nfeatures = 500``.  Those inputs never reach several code paths; each family below is built to reach one of them:

* extreme contrast (checkerboards with 3, 5 and 8 px cells, random binary blocks, binary noise, 0/255 strokes on 0 and on
  255): Harris sums a + b above 2^24, where the float32 conversion in ``orb_harris_angle_kernel`` rounds and
  a b - c^2 cancels on straight edges;
* tie storms (periodic tiles of period 5, 7, 16 and 31 at 640 x 480 and 1920 x 1080): thousands of FAST keypoints with equal
  scores, so ``retainBest`` keeps far more than 2 n_level and ``OrbExtractor`` reallocates its candidate slots; more than
  1,024 keypoints per image, so the drop-in's Hamming slot bank rebuilds itself;
* threshold steps (piecewise-constant images in steps of 20 and of 21, and 20 / 21 steps on a constant background): FAST
  differences of exactly 21 (a corner at threshold 20) and exactly 20 (not a corner), and plateaus where the strict 3 x 3
  suppression rejects equal neighbours;
* symmetry (mirrored about a pixel column, and about a column and a row): intensity moments of exactly 0, so ``fastAtan2``
  returns exactly 0, 90, 180 or 270 degrees and the descriptor samples at rounded products of those angles' cos / sin;
* geometry: level-0 interiors of 1, 2 and 3 rows or columns (and the same at level 3), strips where the 31-pixel border
  empties some levels but not others, upper levels of 1 to 8 px (the blur's reflect101 at widths 1 to 3, resize tables that
  shrink 2 px to 1), widths that are no multiple of 32, sizes whose float32 level size w * (1 / 1.2^k) is exactly x.5 or
  is rounded differently from w / 1.2^k, and 3840 x 2160 and 7680 x 4320;
* natural texture (cubic-upsampled noise): the control.

The references are cv2 itself and, where one stage is isolated, ``oracle/orb_detect_oracle.py`` and ``oracle/orb_oracle.py``.
CPU tests check that every family builds what it claims and that the oracle equals cv2 on every family and budget; GPU tests
(marked, skipped one by one without a GPU) hold ``sfm_b200.orb`` and the drop-in to cv2 bit for bit.
"""
from __future__ import annotations

import ctypes as C
import functools
import os
import time

import numpy as np
import pytest

torch = pytest.importorskip("torch")
cv2 = pytest.importorskip("cv2")

from oracle import orb_detect_oracle as od  # noqa: E402
from oracle import orb_oracle as oo  # noqa: E402
from sfm_b200 import orb  # noqa: E402

HAS_CUDA = torch.cuda.is_available()
F32 = np.float32
BUDGETS = (1, 7, 8, 100, 500, 5000, 20000)
EXACT_AXES = (0.0, 90.0, 180.0, 270.0)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gpu_test(fn):
    """GPU tests are marked and skipped one by one: the CPU tests of this file must still run without one."""
    return pytest.mark.gpu(pytest.mark.skipif(not HAS_CUDA, reason="needs a GPU")(fn))


# ================================================================================================================ families

def textured(seed, h, w):
    """Natural texture (the control): cubic-upsampled noise plus pixel noise, as tests/test_gpu_orb.py builds it."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (h // 8 + 2, w // 8 + 2), dtype=np.uint8)
    img = cv2.resize(base, (w, h), interpolation=cv2.INTER_CUBIC)
    return np.clip(img.astype(int) + rng.normal(0, 10, (h, w)).astype(int), 0, 255).astype(np.uint8)


def checker(h, w, cell):
    """0/255 checkerboard: every corner is a saddle of full contrast, the Harris sums reach ~2.7e7 > 2^24."""
    y, x = np.mgrid[:h, :w]
    return (((y // cell + x // cell) & 1) * 255).astype(np.uint8)


def binary_blocks(seed, h, w, block=4):
    """Random 0/255 blocks: straight full-contrast edges, where a b - c^2 cancels in float32."""
    rng = np.random.default_rng(seed)
    b = rng.integers(0, 2, (h // block + 1, w // block + 1), dtype=np.uint8) * 255
    return np.ascontiguousarray(np.repeat(np.repeat(b, block, 0), block, 1)[:h, :w])


def binary_noise(seed, h, w):
    """Per-pixel 0/255 noise: the largest Harris sums (~3e7) and FAST scores of 254."""
    return np.random.default_rng(seed).integers(0, 2, (h, w), dtype=np.uint8) * 255


def strokes(seed, h, w, background):
    """0/255 line strokes (1 to 3 px) on a 0 or 255 background: full-contrast corners at line ends and crossings."""
    rng = np.random.default_rng(seed)
    img = np.full((h, w), background, np.uint8)
    for _ in range(120):
        p = (int(rng.integers(0, w)), int(rng.integers(0, h)))
        q = (int(rng.integers(0, w)), int(rng.integers(0, h)))
        cv2.line(img, p, q, 255 - background, int(rng.integers(1, 4)))
    return img


def periodic(seed, h, w, period):
    """A random uint8 tile of ``period`` px repeated: every FAST score repeats, so retainBest meets ties by the thousand."""
    tile = np.random.default_rng(seed).integers(0, 256, (period, period), dtype=np.uint8)
    return np.ascontiguousarray(np.tile(tile, (h // period + 1, w // period + 1))[:h, :w])


def steps(seed, h, w, step, block=6):
    """Piecewise-constant blocks whose levels are multiples of ``step`` (20 or 21): every FAST difference is a multiple of
    the step, so corners sit exactly at (21) or just below (20) the strict threshold."""
    rng = np.random.default_rng(seed)
    b = (rng.integers(0, 255 // step + 1, (h // block + 1, w // block + 1)) * step).astype(np.uint8)
    return np.ascontiguousarray(np.repeat(np.repeat(b, block, 0), block, 1)[:h, :w])


def step_rects(seed, h, w):
    """Rectangles 20 or 21 grey levels above or below a constant background of 100: the corners of the 21-rectangles are FAST
    corners with score 20 (the threshold), those of the 20-rectangles are rejected; their flat sides are suppression plateaus."""
    rng = np.random.default_rng(seed)
    img = np.full((h, w), 100, np.uint8)
    for _ in range(400):
        x, y = int(rng.integers(0, w - 12)), int(rng.integers(0, h - 12))
        dx, dy = int(rng.integers(4, 12)), int(rng.integers(4, 12))
        img[y: y + dy, x: x + dx] = 100 + int(rng.choice([-21, -20, 20, 21]))
    return img


def mirrored(seed, h, w, rows=False):
    """Texture mirrored about its middle pixel column (odd width) -- and about its middle row (odd height) when ``rows``: a
    keypoint on the axis has m10 = 0 (m01 = 0), so its angle is exactly 90 or 270 (0 or 180) degrees."""
    img = textured(seed, h, w)
    c = w // 2
    img[:, c + 1:] = img[:, :c][:, ::-1]
    if rows:
        r = h // 2
        img[r + 1:] = img[:r][::-1]
    return np.ascontiguousarray(img)


def _interior_size(level, extra):
    """Smallest image side whose ``level`` side is 2 * 31 + ``extra``: a level interior of exactly ``extra`` rows."""
    for s in range(1, 8192):
        if orb.level_sizes(s, s)[level][0] == 2 * od.EDGE + extra:
            return s
    raise AssertionError("no such size")


def _half_size(min_side=400):
    """Smallest side >= ``min_side`` whose float32 level size w * (1 / 1.2^k) is exactly x.5 with x even: round half to even
    and round half up disagree there."""
    for s in range(min_side, 8192):
        for k in range(1, 8):
            p = F32(F32(s) * F32(F32(1.0) / orb.level_scale(k)))
            if p - np.floor(p) == 0.5 and int(np.floor(p)) % 2 == 0:
                return s, k
    raise AssertionError("no such size")


def _div_size(min_side=400):
    """Smallest side >= ``min_side`` where round(w * float32(1 / 1.2^k)) != round(w / 1.2^k) for some level k."""
    for s in range(min_side, 8192):
        for k in range(1, 8):
            inv = F32(F32(1.0) / orb.level_scale(k))
            if np.rint(F32(F32(s) * inv)) != np.rint(F32(F32(s) / orb.level_scale(k))):
                return s, k
    raise AssertionError("no such size")


I1, I2, I3 = (_interior_size(0, e) for e in (1, 2, 3))                 # 63, 64, 65
L3 = [_interior_size(3, e) for e in (1, 2, 3)]                          # level 3 interior of 1, 2, 3 rows
HALF_SIDE, HALF_LEVEL = _half_size()
DIV_SIDE, DIV_LEVEL = _div_size()

# name -> (family, generator); the generators are seeded, so every run sees the same images
FAMILIES = {
    "checker3": ("contrast", lambda: checker(480, 640, 3)),
    "checker5": ("contrast", lambda: checker(480, 640, 5)),
    "checker8": ("contrast", lambda: checker(480, 640, 8)),
    "binary_blocks": ("contrast", lambda: binary_blocks(1, 480, 640)),
    "binary_noise": ("contrast", lambda: binary_noise(2, 480, 640)),
    "strokes_on_0": ("contrast", lambda: strokes(3, 480, 640, 0)),
    "strokes_on_255": ("contrast", lambda: strokes(4, 480, 640, 255)),
    "tile5_vga": ("ties", lambda: periodic(5, 480, 640, 5)),
    "tile7_vga": ("ties", lambda: periodic(7, 480, 640, 7)),
    "tile16_vga": ("ties", lambda: periodic(16, 480, 640, 16)),
    "tile31_vga": ("ties", lambda: periodic(31, 480, 640, 31)),
    "tile5_1080p": ("ties", lambda: periodic(5, 1080, 1920, 5)),
    "tile7_1080p": ("ties", lambda: periodic(7, 1080, 1920, 7)),
    "tile16_1080p": ("ties", lambda: periodic(16, 1080, 1920, 16)),
    "tile31_1080p": ("ties", lambda: periodic(31, 1080, 1920, 31)),
    "steps20": ("threshold", lambda: steps(20, 480, 640, 20)),
    "steps21": ("threshold", lambda: steps(21, 480, 640, 21)),
    "step_rects": ("threshold", lambda: step_rects(22, 480, 640)),
    "mirror_col": ("symmetry", lambda: mirrored(30, 481, 641)),
    "mirror_col_row": ("symmetry", lambda: mirrored(31, 481, 641, rows=True)),
    "interior1": ("geometry", lambda: textured(40, I1, 517)),
    "interior2": ("geometry", lambda: textured(41, 517, I2)),
    "interior3": ("geometry", lambda: textured(42, I3, I3)),
    "level3_interiors": ("geometry", lambda: textured(43, L3[0], L3[2])),
    "level3_interior2": ("geometry", lambda: textured(44, L3[1], 700)),
    "strip_63x2000": ("geometry", lambda: textured(45, 63, 2000)),
    "strip_2000x63": ("geometry", lambda: textured(46, 2000, 63)),
    "strip_70x900": ("geometry", lambda: textured(47, 70, 900)),
    "strip_900x70": ("geometry", lambda: textured(48, 900, 70)),
    "small_100x130": ("geometry", lambda: textured(49, 100, 130)),
    "tiny_4x700": ("geometry", lambda: textured(50, 4, 700)),
    "tiny_9x33": ("geometry", lambda: textured(51, 9, 33)),
    "tiny_30x37": ("geometry", lambda: binary_noise(52, 30, 37)),
    "odd_333x517": ("geometry", lambda: textured(53, 333, 517)),
    "half_size": ("geometry", lambda: textured(54, 480, HALF_SIDE)),
    "div_size": ("geometry", lambda: textured(55, DIV_SIDE, 640)),
    "uhd_4k": ("geometry", lambda: textured(56, 2160, 3840)),
    "uhd_8k": ("geometry", lambda: textured(57, 4320, 7680)),
    "textured_vga": ("texture", lambda: textured(60, 480, 640)),
    "textured_1080p": ("texture", lambda: textured(61, 1080, 1920)),
    "textured_odd": ("texture", lambda: textured(62, 481, 703)),
}
TOO_BIG_FOR_ORACLE = {"uhd_4k", "uhd_8k"}          # the numpy FAST stage holds 16 int32 planes of the image


@functools.lru_cache(maxsize=None)
def image(name):
    img = FAMILIES[name][1]()
    assert img.dtype == np.uint8 and img.ndim == 2 and img.flags.c_contiguous
    return img


def family(fam):
    return [n for n, (f, _) in FAMILIES.items() if f == fam]


@functools.lru_cache(maxsize=8)
def oracle_levels(name):
    """(pyramid, FAST candidates per level) of the oracle: independent of nfeatures, shared by every budget."""
    lv = oo.build_pyramid(image(name))
    return lv, od.level_candidates(lv)


@functools.lru_cache(maxsize=None)
def cv2_detect(name, nfeatures):
    kp, des = cv2.ORB_create(nfeatures=nfeatures).detectAndCompute(image(name), None)
    return kp, (np.zeros((0, 32), np.uint8) if des is None else des)


def rows_of(kp):
    return np.array([[k.pt[0], k.pt[1], k.size, k.angle, k.response, k.octave] for k in kp], F32).reshape(-1, 6)


def _arc_strength(img):
    """int32 [h, w]: the largest m such that 9 contiguous circle pixels all differ from the centre by >= m with one sign (0 in
    the 3-pixel frame).  A pixel is a FAST corner at threshold 20 iff this is >= 21; its score is this minus 1."""
    h, w = img.shape
    out = np.zeros((h, w), np.int32)
    I = img.astype(np.int32)
    c = I[3: h - 3, 3: w - 3]
    d = np.stack([c - I[3 + dy: h - 3 + dy, 3 + dx: w - 3 + dx] for dx, dy in od.CIRCLE], 0)
    best = np.zeros(c.shape, np.int32)
    for sgn in (1, -1):
        for s in range(16):
            best = np.maximum(best, np.minimum.reduce([sgn * d[(s + k) % 16] for k in range(9)]))
    out[3: h - 3, 3: w - 3] = best
    return out


# ======================================================================================================= CPU: the families

def test_level_sizes_equal_cv2_rounding():
    """cv2.ORB sizes level k as cvRound(w * (1.f / scale_k)) in float32 (round half to even).  Division by the scale rounds
    the other way on 281 (side, level) pairs below 8192; the half-size and division-size families are two of them, and on
    both the oracle's pyramid (built with the rule) gives cv2's keypoints while the division rule does not."""
    n_diff = 0
    for k in range(1, 8):
        s = np.arange(1, 8192)
        inv = F32(F32(1.0) / orb.level_scale(k))
        n_diff += int((np.rint((s.astype(F32) * inv).astype(F32)) != np.rint((s.astype(F32) / orb.level_scale(k)).astype(F32))).sum())
        assert [orb.level_sizes(int(v), 1)[k][0] for v in s[::97]] == [int(np.rint(F32(F32(v) * inv))) for v in s[::97]]
    assert n_diff == 281
    def half_up(v, k):
        return int(np.floor(F32(F32(v) * F32(F32(1.0) / orb.level_scale(k))) + F32(0.5)))

    def divided(v, k):
        return int(np.rint(F32(v) / orb.level_scale(k)))

    for name, other in (("half_size", half_up), ("div_size", divided)):
        img = image(name)
        h, w = img.shape
        sizes = orb.level_sizes(w, h)
        assert [lv.shape[::-1] for lv in oo.build_pyramid(img)] == sizes
        alt = [(w, h)] + [(other(w, k), other(h, k)) for k in range(1, 8)]
        assert alt != sizes, name
        prev, wrong = img, [img]
        for sz in alt[1:]:
            prev = cv2.resize(prev, sz, interpolation=cv2.INTER_LINEAR_EXACT)
            wrong.append(prev)
        ref = rows_of(cv2_detect(name, 5000)[0])
        assert np.array_equal(od.detect(img, 5000), ref), name
        assert not np.array_equal(od.detect(img, 5000, levels=wrong), ref), name
    p = F32(F32(HALF_SIDE) * F32(F32(1.0) / orb.level_scale(HALF_LEVEL)))
    assert p - np.floor(p) == 0.5 and orb.level_sizes(HALF_SIDE, 1)[HALF_LEVEL][0] == int(np.floor(p))      # half to even


def test_contrast_family_exceeds_2_24_in_harris():
    """Some kept keypoint of every extreme-contrast image has a + b > 2^24 (the float32 conversion of the Harris sums rounds)."""
    worst = {}
    for name in family("contrast"):
        lv, _ = oracle_levels(name)
        kp = od.detect(image(name), 500, levels=lv, candidates=oracle_levels(name)[1])
        best = 0
        for k in range(8):
            sel = kp[kp[:, 5] == k]
            if len(sel):
                x = np.rint(sel[:, 0] / orb.level_scale(k)).astype(np.int64)
                y = np.rint(sel[:, 1] / orb.level_scale(k)).astype(np.int64)
                best = max(best, int(od.harris_sums(lv[k], x, y).max()))
        worst[name] = best
    print(f"\nlargest Harris a + b of a kept keypoint (2^24 = {1 << 24}): {worst}")
    assert sum(v > (1 << 24) for v in worst.values()) >= 5 and max(worst.values()) > 2.5e7


def test_tie_family_overflows_candidates_and_slot_bank():
    """Every tie storm keeps more than 2 max(n_level) + 64 candidates on some level at some budget (OrbExtractor reallocates its
    slots) and, at nfeatures = 500, all but the sparsest keep more than 1,024 keypoints in all (the drop-in's slot bank
    rebuilds)."""
    report = {}
    for name in family("ties"):
        _, cand = oracle_levels(name)
        over = []
        for nf in BUDGETS:
            per = od.features_per_level(nf)
            sel = max(len(od.retain_best(cand[k][2], 2 * per[k])) for k in range(8))
            if sel > 2 * max(per) + 64:
                over.append(nf)
        n500 = len(cv2_detect(name, 500)[0])
        report[name] = (over, n500)
        assert over, name
        assert n500 > 1024 or name == "tile31_vga", name                 # a 31-px tile repeats only 20 x 15 times in 640 x 480
    print(f"\ntie storms: budgets that reallocate, keypoints at nfeatures=500: {report}")


def test_threshold_family_hits_20_and_21():
    """A FAST difference of exactly 21 at a kept corner (FAST score 20, the threshold, at a final keypoint) and of exactly 20 at
    a rejected one (arc strength 20: no corner); on the step images, corner plateaus that the strict 3 x 3 suppression
    removes whole (a local maximum with an equal neighbour)."""
    img = image("step_rects")
    strength, score = _arc_strength(img), od.fast_scores(img)
    kp = od.detect(img, 5000)
    lv0 = kp[kp[:, 5] == 0]
    x, y = lv0[:, 0].astype(int), lv0[:, 1].astype(int)
    assert (strength[y, x] == 21).any() and (score[y, x] == 20).any()
    assert (strength == 20).any() and not score[strength == 20].any()
    plateaus = {}
    for name in ("steps20", "steps21"):
        img = image(name)
        step = int(name[-2:])
        strength, score = _arc_strength(img), od.fast_scores(img)
        assert (strength == step).any() and (strength == 2 * step).any(), name
        assert bool(score[strength == 20].any()) is False and (score[strength == 21] == 20).all(), name
        P = np.pad(score, 1)
        nb = np.maximum.reduce([P[1 + dy: 1 + dy + score.shape[0], 1 + dx: 1 + dx + score.shape[1]]
                                for dy in (-1, 0, 1) for dx in (-1, 0, 1) if (dx, dy) != (0, 0)])
        plateaus[name] = int(((score > 0) & (score == nb)).sum())
        assert plateaus[name] > 0 and len(od.fast_keypoints(img)[0]) < int((score > 0).sum()), name
    print(f"\nthreshold steps: corner pixels on plateaus that the strict suppression rejects: {plateaus}")


def test_symmetry_family_gives_exact_axis_angles():
    """The column mirror gives keypoints at exactly 90 / 270 degrees; the column-and-row mirror also at exactly 0 / 180."""
    seen = {}
    for name in family("symmetry"):
        ang = rows_of(cv2_detect(name, 5000)[0])[:, 3]
        seen[name] = {a: int((ang == a).sum()) for a in EXACT_AXES}
        assert seen[name][90.0] + seen[name][270.0] > 0, name
    assert seen["mirror_col_row"][0.0] + seen["mirror_col_row"][180.0] > 0
    print(f"\nexact-axis angles at nfeatures=5000: {seen}")


def test_geometry_family_has_the_intended_level_interiors():
    assert (I1, I2, I3) == (63, 64, 65)
    for e, s in zip((1, 2, 3), L3):
        assert orb.level_sizes(s, s)[3][0] - 2 * od.EDGE == e
    assert orb.level_sizes(517, I1)[0][1] - 62 == 1 and orb.level_sizes(I2, 517)[0][0] - 62 == 2
    # the 31-pixel border empties some levels of the strips but not all
    for name in ("strip_70x900", "strip_900x70", "small_100x130", "level3_interiors"):
        _, cand = oracle_levels(name)
        counts = [len(c[0]) for c in cand]
        assert counts[0] > 0 and counts[-1] == 0, (name, counts)
    # upper levels of 1 to 8 px; the 4-row image reaches a 1-px level and 2-px levels resized to 1
    tops = {min(orb.level_sizes(*image(n).shape[::-1])[-1]) for n in ("tiny_4x700", "tiny_9x33", "tiny_30x37")}
    assert tops <= set(range(1, 9)) and 1 in tops
    assert [s[1] for s in orb.level_sizes(700, 4)] == [4, 3, 3, 2, 2, 2, 1, 1]
    assert any(image(n).shape[1] % 32 for n in family("geometry"))
    assert image("uhd_8k").shape == (4320, 7680) and image("uhd_4k").shape == (2160, 3840)


@pytest.mark.parametrize("name", [n for n in FAMILIES if n not in TOO_BIG_FOR_ORACLE])
def test_oracle_equals_cv2(name):
    """oracle/orb_detect_oracle.detect == cv2.ORB_create(nfeatures=n).detect, every field and the order, at every budget."""
    lv, cand = oracle_levels(name)
    for nf in BUDGETS:
        ref = rows_of(cv2_detect(name, nf)[0])
        got = od.detect(image(name), nf, levels=lv, candidates=cand)
        assert got.shape == ref.shape and np.array_equal(got, ref), (name, nf)


# =========================================================================================================== GPU: extraction

REALLOCATIONS = []


@pytest.fixture
def count_reallocations(monkeypatch):
    """Counts OrbExtractor._alloc_candidates calls that replace existing slots (the tie branch of detect)."""
    real = orb.OrbExtractor._alloc_candidates

    def wrapped(self, m):
        if hasattr(self, "m"):
            REALLOCATIONS.append((self.sizes[0], self.m, int(m)))
        return real(self, m)

    monkeypatch.setattr(orb.OrbExtractor, "_alloc_candidates", wrapped)
    return REALLOCATIONS


_EXTRACTORS = {}


def extractor(w, h, nfeatures):
    key = (w, h, nfeatures)
    if key not in _EXTRACTORS:
        if len(_EXTRACTORS) > 16:
            _EXTRACTORS.clear()
        _EXTRACTORS[key] = orb.OrbExtractor(w, h, nfeatures=nfeatures)
    return _EXTRACTORS[key]


def _assert_equal_cv2(img, nfeatures, e=None, what=""):
    h, w = img.shape
    e = extractor(w, h, nfeatures) if e is None else e
    kp, des = cv2.ORB_create(nfeatures=nfeatures).detectAndCompute(np.ascontiguousarray(img), None)
    rows, d = e.detect_and_compute(img)
    ref = rows_of(kp)
    assert rows.shape == ref.shape, f"{what} n={nfeatures}: {rows.shape[0]} keypoints, cv2 {ref.shape[0]}"
    bad = np.nonzero((rows != ref).any(1))[0]
    assert len(bad) == 0, f"{what} n={nfeatures}: {len(bad)} rows differ, first {bad[0]}: {rows[bad[0]]} vs {ref[bad[0]]}"
    assert np.array_equal(d.cpu().numpy(), des if des is not None else np.zeros((0, 32), np.uint8)), f"{what} n={nfeatures}: descriptors"
    return rows


@gpu_test
@pytest.mark.parametrize("fam", ["contrast", "ties", "threshold", "symmetry", "geometry", "texture"])
def test_detect_and_compute_equals_cv2(fam, count_reallocations):
    """OrbExtractor(w, h, nfeatures=n).detect_and_compute == cv2.ORB_create(nfeatures=n).detectAndCompute: keypoint rows in order
    and descriptors, for every image of the family and every budget."""
    t0 = time.perf_counter()
    before = len(count_reallocations)
    counts = {}
    for name in family(fam):
        img = image(name)
        counts[name] = [len(_assert_equal_cv2(img, nf, what=name)) for nf in BUDGETS]
    _EXTRACTORS.clear()
    angles = {}
    for name in family(fam):
        kp = rows_of(cv2_detect(name, 5000)[0])
        angles[name] = int(np.isin(kp[:, 3], EXACT_AXES).sum())
    print(f"\n{fam}: keypoints per budget {BUDGETS}: {counts}")
    print(f"{fam}: exact-axis angles at nfeatures=5000: {angles}; candidate reallocations: {len(count_reallocations) - before}; "
          f"{time.perf_counter() - t0:.1f} s")
    if fam == "ties":
        assert len(count_reallocations) > before


def _fast_level(e, k):
    from sfm_b200 import _lib

    w, h = e.sizes[k]
    _lib.check(_lib.lib().sfm_orb_fast_detect(_lib.ptr(e.raw[k]), w, h, w, 20, 31, _lib.ptr(e.score[k]), _lib.ptr(e.row_count[k]),
                                              C.c_void_p(e.totals.data_ptr() + 4 * k), _lib.ptr(e.xy[k]), _lib.ptr(e.resp[k]),
                                              _lib.current_stream_ptr()), "sfm_orb_fast_detect")
    n = int(e.totals[k].item())
    return e.xy[k][:n].cpu().numpy(), e.resp[k][:n].cpu().numpy()


@gpu_test
@pytest.mark.parametrize("name", family("contrast")[3:5] + family("symmetry") + ["tiny_4x700", "tiny_9x33", "tiny_30x37", "strip_70x900",
                                                                                   "half_size", "div_size"])
def test_stages_equal_cv2_and_oracle(name):
    """Stage by stage, so that a failure names its stage: raw and blurred levels == the cv2 resize / sepFilter2D chain (tiny
    levels included); sfm_orb_fast_detect == cv2.FastFeatureDetector_create(20, True) inside the border; Harris responses and
    angles of the selected candidates == the oracle's harris_responses / ic_angles."""
    img = image(name)
    h, w = img.shape
    e = orb.OrbExtractor(w, h, nfeatures=500)
    e.pyramid(img)
    torch.cuda.synchronize()
    g = cv2.getGaussianKernel(7, 2, cv2.CV_32F)
    lv = oo.build_pyramid(img)
    for k, ref in enumerate(lv):
        assert e.sizes[k] == ref.shape[::-1], f"level {k} size"
        assert np.array_equal(e.raw[k].cpu().numpy(), ref), f"level {k} pyramid"
        assert np.array_equal(e.blur[k].cpu().numpy(), cv2.sepFilter2D(ref, cv2.CV_8U, g, g, borderType=cv2.BORDER_REFLECT_101)), f"level {k} blur"
    for k, im in enumerate(lv):
        lh, lw = im.shape
        xy, resp = _fast_level(e, k)
        ref = [p for p in cv2.FastFeatureDetector_create(20, True).detect(im, None) if 31 <= p.pt[0] < lw - 31 and 31 <= p.pt[1] < lh - 31]
        assert xy.tolist() == [[int(p.pt[0]), int(p.pt[1])] for p in ref], f"level {k} FAST positions"
        assert resp.tolist() == [p.response for p in ref], f"level {k} FAST scores"
    e.detect(img, _pyramid_done=True)
    torch.cuda.synchronize()
    cand = e.cand_h.numpy()
    _, ocand = oracle_levels(name) if name not in TOO_BIG_FOR_ORACLE else (None, od.level_candidates(lv))
    for k, im in enumerate(lv):
        n = len(od.retain_best(ocand[k][2], 2 * e.per_level[k]))
        if n == 0:
            continue
        xy = cand[k, 0:2].reshape(-1)[: 2 * n].reshape(n, 2)
        hr, ang = cand[k, 2, :n].view(F32), cand[k, 3, :n].view(F32)
        assert np.array_equal(hr, od.harris_responses(im, xy[:, 0], xy[:, 1])), f"level {k} Harris"
        assert np.array_equal(ang, od.ic_angles(im, xy[:, 0], xy[:, 1])), f"level {k} angle"


@gpu_test
def test_describe_exact_axes_and_near_border_keypoints():
    """describe() == cv2 on the exact-axis keypoints of the symmetric family; keypoints placed 22 to 30 px from a level's border
    (which cv2's compute drops) are accepted and equal oracle/orb_oracle.describe; 21 px raises ValueError."""
    pat = np.load(os.path.join(GOLDEN, "orb_pattern.npz"))["pattern"]
    n_axes = 0
    for name in family("symmetry"):
        img = image(name)
        kp, des = cv2_detect(name, 5000)
        pick = [i for i, k in enumerate(kp) if k.angle in EXACT_AXES]
        got = orb.describe(img, [kp[i] for i in pick]).cpu().numpy()
        assert len(pick) and np.array_equal(got, des[pick]), name
        n_axes += len(pick)
    img = image("textured_vga")
    h, w = img.shape
    rows = []
    rng = np.random.default_rng(70)
    for k in range(4):
        lw, lh = orb.level_sizes(w, h)[k]
        sf = orb.level_scale(k)
        for dist in range(22, 31):
            for x, y in ((dist, lh // 2), (lw - 1 - dist, lh // 3), (lw // 2, dist), (lw // 3, lh - 1 - dist)):
                for ang in (0.0, 90.0, 180.0, 270.0, float(rng.uniform(0, 360))):
                    px, py = (F32(x) * sf, F32(y) * sf) if k else (F32(x), F32(y))
                    rows.append((px, py, ang, k))
    rows = np.array(rows, F32)
    rec, _ = orb.keypoint_records(rows)
    lvl = rows[:, 3].astype(int)
    lws = np.array([s[0] for s in orb.level_sizes(w, h)])[lvl]
    lhs = np.array([s[1] for s in orb.level_sizes(w, h)])[lvl]
    near = np.minimum.reduce([rec[:, 0], rec[:, 1], lws - 1 - rec[:, 0], lhs - 1 - rec[:, 1]])
    assert near.min() == 22 and near.max() == 30                     # the rounding lands the keypoints where they were placed
    got = orb.describe(img, rows).cpu().numpy()
    assert np.array_equal(got, oo.describe(img, rows, pat))
    for k in range(3):
        lw, lh = orb.level_sizes(w, h)[k]
        sf = orb.level_scale(k)
        for x, y in ((21, lh // 2), (lw - 22, lh // 2), (lw // 2, 21), (lw // 2, lh - 22)):
            px, py = (F32(x) * sf, F32(y) * sf) if k else (F32(x), F32(y))
            with pytest.raises(ValueError):
                orb.describe(img, np.array([[px, py, 0.0, k]], F32))
    print(f"\ndescribe: {n_axes} exact-axis keypoints and {len(rows)} keypoints 22-30 px from a level border equal the references")


@gpu_test
def test_extractor_reuse_and_input_kinds(count_reallocations):
    """One cached extractor per size runs textured -> binary -> blank -> periodic (reallocation) -> textured; every result
    equals cv2, and so do a CUDA-tensor input and a non-contiguous numpy view of a larger image."""
    before = len(count_reallocations)
    for h, w in ((480, 640), (1080, 1920)):
        e = orb.OrbExtractor(w, h, nfeatures=500)
        seq = [textured(80, h, w), binary_noise(81, h, w), np.zeros((h, w), np.uint8), periodic(82, h, w, 7), textured(83, h, w),
               binary_blocks(84, h, w), textured(80, h, w)]
        for i, img in enumerate(seq):
            _assert_equal_cv2(img, 500, e=e, what=f"reuse {w}x{h} image {i}")
        assert e.m > 2 * max(e.per_level) + 64                          # the slots grew and stayed grown
        img = seq[1]
        rows, d = e.detect_and_compute(torch.from_numpy(img).cuda())
        kp, des = cv2.ORB_create().detectAndCompute(img, None)
        assert np.array_equal(rows, rows_of(kp)) and np.array_equal(d.cpu().numpy(), des)
        big = textured(85, h + 37, 2 * w + 10)
        view = big[11: 11 + h, 5: 5 + 2 * w: 2]
        assert not view.flags.c_contiguous
        _assert_equal_cv2(view, 500, e=e, what=f"view {w}x{h}")
    assert len(count_reallocations) - before >= 2


def _nearest_ties(d1, d2):
    """Number of query rows whose smallest Hamming distance is reached by two or more train rows (popcounts as a float32
    GEMM of unpacked bits: exact, every value is at most 256)."""
    a = np.unpackbits(d1, axis=1).astype(F32)
    b = np.unpackbits(d2, axis=1).astype(F32)
    D = a.sum(1)[:, None] + b.sum(1)[None, :] - 2 * (a @ b.T)
    return int(((D == D.min(1, keepdims=True)).sum(1) > 1).sum())


@gpu_test
def test_dropin_on_ties_and_binary_equals_reference(monkeypatch, count_reallocations):
    """feature_matching.extract_and_match on periodic and binary pairs (> 1,024 keypoints, many equal-distance Hamming ties)
    == cv2_ref.orb_extract + cv2_ref.hamming_crosscheck, stably sorted by distance, prefix < 26; with GPU detection and with
    cv2's detection + GPU descriptors."""
    import feature_matching as fm
    from oracle import cv2_ref

    rebuilds = []
    real = fm._SlotBank

    class Counting(real):
        def __init__(self, *a, **k):
            rebuilds.append(a)
            super().__init__(*a, **k)

    monkeypatch.setattr(fm, "_SlotBank", Counting)
    t1, b1 = periodic(90, 480, 640, 16), binary_blocks(93, 480, 640)
    pairs = [(b1, np.ascontiguousarray(np.roll(b1, 9, 1))), (t1, np.ascontiguousarray(np.roll(t1, (3, 5), (0, 1)))),
             (periodic(91, 480, 640, 7), periodic(92, 480, 640, 7)), (t1, binary_noise(94, 480, 640))]
    report = []
    for det in (True, False):
        monkeypatch.setattr(fm, "GPU_DESCRIPTORS", True)
        monkeypatch.setattr(fm, "GPU_DETECTION", det)
        fm._ORB_CACHE.clear()
        fm._SEEN.clear()
        fm._SLOTS = None
        n0 = len(rebuilds)
        for a, b in pairs:
            m = fm.extract_and_match(a, b)
            (k1, d1), (k2, d2) = cv2_ref.orb_extract(a), cv2_ref.orb_extract(b)
            q, t, d = cv2_ref.hamming_crosscheck(d1, d2)
            o = np.argsort(d, kind="stable")
            keep = o[d[o] < 26]
            assert [x.queryIdx for x in m] == q[keep].tolist() and [x.trainIdx for x in m] == t[keep].tolist()
            assert [x.distance for x in m] == d[keep].tolist()
            report.append((det, len(k1), len(k2), len(m), _nearest_ties(d1, d2)))
        assert len(rebuilds) - n0 >= 2                                   # the first bank, then the rebuild above 1,024 rows
    assert max(r[1] for r in report) > 1024 and max(r[4] for r in report) > 100
    print(f"\ndrop-in (GPU detection, keypoints 1, keypoints 2, matches, queries with a tied nearest row): {report}; "
          f"slot banks built: {len(rebuilds)}")
