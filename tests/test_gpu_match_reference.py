"""The L2 and Hamming matchers against an exact integer reference, on adversarial descriptors, at 32,768 features per image
and in banks whose descriptor section passes 2^31 and 2^32 bytes.

The other matcher tests compare the kernels with ``oracle/match_oracle.py`` (which builds the whole int64 distance matrix, too
big at 32,768^2), with cv2 on benign SIFT-like rows, or with each other (the fused refinement against the kNN-table path:
both read the same sweep records, so a wrong record passes both).  The reference here is written from the definitions:

* ``knn2_ref`` and ``filter_ref`` (in ``oracle/exact_match.py``, which tests/test_gpu_pipeline_reference.py shares):

  - ``knn2_ref``: squared L2 as |a|^2 + |b|^2 - 2 a.b with the dot products as a float64 GEMM in row chunks (exact: every
    value is an integer below 2^53), top-2 by the int64 key D * 2^16 + trainIdx, so the lowest index wins a tie without
    relying on any library's argmin;
  - ``filter_ref``: Lowe's test as ``float64(sqrt_f32(D1)) < ratio * float64(sqrt_f32(D2))`` (cv2_f32) or
    ``D1 den^2 < D2 num^2`` with ``Fraction(ratio).limit_denominator(1024)`` (exact_int), the strict bound D1 < max_d, the
    mutual check on the reverse table's nearest; rows in ascending queryIdx;
* ``hamming_ref``: popcount distances through ``unpackbits`` and a float32 GEMM (exact: values <= 256), cross-check with
  lowest-index ties in both directions, stable sort by distance, the ``< max_distance`` prefix;
* ``tile_model``: the sweep's bookkeeping restated from DESIGN.md §4 K2 on exact accumulators acc = a_s.b_s + H0 -
  floor(|b_s|^2 / 2) (per-tile maxima M1 >= M2 >= M3): which rows must be brute-forced (M2 == M3 and a fourth tile reaches
  M3) and the prefilter's distance bounds.  It predicts the refinement's brute-force counter and the prefilter's blanks, so
  the coverage of the tie4 path and of the prefilter is asserted, not assumed.

Its CPU tests (no ``gpu`` mark) pin the reference to cv2 (``BFMatcher(NORM_L2).knnMatch(k=2)`` + the ratio idiom,
``BFMatcher(NORM_HAMMING, crossCheck=True)``), to the numpy oracle and to the golden files, and check that every
adversarial family builds what it claims.  The families, each aimed at one argument of the exactness proof:

* cross-tile ties: exact duplicates of a query's nearest row in 2, 3, 4, 5 and 8 tiles (tile 0 and the last, partial tile
  among them), the two-letter alphabet at 32,768 x 32,768, and a tile outside the top three whose maximum equals M3 but
  not M2 (must not be brute-forced);
* parity: train rows b and b + e_k with a_k = b_k = 0 (equal accumulators, distances one apart), in different tiles and
  inside one 8-row sub-group;
* ratio boundaries: queries at the offset-zero vector (D = |b_s|^2) against rows of chosen norms in chosen tiles, at
  16 D1 == 9 D2 style boundaries and one unit either side, for ratios 0.5, 0.75, 0.8 and 0.999, so that the prefilter and
  the fused refinement's early stop (dlo = C - 2 M2 against dlo + 1) decide on both sides;
* extreme norms (rows all 0, all 255, alternating 0/255, values in {127, 128, 129}) and ragged images of 0 to 32,768 rows,
  in both directions of every pair and as self pairs.
"""
from __future__ import annotations

import ctypes as C
import os
import time
from math import isqrt
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")
cv2 = pytest.importorskip("cv2")

from oracle import match_oracle as mo  # noqa: E402
from oracle.exact_match import _step, _tensor, filter_ref, knn2_ref, ratio_pass  # noqa: E402,F401
from sfm_b200 import synth  # noqa: E402

HAS_CUDA = torch.cuda.is_available()


def gpu_test(fn):
    """GPU tests are marked and skipped one by one: the reference's own CPU tests in this file must still run without one."""
    return pytest.mark.gpu(pytest.mark.skipif(not HAS_CUDA, reason="needs a GPU")(fn))


N = 32768                     # BASELINE configs[3] features per image: 256 train tiles, 128 query units
TILE = 128                    # train rows per sweep tile
H0 = 1 << 20                  # the K-extension offset of the accumulators (DESIGN.md §3)


# ====================================================================================================== exact reference

def hamming_ref(A, B, max_distance=26, device=None):
    """cv2.BFMatcher(NORM_HAMMING, crossCheck=True).match -> stable sort by distance -> prefix distance < max_distance."""
    z = np.zeros(0, np.int32)
    if len(A) == 0 or len(B) == 0:
        return z, z.copy(), z.copy()
    dev = device or (B.device if isinstance(B, torch.Tensor) else "cpu")
    a = _tensor(np.unpackbits(np.asarray(_tensor(A).cpu()), axis=1), dev).float()
    b = _tensor(np.unpackbits(np.asarray(_tensor(B).cpu()), axis=1), dev).float()
    nq, nt = a.shape[0], b.shape[0]
    na, nb = a.sum(1), b.sum(1)
    tidx = torch.arange(nt, device=a.device, dtype=torch.int64)
    row_key = torch.empty(nq, dtype=torch.int64, device=a.device)
    col_key = torch.full((nt,), 1 << 62, dtype=torch.int64, device=a.device)
    step = _step(nt, a.device)
    for r0 in range(0, nq, step):
        r1 = min(nq, r0 + step)
        H = (na[r0:r1, None] + nb[None, :] - 2.0 * (a[r0:r1] @ b.T)).to(torch.int64)     # popcounts, exact in float32
        row_key[r0:r1] = (H * 65536 + tidx[None, :]).min(1).values
        qidx = torch.arange(r0, r1, device=a.device, dtype=torch.int64)
        col_key = torch.minimum(col_key, (H * 65536 + qidx[:, None]).min(0).values)
    rk, ck = row_key.cpu().numpy(), col_key.cpu().numpy()
    nn12, d12, nn21 = rk & 0xFFFF, rk >> 16, ck & 0xFFFF
    q = np.nonzero(nn21[nn12] == np.arange(nq))[0]
    t, d = nn12[q], d12[q]
    order = np.argsort(d, kind="stable")
    q, t, d = q[order], t[order], d[order]
    n = int(np.searchsorted(d, max_distance, side="left"))
    return q[:n].astype(np.int32), t[:n].astype(np.int32), d[:n].astype(np.int32)


def tile_model(A, B, device=None):
    """The sweep's per-row bookkeeping (DESIGN.md §4 K2) on exact accumulators.  Returns numpy (brute, lo1, hi2):
    brute = the row must be brute-forced (M2 == M3 and at least four tiles reach M3); lo1 = max(C - 2 M1, 0) and
    hi2 = C - 2 M2 + 1 are the prefilter's bounds on D1 and D2 (hi2 = -1 when the image has a single tile)."""
    B = _tensor(B, device)
    A = _tensor(A, B.device)
    nq, nt = A.shape[0], B.shape[0]
    brute = np.zeros(nq, bool)
    lo1 = np.zeros(nq, np.int64)
    hi2 = np.full(nq, -1, np.int64)
    if nq == 0 or nt == 0:
        return brute, lo1, hi2
    b = B.double() - 128.0
    bias = H0 - torch.floor((b * b).sum(1) / 2.0)
    tiles = (nt + TILE - 1) // TILE
    pad = tiles * TILE - nt
    step = _step(tiles * TILE, B.device)
    for r0 in range(0, nq, step):
        a = A[r0: r0 + step].double() - 128.0
        acc = a @ b.T + bias[None, :]
        if pad:
            acc = torch.nn.functional.pad(acc, (0, pad), value=float("-inf"))
        tm = acc.view(acc.shape[0], tiles, TILE).amax(2)
        top = torch.topk(tm, min(3, tiles), dim=1).values
        c = (a * a).sum(1) + 2.0 * H0
        sl = slice(r0, r0 + acc.shape[0])
        lo1[sl] = torch.clamp(c - 2.0 * top[:, 0], min=0).cpu().numpy().astype(np.int64)
        if tiles >= 2:
            hi2[sl] = (c - 2.0 * top[:, 1] + 1.0).cpu().numpy().astype(np.int64)
        if tiles >= 3:
            m3 = top[:, 2:3]
            brute[sl] = ((top[:, 1:2] == m3)[:, 0] & ((tm >= m3).sum(1) >= 4)).cpu().numpy()
    return brute, lo1, hi2


def prefilter_blanks(model, ratio, mode):
    """Rows the sweep's prefilter must blank: their distance bounds already fail the ratio test."""
    _, lo1, hi2 = model
    return (hi2 >= 0) & ~ratio_pass(lo1, np.maximum(hi2, 0), ratio, mode)


# ====================================================================================================== adversarial families

ZERO_ROWS = np.r_[0:8, 256, 20000:20008]          # offset-zero query rows (all bytes 128): D = |b_s|^2 against any train row
RATIO_BOUNDARY = {0.5: (9, 36), 0.75: (9, 16), 0.8: (64, 100), 0.999: (998001, 1000000)}   # D1 den^2 == D2 num^2, D2 even
BOUNDARY_DELTAS = [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)]
BOUNDARY_TILES = [(200, 3), (3, 200)]              # (tile of the nearest, tile of the second nearest)
TILE_CASES = {                                      # name: ((D, tile) of the planted rows, brute-forced by the proof?)
    "m3_tie_below_m2": ([(100, 10), (140, 20), (200, 30), (200, 40), (200, 50)], False),
    "use3": ([(100, 10), (140, 20), (140, 30)], False),
    "use3_parity": ([(100, 10), (141, 20), (140, 30)], False),
    "tie4_parity": ([(100, 10), (141, 20), (140, 30), (141, 40)], True),
    "second_in_first_tile": ([(100, 200), (120, 200), (121, 5)], False),
    "nearest_ties_across_tiles": ([(101, 3), (100, 200)], False),
}
RAGGED = (0, 1, 2, 127, 128, 129, 255, 256, 257, 32767, 32768)


def row_with_norm(rng, d):
    """uint8 row 128 + v with |v|^2 == d (greedy squares on distinct coordinates, random signs)."""
    v = np.zeros(128, np.int64)
    coords = rng.permutation(128)
    rem, i = int(d), 0
    while rem:
        s = min(isqrt(rem), 127)
        v[coords[i]] = s if rng.random() < 0.5 else -s
        rem -= s * s
        i += 1
    assert (v * v).sum() == d
    return (v + 128).astype(np.uint8)


def far_filler(rng, n):
    """Rows with every |b - 128| >= 111: offset norms >= 1.57e6, farther from an offset-zero query than any planted row."""
    v = rng.integers(0, 34, (n, 128))
    return np.where(v < 17, v, v + 222).astype(np.uint8)


def scenario_train(rng, planted, n=N):
    B = far_filler(rng, n)
    used = set()
    for d, tile in planted:
        while True:
            r = tile * TILE + int(rng.integers(0, TILE))
            if r not in used:
                break
        used.add(r)
        B[r] = row_with_norm(rng, d)
    return B


def zero_query_image(rng, n=N):
    A = synth.sift_like(rng, n)
    A[ZERO_ROWS] = 128
    return A


def boundary_scenarios():
    """(ratio, delta, tiles, planted) for every ratio-test boundary case."""
    out = []
    for ratio, (d1, d2) in RATIO_BOUNDARY.items():
        for dd in BOUNDARY_DELTAS:
            for tn, ts in BOUNDARY_TILES:
                out.append((ratio, dd, (tn, ts), [(d1 + dd[0], tn), (d2 + dd[1], ts)]))
    return out


def tie_family(rng, nq=N, nt=N - 1):
    """Queries whose nearest train row is duplicated in k = 2, 3, 4, 5 and 8 different tiles (tile 0 and the last, partial
    tile among them; sometimes a second copy in the same tile), queried by an exact copy and by two noisy observations.
    Returns (A, B, {k: planted query rows})."""
    B = synth.sift_like(rng, nt)
    A = synth.sift_like(rng, nq)
    A[:8000] = synth.observe(rng, B[rng.permutation(nt)[:8000]])
    last = (nt - 1) // TILE
    planted, q, used = {}, 8000, set()
    for k in (2, 3, 4, 5, 8):
        planted[k] = []
        for g in range(8):
            tiles = rng.choice(np.arange(1, last), k, replace=False)
            if g % 2 == 0:
                tiles[0] = 0
            if g % 4 < 2:
                tiles[-1] = last
            x = synth.sift_like(rng, 1)[0]
            for tl in tiles:
                free = [r for r in range(tl * TILE, min(nt, tl * TILE + TILE)) if r not in used]
                rows = rng.choice(free, 2 if g == 7 else 1, replace=False)    # group 7: two copies in every tile
                used.update(rows.tolist())
                B[rows] = x
            A[q] = x
            A[q + 1: q + 3] = synth.observe(rng, np.stack([x, x]), sigma=3.0)
            planted[k].extend([q, q + 1, q + 2])
            q += 3
    return A, B, planted


def two_letter_family(rng, n=N):
    """test_gpu_matcher's two-letter alphabet at 32,768 x 32,768: distances collide all over the image; plus exact copies and
    copies one unit away."""
    def draw(m):
        d = np.where(rng.random((m, 128)) < 0.2, 65, 0).astype(np.uint8)
        d[::7] = np.where(rng.random((len(d[::7]), 128)) < 0.2, 64, 1).astype(np.uint8)
        return d

    a, b = draw(n), draw(n)
    perm = rng.permutation(n)
    b[:8000] = a[perm[:8000]]
    b[8000:12000] = a[perm[8000:12000]]
    b[8000 + np.arange(4000), rng.integers(0, 128, 4000)] ^= 1
    return a, b


def parity_family(rng, n=N, m=600):
    """Query a with a_k = 128 (offset 0); train b near a with b_k = 128 and |b_s|^2 even, and b' = b + e_k: equal accumulators,
    D(b') = D(b) + 1.  b' always gets the lower index (a parity-blind tie break would pick it).  Placement by i % 3: one
    8-row sub-group, different tiles.  Returns (A, B, rows [m, 3] = (query, b row, b' row))."""
    A = synth.sift_like(rng, n)
    B = synth.sift_like(rng, n)
    groups = iter(rng.permutation(n // 8))
    rows = []
    for i in range(m):
        k = int(rng.integers(0, 128))
        A[i, k] = 128
        b = synth.observe(rng, A[i:i + 1], sigma=4.0)[0].astype(np.int64)
        b[k] = 128
        j = (k + 1) % 128
        while ((b - 128) ** 2).sum() % 2:
            b[j] = b[j] + 1 if b[j] < 255 else b[j] - 1
        g1 = next(groups)
        if i % 3 == 0:
            lo, hi = np.sort(rng.choice(8, 2, replace=False))
            rb2, rb = 8 * g1 + lo, 8 * g1 + hi
        else:
            g2 = next(groups)
            while g2 * 8 // TILE == g1 * 8 // TILE:
                g2 = next(groups)
            lo_g, hi_g = min(g1, g2), max(g1, g2)
            rb2, rb = 8 * lo_g + int(rng.integers(8)), 8 * hi_g + int(rng.integers(8))
        B[rb] = b.astype(np.uint8)
        b[k] = 129
        B[rb2] = b.astype(np.uint8)
        rows.append((i, rb, rb2))
    return A, B, np.array(rows)


def extreme_rows(rng, m):
    """m rows of each extreme kind: all 0, all 255, alternating 0/255 (both phases), values in {127, 128, 129}."""
    alt = np.tile(np.array([0, 255], np.uint8), 64)
    kinds = [np.zeros(128, np.uint8), np.full(128, 255, np.uint8), alt, alt[::-1].copy()]
    out = [np.stack([k] * m) for k in kinds]
    out.append(rng.integers(127, 130, (m, 128)).astype(np.uint8))
    return np.concatenate(out)


def ragged_images(rng, sizes=RAGGED):
    """SIFT-like images of the given sizes with half their rows observed from a shared pool, extreme rows mixed in and one
    duplicated row; images of fewer than five rows are all extreme rows."""
    pool = synth.sift_like(rng, 4096)
    out = []
    for n in sizes:
        if n < 5:
            out.append(extreme_rows(rng, 1)[:n].copy())
            continue
        d = synth.sift_like(rng, n)
        d[: n // 2] = synth.observe(rng, pool[rng.integers(0, 4096, n // 2)])
        ex = extreme_rows(rng, max(1, n // 64))
        d[rng.choice(n, len(ex), replace=False)] = ex
        d[n - 1] = d[0]
        out.append(d)
    return out


def l2_family_images(seed=2024):
    """Every L2 image of the adversarial bank and the pair groups over it: {family: [(query image, train image), ...]}."""
    rng = np.random.default_rng(seed)
    imgs, names = [], []

    def add(name, d):
        imgs.append(d)
        names.append(name)
        return len(imgs) - 1

    tq, tt, tie_rows = tie_family(rng)
    tq, tt = add("tie_q", tq), add("tie_t", tt)
    la, lb = two_letter_family(rng)
    la, lb = add("letters_a", la), add("letters_b", lb)
    pq, pt, parity_rows = parity_family(rng)
    pq, pt = add("parity_q", pq), add("parity_t", pt)
    zq = add("zero_q", zero_query_image(rng))
    z1 = add("zero_1", np.full((1, 128), 128, np.uint8))          # one offset-zero row: refinement work fully predictable
    bnd = [(add(f"bnd_{r}_{dd}_{tl}", scenario_train(rng, planted)), r, dd, tl, planted)
           for r, dd, tl, planted in boundary_scenarios()]
    cases = {name: add(f"case_{name}", scenario_train(rng, planted)) for name, (planted, _) in TILE_CASES.items()}
    rag = [add(f"ragged_{n}", d) for n, d in zip(RAGGED, ragged_images(rng))]
    both = lambda i, j: [(i, j), (j, i)]  # noqa: E731
    groups = {
        "ties": both(tq, tt) + [(tt, tt), (tq, tq)],
        "two_letter": both(la, lb) + [(la, la)],
        "parity": both(pq, pt) + [(pt, pt)],
        "boundary": [p for b in bnd for p in both(zq, b[0])],
        "tile_cases": [p for i in cases.values() for p in both(zq, i)],
        "ragged": [(i, j) for i in rag for j in rag],
    }
    xys = [rng.uniform(-1000.0, 5000.0, (len(d), 2)).astype(np.float32) for d in imgs]
    meta = SimpleNamespace(tie_rows=tie_rows, parity_rows=parity_rows, zq=zq, z1=z1, bnd=bnd, cases=cases, tq=tq, tt=tt, pq=pq, pt=pt)
    return imgs, names, xys, groups, meta


def hamming_family_images(seed=77):
    rng = np.random.default_rng(seed)
    b = rng.integers(0, 256, (N, 32), dtype=np.uint8)
    a = rng.integers(0, 256, (N, 32), dtype=np.uint8)
    perm = rng.permutation(N)
    a[:12000] = b[perm[:12000]] ^ np.packbits(rng.random((12000, 256)) < 0.03, axis=1)     # near copies
    a[12000:13000] = b[perm[12000:13000]]                                                  # exact copies: distance 0
    b[perm[20000:20500]] = b[perm[:500]]                     # duplicate train rows: row argmins tie
    a[13000:13500] = a[:500]                                 # duplicate query rows: column argmins tie
    a[13500:13600] = 0
    b[perm[21000:21050]] = 0                                 # all-zero rows on both sides
    small = [rng.integers(0, 256, (n, 32), dtype=np.uint8) for n in (1, 257, 32767)]
    small[1][:100] = b[perm[600:700]]
    small[2][:5000] = a[rng.permutation(N)[:5000]] ^ np.packbits(rng.random((5000, 256)) < 0.02, axis=1)
    imgs = [a, b] + small
    pairs = [(0, 1), (1, 0), (0, 0), (1, 1), (2, 1), (1, 2), (3, 4), (4, 3), (4, 0), (0, 4), (2, 2)]
    return imgs, pairs


# ====================================================================================================== CPU: pin the reference

def _planted_pair(rng, n1, n2):
    B = synth.sift_like(rng, n2)
    A = synth.sift_like(rng, n1)
    k = min(n1, n2) // 2
    A[:k] = synth.observe(rng, B[rng.permutation(n2)[:k]])
    return A, B


def test_knn2_and_filter_reference_equal_cv2_knnmatch():
    from oracle import cv2_ref

    rng = np.random.default_rng(1)
    A, B = _planted_pair(rng, 3000, 2500)
    B[100:110] = B[7]                          # exact duplicate train rows across tiles
    B[2400] = B[7]
    A[0] = B[7]
    A[1:20] = synth.observe(rng, np.repeat(B[7:8], 19, 0), sigma=2.0)
    A[20], A[21] = 0, 255
    knn = knn2_ref(A, B)
    i1, d1, i2, d2 = cv2_ref.l2_knn2(A, B)
    assert np.array_equal(knn[:, 0], i1) and np.array_equal(knn[:, 2], i2)
    assert np.array_equal(np.sqrt(knn[:, 1].astype(np.float32)), d1) and np.array_equal(np.sqrt(knn[:, 3].astype(np.float32)), d2)
    assert knn[0].tolist() == [7, 0, 100, 0]
    for ratio in (0.5, 0.75, 0.8, 0.999):
        q, t, d = filter_ref(knn, ratio=ratio, mode="cv2_f32")
        cq, ct, cd = cv2_ref.l2_ratio_match(A, B, ratio)
        assert np.array_equal(q, cq) and np.array_equal(t, ct) and np.array_equal(np.sqrt(d.astype(np.float32)), cd)
    q, t, _ = filter_ref(knn, knn2_ref(B, A), ratio=None, mutual=True)
    cq, ct, _ = cv2_ref.l2_crosscheck(A, B)
    assert np.array_equal(q, cq) and np.array_equal(t, ct)


def test_hamming_reference_equals_cv2_crosscheck():
    from oracle import cv2_ref

    rng = np.random.default_rng(2)
    b = rng.integers(0, 256, (1500, 32), dtype=np.uint8)
    a = rng.integers(0, 256, (1200, 32), dtype=np.uint8)
    a[:600] = b[rng.permutation(1500)[:600]] ^ np.packbits(rng.random((600, 256)) < 0.04, axis=1)
    b[1400:1450] = b[:50]                                    # duplicate train rows
    a[700:750] = a[:50]                                      # duplicate query rows
    for X, Y in ((a, b), (b, a), (a, a)):
        q, t, d = hamming_ref(X, Y, 26)
        cq, ct, cd = cv2_ref.hamming_crosscheck(X, Y)
        order = np.argsort(cd, kind="stable")
        n = int(np.searchsorted(cd[order], 26, side="left"))
        assert np.array_equal(q, cq[order][:n]) and np.array_equal(t, ct[order][:n]) and np.array_equal(d, cd[order][:n])
        assert len(q) > 100


@pytest.mark.parametrize("n1,n2", [(300, 257), (1, 50), (64, 1), (5, 0), (0, 7), (129, 129)])
def test_references_equal_the_numpy_oracle(n1, n2):
    rng = np.random.default_rng(n1 * 1000 + n2)
    A, B = _planted_pair(rng, n1, n2)
    if n2 > 3:
        B[n2 - 1] = B[0]
    knn = knn2_ref(A, B)
    assert np.array_equal(knn, np.stack(mo.l2_knn2(A, B), 1))
    rev = knn2_ref(B, A)
    for ratio, mode, mutual in [(0.75, "cv2_f32", False), (0.8, "exact_int", False), (0.75, "cv2_f32", True), (None, "cv2_f32", True)]:
        got = filter_ref(knn, rev, ratio=ratio, mode=mode, mutual=mutual)
        want = mo.match_l2(A, B, ratio=ratio, ratio_mode=mode, mutual=mutual)
        assert all(np.array_equal(x, y) for x, y in zip(got, want))
    ha = rng.integers(0, 256, (n1, 32), dtype=np.uint8)
    hb = rng.integers(0, 256, (n2, 32), dtype=np.uint8)
    if n1 and n2:
        ha[: min(n1, n2) // 2] = hb[: min(n1, n2) // 2] ^ 1
    for md in (0, 1, 26, 257):
        got = hamming_ref(ha, hb, md)
        want = mo.match_hamming_reference(ha, hb, md)
        assert all(np.array_equal(x, y) for x, y in zip(got, want))


def test_references_reproduce_the_golden_files(golden_dir):
    g = np.load(os.path.join(golden_dir, "cv2_l2_knn.npz"))
    knn = knn2_ref(g["A"], g["B"])
    assert knn[:, 0].tolist() == g["idx1"].tolist() and knn[:, 2].tolist() == g["idx2"].tolist()
    assert np.sqrt(knn[:, 1].astype(np.float32)).tolist() == g["d1"].tolist()
    assert np.sqrt(knn[:, 3].astype(np.float32)).tolist() == g["d2"].tolist()
    q, t, d = filter_ref(knn, ratio=0.75, mode="cv2_f32")
    assert q.tolist() == g["ratio_q"].tolist() and t.tolist() == g["ratio_t"].tolist()
    assert np.sqrt(d.astype(np.float32)).tolist() == g["ratio_d"].tolist()
    q, t, d = filter_ref(knn, knn2_ref(g["B"], g["A"]), ratio=None, mutual=True)
    assert q.tolist() == g["cross_q"].tolist() and t.tolist() == g["cross_t"].tolist()
    qi = filter_ref(knn, ratio=0.75, mode="exact_int")[0]
    assert sorted(set(g["ratio_q"].tolist()) - set(qi.tolist())) == [202, 203]       # 16 D1 == 9 D2 rows
    h = np.load(os.path.join(golden_dir, "ref_orb_hamming.npz"))
    n = h["images"].shape[0]
    for i in range(n):
        for j in range(n):
            if i != j:
                q, t, d = hamming_ref(h[f"des{i}"], h[f"des{j}"], 26)
                assert q.tolist() == h[f"q_{i}_{j}"].tolist() and t.tolist() == h[f"t_{i}_{j}"].tolist()
                assert d.astype(np.float32).tolist() == h[f"d_{i}_{j}"].tolist()


def test_tile_model_follows_the_definition():
    """The model's flags on hand-built accumulators: a fourth tile tying M3 == M2 forces brute force, a tie below M2 does not."""
    rng = np.random.default_rng(3)
    zero = np.full((1, 128), 128, np.uint8)
    for name, (planted, brute) in TILE_CASES.items():
        B = scenario_train(rng, planted)
        got, lo1, hi2 = tile_model(zero, B)
        assert got[0] == brute, name
        ds = sorted(d for d, _ in planted)
        knn = knn2_ref(zero, B)[0]
        assert (knn[1], knn[3]) == (ds[0], ds[1]), name
        assert lo1[0] <= knn[1] and hi2[0] >= knn[3]                 # the prefilter's bounds hold
    assert not tile_model(zero, scenario_train(rng, [(5, 0)], n=TILE))[0][0]


def test_families_build_what_they_claim():
    """Each generator plants what its docstring says, checked with the reference (planted rows only: cheap on a CPU)."""
    rng = np.random.default_rng(4)
    A, B, planted = tie_family(rng)
    copies = {k: [] for k in planted}
    for k, rows in planted.items():
        model = tile_model(A[rows], B)[0]
        assert model.all() if k >= 4 else not model.any(), k
        knn = knn2_ref(A[rows], B)
        assert (knn[:, 1] == knn[:, 3]).all() and (knn[::3, 1] == 0).all()       # nearest duplicated: D1 == D2
        copies[k] = (np.nonzero((B == A[rows[0]]).all(1))[0] // TILE)
    assert len(set(copies[4])) == 4 and 0 in copies[2] and (len(B) - 1) // TILE in copies[2]
    A, B, rows = parity_family(rng, m=60)
    knn = knn2_ref(A[rows[:, 0]], B)
    assert np.array_equal(knn[:, 0], rows[:, 1]) and np.array_equal(knn[:, 2], rows[:, 2])
    assert (knn[:, 3] == knn[:, 1] + 1).all() and (rows[:, 2] < rows[:, 1]).all()
    bs = B[rows[:, 1]].astype(np.int64) - 128
    b2 = B[rows[:, 2]].astype(np.int64) - 128
    a = A[rows[:, 0]].astype(np.int64) - 128
    assert ((a * bs).sum(1) == (a * b2).sum(1)).all() and ((bs * bs).sum(1) % 2 == 0).all()     # equal accumulators
    same = rows[0::3]
    assert (same[:, 1] // 8 == same[:, 2] // 8).all() and (rows[1::3, 1] // TILE != rows[1::3, 2] // TILE).all()
    zero = np.full((1, 128), 128, np.uint8)
    sides = {}
    for ratio, dd, tl, planted in boundary_scenarios():
        B = scenario_train(rng, planted)
        knn = knn2_ref(zero, B)[0]
        assert (knn[1], knn[3]) == (planted[0][0], planted[1][0]) and knn[0] // TILE == tl[0] and knn[2] // TILE == tl[1]
        for mode in ("cv2_f32", "exact_int"):
            dlo = knn[3] & ~1                                         # C - 2 M2 of the second nearest's tile
            sides.setdefault((ratio, mode), set()).add(bool(ratio_pass(knn[1], knn[3], ratio, mode)))
            sides.setdefault((ratio, mode, "dlo"), set()).add(bool(ratio_pass(knn[1], dlo, ratio, mode) != ratio_pass(knn[1], dlo + 1, ratio, mode)))
    assert all(v == {True, False} for k, v in sides.items() if len(k) == 2)        # both sides of every ratio
    assert all(True in v for k, v in sides.items() if len(k) == 3)                   # and rows whose early stop must read on
    imgs = ragged_images(rng)
    assert [len(d) for d in imgs] == list(RAGGED)
    big = imgs[-1]
    assert (big == 0).all(1).any() and (big == 255).all(1).any() and ((big >= 127) & (big <= 129)).all(1).any()


# ====================================================================================================== GPU helpers

def _lib():
    from sfm_b200 import _lib as L

    return L


def l2_bank(imgs, xys, max_images=None, ids=None, max_feats=N):
    import sfm_b200

    ids = list(range(len(imgs))) if ids is None else ids
    bank = sfm_b200.DescriptorBank(max_images or len(imgs), max_feats)
    for i, d, xy in zip(ids, imgs, xys):
        if len(d):
            bank.put(i, d[None], xy=xy[None])
        else:
            bank.put(i, np.zeros((1, 1, 128), np.uint8), counts=[0])
    torch.cuda.synchronize()
    return bank


def stats_delta(fn):
    """(result of fn(), rows brute-forced by the refinement during it, candidate rows it recomputed)."""
    from sfm_b200 import matcher

    before = matcher.refine_stats(True)
    out = fn()
    torch.cuda.synchronize()
    after = matcher.refine_stats(True)
    return out, after[0] - before[0], after[1] - before[1]


def brute_delta(fn):
    """(result of fn(), rows brute-forced by the refinement during it)."""
    return stats_delta(fn)[:2]


def knn2_prefiltered(bank, pairs, ratio, mode):
    """The raw sweep + refinement with the ratio-test prefilter on (rows whose bounds fail read as -1)."""
    from sfm_b200 import matcher

    L = _lib()
    pairs_t = torch.tensor(np.asarray(pairs, np.int32), device="cuda")
    fp = matcher.filter_params(ratio, mode, False)
    prm = L.MatchParams()
    prm.impl = L.MATCH_IMPLS["tcgen05"]
    prm.prefilter_mode, prm.prefilter_ratio = fp.ratio_mode, fp.ratio
    prm.prefilter_num, prm.prefilter_den = int(fp.ratio_num), int(fp.ratio_den)
    out = torch.empty((len(pairs), bank.feat_stride, 4), dtype=torch.int32, device="cuda")
    L.check(L.lib().sfm_match_knn2(bank.handle, L.ptr(pairs_t), len(pairs), C.byref(prm), L.ptr(out), L.current_stream_ptr()),
            "sfm_match_knn2 (prefilter)")
    return out


def assert_table(got, ref, where):
    n = len(ref)
    bad = np.nonzero((got[:n] != ref).any(1))[0]
    assert len(bad) == 0, f"{where}: {len(bad)} rows differ, first {bad[:5].tolist()}: got {got[bad[:3]].tolist()} want {ref[bad[:3]].tolist()}"
    assert (got[n:] == -1).all(), f"{where}: padding rows are not -1"


def assert_rows(rows, want, where):
    q, t, d = want
    assert len(rows) == len(q), f"{where}: {len(rows)} matches, reference {len(q)}"
    assert np.array_equal(rows, np.stack([q, t, d], 1).reshape(-1, 3)), f"{where}: match rows differ"


def assert_corr(corr, xy_q, xy_t, want, where):
    q, t, _ = want
    assert np.array_equal(corr, np.concatenate([xy_q[q], xy_t[t]], 1).reshape(-1, 4)), f"{where}: gathered keypoints differ"


# ====================================================================================================== GPU: the adversarial bank

@pytest.fixture(scope="module")
def fam():
    if not HAS_CUDA:
        pytest.skip("needs a GPU")
    from sfm_b200 import matcher

    t0 = time.time()
    imgs, names, xys, groups, meta = l2_family_images()
    bank = l2_bank(imgs, xys)
    dev_imgs = [torch.from_numpy(d).cuda() for d in imgs]
    keys = sorted({p for g in groups.values() for p in g} | {(j, i) for g in groups.values() for i, j in g})
    ref = {k: knn2_ref(dev_imgs[k[0]], dev_imgs[k[1]]) for k in keys}
    model = {k: tile_model(dev_imgs[k[0]], dev_imgs[k[1]]) for k in keys}
    del dev_imgs
    torch.cuda.empty_cache()
    matcher.refine_stats(True)
    print(f"\nadversarial L2 bank: {len(imgs)} images x {bank.feat_stride} features, {bank.storage.numel() / 2**20:.0f} MiB; "
          f"{len(keys)} reference tables in {time.time() - t0:.1f} s")
    yield SimpleNamespace(imgs=imgs, names=names, xys=xys, groups=groups, meta=meta, bank=bank, ref=ref, model=model,
                          all_pairs=[p for g in groups.values() for p in g], t0=t0)
    matcher.refine_stats(False)
    print(f"\nadversarial L2 bank: module wall time {time.time() - t0:.1f} s")


@gpu_test
@pytest.mark.parametrize("impl", ["tcgen05", "simt"])
def test_knn2_tables_equal_the_reference(fam, impl):
    """The whole kNN table of every pair of every family equals the reference; padding rows are -1.  tcgen05: the rows the
    refinement brute-forces are exactly those the tile model says the proof needs (> 0 for the tie families, 0 for the
    hand-built cases that must not be)."""
    import sfm_b200

    seen = {}
    for fname, pairs in fam.groups.items():
        knn, nb = brute_delta(lambda: sfm_b200.knn2(fam.bank, pairs, impl=impl).cpu().numpy())
        for p, (i, j) in enumerate(pairs):
            assert_table(knn[p], fam.ref[(i, j)], f"{impl} {fam.names[i]} -> {fam.names[j]}")
        if impl == "tcgen05":
            want = int(sum(fam.model[k][0].sum() for k in pairs))
            seen[fname] = nb
            assert nb == want, f"{fname}: {nb} rows brute-forced, the tile model says {want}"
    if impl == "tcgen05":
        print(f"\nrows brute-forced per family (prefilter off): {seen}")
        assert seen["ties"] > 0 and seen["two_letter"] > 0 and seen["tile_cases"] > 0
        zr = fam.meta.zq
        for name, (_, brute) in TILE_CASES.items():
            assert (fam.model[(zr, fam.meta.cases[name])][0][ZERO_ROWS] == brute).all(), name
        tie_rows = fam.meta.tie_rows
        tmod = fam.model[(fam.meta.tq, fam.meta.tt)][0]
        assert all(tmod[tie_rows[k]].all() == (k >= 4) and tmod[tie_rows[k]].any() == (k >= 4) for k in tie_rows)
        assert not fam.model[(fam.meta.pq, fam.meta.pt)][0][fam.meta.parity_rows[:, 0]].any()


@gpu_test
@pytest.mark.parametrize("mode", ["cv2_f32", "exact_int"])
def test_prefilter_blanks_only_rows_that_fail_the_ratio_test(fam, mode):
    """The sweep with the prefilter on: a blanked row fails the reference ratio test, every other row is the reference row,
    and the blanked rows are exactly those whose distance bounds fail (the tile model's M1, M2)."""
    counts = {}
    for ratio in RATIO_BOUNDARY:
        pairs = fam.all_pairs
        pre, nb = brute_delta(lambda: knn2_prefiltered(fam.bank, pairs, ratio, mode).cpu().numpy())
        blanks = want_blanks = want_brute = 0
        for p, (i, j) in enumerate(pairs):
            ref, model = fam.ref[(i, j)], fam.model[(i, j)]
            n = len(ref)
            blank = pre[p, :n, 0] < 0
            keep = (ref[:, 2] >= 0) & ratio_pass(ref[:, 1], ref[:, 3], ratio, mode)
            where = f"{mode} {ratio} {fam.names[i]} -> {fam.names[j]}"
            assert not (blank & keep).any(), f"{where}: a row that passes the ratio test was blanked"
            assert np.array_equal(pre[p, :n][~blank], ref[~blank]), f"{where}: a kept row differs from the reference"
            assert (pre[p, n:] == -1).all()
            model_blank = prefilter_blanks(model, ratio, mode)
            assert np.array_equal(blank & (ref[:, 0] >= 0), model_blank), f"{where}: blanks differ from the bounds' verdict"
            blanks += int((blank & (ref[:, 0] >= 0)).sum())          # (rows with no neighbour at all read as -1 too)
            want_blanks += int(model_blank.sum())
            want_brute += int((model[0] & ~model_blank).sum())
        assert blanks == want_blanks > 0
        assert nb == want_brute, f"{mode} {ratio}: {nb} rows brute-forced, the tile model says {want_brute}"
        counts[ratio] = (blanks, nb)
    print(f"\n{mode}: prefilter (blanked rows, brute-forced rows) per ratio over {len(fam.all_pairs)} pairs: {counts}")


FILTER_CONFIGS = [
    ("cv2_f32", 0.5, False, 0), ("exact_int", 0.5, False, 0),
    ("cv2_f32", 0.75, False, 0), ("exact_int", 0.75, False, 0),
    ("cv2_f32", 0.8, False, 0), ("exact_int", 0.8, False, 0),
    ("cv2_f32", 0.999, False, 0), ("exact_int", 0.999, False, 0),
    ("cv2_f32", 0.75, True, 0), ("none", None, True, 0),
    ("exact_int", 0.8, False, 64),            # a bound equal to the D1 of boundary rows (64, 100): strict, so they drop
    ("cv2_f32", 0.8, True, 4608),
]


@gpu_test
@pytest.mark.parametrize("mode,ratio,mutual,max_d", FILTER_CONFIGS)
def test_match_filters_equal_the_reference(fam, mode, ratio, mutual, max_d):
    """match_pairs (strided filter) and match_pairs_packed (fused and kNN-table forms, prefilter on and off): counts,
    offsets, (q, t, D) rows and the gathered keypoints equal filter_ref on the reference tables, for every family."""
    from sfm_b200 import matcher

    pairs = fam.all_pairs
    want = {k: filter_ref(fam.ref[k], fam.ref[(k[1], k[0])], ratio=ratio, mode=mode, mutual=mutual, max_d=max_d) for k in set(pairs)}
    lab = lambda p: f"{mode} {ratio} mutual={mutual} max_d={max_d} {fam.names[pairs[p][0]]} -> {fam.names[pairs[p][1]]}"  # noqa: E731
    mb = matcher.match_pairs(fam.bank, pairs, ratio=ratio, ratio_mode=mode, mutual=mutual, max_distance_sq=max_d)
    cnt, m, c = mb.counts.cpu().numpy(), mb.matches.cpu().numpy(), mb.corr.cpu().numpy()
    for p, (i, j) in enumerate(pairs):
        w = want[(i, j)]
        assert cnt[p] == len(w[0]), f"strided {lab(p)}: {cnt[p]} matches, reference {len(w[0])}"
        assert_rows(m[p, : cnt[p]], w, f"strided {lab(p)}")
        assert_corr(c[p, : cnt[p]], fam.xys[i], fam.xys[j], w, f"strided {lab(p)}")
    del mb, m, c
    for fused in (True, False):
        for prefilter in (True, False):
            def run():
                return [x.cpu().numpy() for x in matcher.match_pairs_packed(fam.bank, pairs, ratio=ratio, ratio_mode=mode, mutual=mutual,
                                                                            prefilter=prefilter, fused=fused, max_distance_sq=max_d)]
            (cnt, off, m, c), nb = brute_delta(run)
            assert off[0] == 0 and np.array_equal(np.diff(off), cnt) and off[-1] == len(m)
            for p, (i, j) in enumerate(pairs):
                w = want[(i, j)]
                where = f"packed fused={fused} prefilter={prefilter} {lab(p)}"
                assert_rows(m[off[p]: off[p + 1]], w, where)
                assert_corr(c[off[p]: off[p + 1]], fam.xys[i], fam.xys[j], w, where)
            pre = prefilter and mode != "none"
            brute = sum(int((fam.model[k][0] & ~prefilter_blanks(fam.model[k], ratio, mode)).sum()) if pre else int(fam.model[k][0].sum())
                        for k in pairs)
            if mutual:                                               # the reverse table: a plain kNN run
                brute += sum(int(fam.model[(j, i)][0].sum()) for i, j in pairs)
            assert nb == brute, f"fused={fused} prefilter={prefilter}: {nb} rows brute-forced, the tile model says {brute}"
    if not mutual and not max_d:
        # The ratio-boundary rows reach both sides of this ratio, and the fused refinement reads past the record's first tile
        # exactly where the test answers differently for dlo and dlo + 1 (dlo = C - 2 M2 = D2 rounded down to even for an
        # offset-zero query).  A one-row offset-zero query against a boundary image records two 8-row sub-groups, the
        # nearest's and the second nearest's, in different tiles: the kNN-table path recomputes both (16 candidate rows), the
        # fused path 8, or 16 when it must read on.  The refinement's candidate counter shows which it did.
        z1, sides, bpairs, want_cand, n_more = fam.meta.z1, set(), [], 0, 0
        for b, r, _, _, _ in fam.meta.bnd:
            if r == ratio:
                k = fam.ref[(fam.meta.zq, b)][ZERO_ROWS[0]]
                sides.add(bool(ratio_pass(k[1], k[3], ratio, mode)))
                dlo = int(k[3]) & ~1
                more = bool(ratio_pass(k[1], dlo, ratio, mode) != ratio_pass(k[1], dlo + 1, ratio, mode))
                bpairs.append((z1, b))
                want_cand += 8 * (1 + more)
                n_more += more
        assert sides == {True, False} and 0 < n_more < len(bpairs)
        for fused, cand_want in ((True, want_cand), (False, 16 * len(bpairs))):
            def run():
                return [x.cpu().numpy() for x in matcher.match_pairs_packed(fam.bank, bpairs, ratio=ratio, ratio_mode=mode, prefilter=False,
                                                                            fused=fused)]
            (cnt, off, m, _), nb, cand = stats_delta(run)
            for p, (_, b) in enumerate(bpairs):
                w = filter_ref(fam.ref[(fam.meta.zq, b)][ZERO_ROWS[:1]], ratio=ratio, mode=mode)
                assert_rows(m[off[p]: off[p + 1]], w, f"one-row boundary query fused={fused} {mode} {ratio} -> {fam.names[b]}")
            assert nb == 0 and cand == cand_want, f"fused={fused}: {cand} candidate rows recomputed, expected {cand_want}"
        print(f"\n{mode} {ratio}: the fused refinement read past the first tile for {n_more} of {len(bpairs)} boundary rows "
              f"({want_cand} candidate rows against {16 * len(bpairs)} on the table path)")


@gpu_test
def test_match_and_verify_rows_equal_the_reference(fam):
    """One adversarial 32,768-feature job through match_and_verify(fetch=True) in batches of two pairs: its packed match rows
    equal filter_ref."""
    import sfm_b200

    m = fam.meta
    pairs = [(m.tq, m.tt), fam.groups["two_letter"][0], (m.pq, m.pt), (m.zq, m.bnd[0][0]), (m.tt, m.tq)]
    h = sfm_b200.match_and_verify(fam.bank, pairs, ratio=0.75, ratio_mode="cv2_f32", fetch=True, pair_batch=2, max_iters=64).to_host()
    for p, (i, j) in enumerate(pairs):
        rows = h["matches"][h["offsets"][p]: h["offsets"][p + 1]]
        assert_rows(rows, filter_ref(fam.ref[(i, j)], ratio=0.75, mode="cv2_f32"), f"match_and_verify {fam.names[i]} -> {fam.names[j]}")


@gpu_test
@pytest.mark.parametrize("max_distance", [0, 1, 26, 257])
def test_hamming_at_32768_features_equals_the_reference(max_distance):
    """match_pairs_hamming at 32,768 features per image (a 128 KB shared-memory bitonic sort per pair) with duplicate rows on
    both sides, exact and near copies, all-zero rows and ragged images."""
    import sfm_b200

    imgs, pairs = hamming_family_images()
    bank = sfm_b200.build_bank(imgs, metric="hamming", max_feats=N)
    res = sfm_b200.match_pairs_hamming(bank, pairs, max_distance).to_host()
    dev = [torch.from_numpy(d).cuda() for d in imgs]
    total = 0
    for (i, j), got in zip(pairs, res):
        want = hamming_ref(dev[i], dev[j], max_distance)
        assert all(np.array_equal(x, y) for x, y in zip(got, want)), f"hamming {i} -> {j}, max_distance {max_distance}"
        total += len(want[0])
    assert (total == 0) == (max_distance == 0)
    print(f"\nhamming max_distance {max_distance}: {total} matches over {len(pairs)} pairs")


# ====================================================================================================== GPU: sizes where offsets and grid limits bite

def _need_free(nbytes, what):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        print(f"\n{what}: skipped, {free / 1e9:.1f} GB of device memory free, {nbytes / 1e9:.1f} GB needed")
        pytest.skip(f"{what} needs {nbytes / 1e9:.0f} GB of free device memory, {free / 1e9:.1f} GB free")


@gpu_test
def test_l2_bank_past_4gib():
    """A bank of 1,040 images x 32,768 features: the descriptor section is 4.06 GiB, so images 1,024 and up lie wholly past byte
    2^32 of it (and images 512 and up past 2^31).  Only nine images are filled (no dense host copy of the bank); a tie family
    on image 1,039 makes the brute-force path read rows there."""
    import sfm_b200
    from sfm_b200 import matcher

    _need_free(8 * 10**9, "L2 bank past 4 GiB")
    rng = np.random.default_rng(31)
    tq, tt, _ = tie_family(rng)
    ids = [0, 1, 511, 512, 513, 1023, 1024, 1038, 1039]
    imgs = {0: tq, 1039: tt}
    for i in ids[1:-1]:
        imgs[i] = synth.sift_like(rng, N - 37 * (i % 3))
    pool = np.concatenate([imgs[1], imgs[512]])
    for i in (511, 513, 1023, 1024, 1038):
        imgs[i][:6000] = synth.observe(rng, pool[rng.integers(0, len(pool), 6000)])
    xys = {i: rng.uniform(0, 4000, (len(imgs[i]), 2)).astype(np.float32) for i in ids}
    bank = l2_bank([imgs[i] for i in ids], [xys[i] for i in ids], max_images=1040, ids=ids)
    desc = bank._off["ext"] - bank._off["desc"]
    print(f"\nL2 bank: {bank.storage.numel()} bytes, descriptor section {desc} bytes (2^32 = {1 << 32}); image 1039 starts at "
          f"descriptor byte {1039 * bank.feat_stride * 128}")
    assert desc > 1 << 32 and 1024 * bank.feat_stride * 128 >= 1 << 32
    pairs = [(0, 1039), (1039, 0), (1039, 1039), (1, 512), (512, 1), (511, 513), (1024, 1038), (1038, 1024), (0, 1023), (1023, 1024), (513, 511)]
    dev = {i: torch.from_numpy(imgs[i]).cuda() for i in ids}
    ref = {k: knn2_ref(dev[k[0]], dev[k[1]]) for k in set(pairs) | {(j, i) for i, j in pairs}}
    brute_model = sum(int(tile_model(dev[i], dev[j])[0].sum()) for i, j in pairs)
    for impl in ("tcgen05", "simt"):
        knn, nb = brute_delta(lambda: sfm_b200.knn2(bank, pairs, impl=impl).cpu().numpy())
        for p, k in enumerate(pairs):
            assert_table(knn[p], ref[k], f"{impl} {k}")
        if impl == "tcgen05":
            assert nb == brute_model > 0, (nb, brute_model)
    for mutual in (False, True):
        cnt, off, m, c = (x.cpu().numpy() for x in matcher.match_pairs_packed(bank, pairs, ratio=0.8, mutual=mutual))
        for p, (i, j) in enumerate(pairs):
            w = filter_ref(ref[(i, j)], ref[(j, i)], ratio=0.8, mutual=mutual)
            assert_rows(m[off[p]: off[p + 1]], w, f"packed {i} -> {j}")
            assert_corr(c[off[p]: off[p + 1]], xys[i], xys[j], w, f"packed {i} -> {j}")
    print(f"L2 bank past 4 GiB: {brute_model} rows brute-forced, {int(cnt.sum())} mutual matches")


@gpu_test
def test_hamming_bank_past_2gib():
    """A Hamming bank of 2,080 images x 32,768 features (descriptor section 2.03 GiB, past 2^31 bytes), seven images filled."""
    import sfm_b200

    _need_free(6 * 10**9, "Hamming bank past 2 GiB")
    rng = np.random.default_rng(32)
    a, b = hamming_family_images(33)[0][:2]
    ids = [0, 1, 1023, 1024, 2047, 2048, 2079]
    imgs = {0: a, 2079: b}
    for i in ids[1:-1]:
        imgs[i] = rng.integers(0, 256, (N - 11 * (i % 5), 32), dtype=np.uint8)
        imgs[i][:4000] = b[rng.integers(0, N, 4000)] ^ np.packbits(rng.random((4000, 256)) < 0.03, axis=1)
    bank = sfm_b200.DescriptorBank(2080, N, metric="hamming")
    for i in ids:
        bank.put(i, imgs[i][None])
    desc = bank._off["ext"] - bank._off["desc"]
    print(f"\nHamming bank: {bank.storage.numel()} bytes, descriptor section {desc} bytes (2^31 = {1 << 31})")
    assert desc > 1 << 31
    pairs = [(0, 2079), (2079, 0), (2079, 2079), (1, 2048), (2048, 1), (1023, 1024), (2047, 2079), (2079, 1023)]
    dev = {i: torch.from_numpy(imgs[i]).cuda() for i in ids}
    for md in (26, 257):
        res = sfm_b200.match_pairs_hamming(bank, pairs, md).to_host()
        for (i, j), got in zip(pairs, res):
            want = hamming_ref(dev[i], dev[j], md)
            assert all(np.array_equal(x, y) for x, y in zip(got, want)), f"hamming {i} -> {j}, max_distance {md}"


@gpu_test
def test_more_than_65535_pairs_in_one_call():
    """70,001 pairs over seven small images (0 to 256 rows, every ordered pair and self pair): the Hamming distance kernel and
    the SIMT matcher chunk the pair list over gridDim.y; the tcgen05 sweep, the filters and the packed path take it whole.
    Per-pair counts and rows equal the reference, computed once per distinct pair."""
    import sfm_b200
    from sfm_b200 import matcher

    rng = np.random.default_rng(41)
    sizes = (256, 200, 129, 1, 77, 250, 0)
    l2 = ragged_images(rng, sizes)
    ham = [rng.integers(0, 256, (n, 32), dtype=np.uint8) for n in sizes]
    for d in ham[1:]:
        k = min(len(d), 60)
        d[:k] = ham[0][rng.integers(0, 256, k)] ^ np.packbits(rng.random((k, 256)) < 0.03, axis=1)
    xys = [rng.uniform(0, 1000, (n, 2)).astype(np.float32) for n in sizes]
    distinct = [(i, j) for i in range(len(sizes)) for j in range(len(sizes))]
    P = 70001
    sel = np.concatenate([np.arange(len(distinct))] * (P // len(distinct) + 1))[:P]
    sel = sel[rng.permutation(P)]
    pairs = np.array(distinct, np.int32)[sel]
    groups = [np.nonzero(sel == g)[0] for g in range(len(distinct))]

    def check_strided(cnt, m, want, where):
        for g, (i, j) in enumerate(distinct):
            ps, w = groups[g], want[(i, j)]
            assert (cnt[ps] == len(w[0])).all(), f"{where} {i} -> {j}: counts"
            rows = m[ps, : len(w[0])]
            assert (rows == np.stack(w, 1)[None]).all(), f"{where} {i} -> {j}: rows"

    hb = sfm_b200.build_bank(ham, metric="hamming")
    mb = sfm_b200.match_pairs_hamming(hb, pairs, 40)
    check_strided(mb.counts.cpu().numpy(), mb.matches.cpu().numpy(), {k: hamming_ref(ham[k[0]], ham[k[1]], 40) for k in distinct}, "hamming")
    del mb, hb
    bank = l2_bank(l2, xys, max_feats=256)
    ref = {k: knn2_ref(l2[k[0]], l2[k[1]]) for k in distinct}
    for impl in ("tcgen05", "simt"):
        knn = sfm_b200.knn2(bank, pairs, impl=impl).cpu().numpy()
        for g, (i, j) in enumerate(distinct):
            n = len(l2[i])
            assert (knn[groups[g], :n] == ref[(i, j)][None]).all() and (knn[groups[g], n:] == -1).all(), f"{impl} {i} -> {j}"
        del knn
    want = {k: filter_ref(ref[k], ref[(k[1], k[0])], ratio=0.8, mutual=True) for k in distinct}
    mb = matcher.match_pairs(bank, pairs, ratio=0.8, mutual=True)
    check_strided(mb.counts.cpu().numpy(), mb.matches.cpu().numpy(), want, "match_pairs")
    del mb
    for fused in (True, False):
        cnt, off, m, _ = (x.cpu().numpy() for x in matcher.match_pairs_packed(bank, pairs, ratio=0.8, mutual=True, fused=fused))
        assert np.array_equal(np.diff(off), cnt)
        for g, (i, j) in enumerate(distinct):
            ps, w = groups[g], want[(i, j)]
            k = len(w[0])
            assert (cnt[ps] == k).all(), f"packed fused={fused} {i} -> {j}: counts"
            idx = off[ps][:, None] + np.arange(k)[None]
            assert (m[idx] == np.stack(w, 1)[None]).all(), f"packed fused={fused} {i} -> {j}: rows"
