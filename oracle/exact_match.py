"""Exact integer reference of the L2 matcher: kNN(k=2) and the ratio / distance / mutual filter, written from the
definitions and sharing no code with the kernels.  TEST INFRASTRUCTURE ONLY.

* ``knn2_ref``: squared L2 as |a|^2 + |b|^2 - 2 a.b with the dot products as a float64 GEMM in row chunks (exact: every
  value is an integer below 2^53), top-2 by the int64 key D * 2^16 + trainIdx, so the lowest index wins a tie without
  relying on any library's argmin;
* ``filter_ref``: Lowe's test as ``float64(sqrt_f32(D1)) < ratio * float64(sqrt_f32(D2))`` (cv2_f32) or
  ``D1 den^2 < D2 num^2`` with ``Fraction(ratio).limit_denominator(1024)`` (exact_int), the strict bound D1 < max_d, the
  mutual check on the reverse table's nearest; rows in ascending queryIdx.

Pinned to cv2, to oracle/match_oracle.py and to the golden files by tests/test_gpu_match_reference.py.
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np
import torch

CHUNK_ELEMS = {"cpu": 1 << 24, "cuda": 1 << 27}     # elements of one reference chunk (query rows x train rows)


def _tensor(x, device=None):
    if isinstance(x, torch.Tensor):
        return x if device is None else x.to(device)
    return torch.from_numpy(np.ascontiguousarray(x)).to(device or "cpu")


def _step(nt, device):
    return max(1, CHUNK_ELEMS[torch.device(device).type] // max(nt, 1))


def knn2_ref(A, B, device=None):
    """Exact kNN(k=2) of uint8 rows: int32 [nq, 4] = (idx1, D1, idx2, D2), -1 for a missing neighbour.  A and B are
    numpy arrays or torch tensors (the work runs on B's device, or ``device``)."""
    B = _tensor(B, device)
    A = _tensor(A, B.device)
    nq, nt = A.shape[0], B.shape[0]
    out = np.full((nq, 4), -1, np.int32)
    if nq == 0 or nt == 0:
        return out
    b = B.double()
    nb = (b * b).sum(1)
    idx = torch.arange(nt, device=B.device, dtype=torch.int64)
    k = min(2, nt)
    step = _step(nt, B.device)
    for r0 in range(0, nq, step):
        a = A[r0: r0 + step].double()
        D = (a * a).sum(1, keepdim=True) + nb[None, :] - 2.0 * (a @ b.T)          # exact integers in float64
        key = D.to(torch.int64) * 65536 + idx[None, :]
        v = torch.topk(key, k, dim=1, largest=False, sorted=True).values.cpu().numpy()
        for j in range(k):
            out[r0: r0 + len(v), 2 * j] = v[:, j] & 0xFFFF
            out[r0: r0 + len(v), 2 * j + 1] = v[:, j] >> 16
    return out


def ratio_pass(d1, d2, ratio, mode):
    """Lowe's test on squared distances: cv2's idiom on float32 distances promoted to double, or exact integers."""
    d1 = np.asarray(d1, np.int64)
    d2 = np.asarray(d2, np.int64)
    if mode == "cv2_f32":
        s1 = np.sqrt(np.maximum(d1, 0).astype(np.float32)).astype(np.float64)
        s2 = np.sqrt(np.maximum(d2, 0).astype(np.float32)).astype(np.float64)
        return s1 < np.float64(ratio) * s2
    f = Fraction(ratio).limit_denominator(1024)
    return d1 * (f.denominator ** 2) < d2 * (f.numerator ** 2)


def filter_ref(knn_fwd, knn_rev=None, ratio=0.75, mode="cv2_f32", mutual=False, max_d=0):
    """(q, t, D1) int32 of the rows that pass: ratio test (mode None / "none": none), D1 < max_d when max_d > 0, and the
    mutual check against the reverse table's nearest."""
    i1, d1, i2, d2 = (knn_fwd[:, c].astype(np.int64) for c in range(4))
    keep = i1 >= 0
    if ratio is not None and mode not in (None, "none"):
        keep &= (i2 >= 0) & ratio_pass(d1, d2, ratio, mode)
    if max_d > 0:
        keep &= d1 < max_d
    if mutual:
        back = np.full(len(i1), -2, np.int64)
        back[i1 >= 0] = knn_rev[i1[i1 >= 0], 0]
        keep &= back == np.arange(len(i1))
    q = np.nonzero(keep)[0]
    return q.astype(np.int32), i1[q].astype(np.int32), d1[q].astype(np.int32)
