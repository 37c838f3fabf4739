"""Numpy twin of SS_DTW_TARGET (spec A13, DESIGN.md §3.1h) and a float32 restatement of the fp32 scan it filters with.

  target_topk     the k best (e, index) per query from a matrix of SS_DTW distances D [nq, nseg] and targets t [nq]:
                  e = fabs(D - t) in f64, NaN and +inf dropped, ascending by (e, index), unfilled (inf, 0xFFFFFFFF).
  scan_f32        the scan's distance of one pair, operation for operation as k_dtw_scan computes it in fp32: frames rounded
                  to float, the local cost as the two packed-FMA chains and their sum, the DP step as a min and one add,
                  the band as +inf cells, the normalisation by a rounded reciprocal. (An FMA is emulated as an exact product
                  and a double rounding, f64 then f32, which is within the bound's slack.)
  dtw_f64         the same recurrence in f64 on the unrounded frames (A8's cost order), for the bound's check.
  scan_bound      E(pair): the bound on |scan - D| the TARGET scan's keys subtract (dtw.cu target_key).
  target_key      the key itself: max(0, |s - t| - E).
"""
import math

import numpy as np

NONE = 0xFFFFFFFF
CELL_EPS = 4e-6  # dtw.cu kScanCellEps: the error of one computed local cost, in units of max|a|^2 + max|b|^2
U32 = 2.0 ** -24


def target_topk(D, targets, k):
    """-> (idx u32 [nq, k], e f64 [nq, k]); targets None means t = 0"""
    D = np.asarray(D, dtype=np.float64)
    nq, nseg = D.shape
    t = np.zeros(nq) if targets is None else np.asarray(targets, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        E = np.abs(D - t[:, None])
    idx = np.full((nq, k), NONE, dtype=np.uint32)
    out = np.full((nq, k), np.inf)
    cols = np.arange(nseg)
    for q in range(nq):
        ok = E[q] < np.inf  # (NaN compares false)
        e, j = E[q][ok], cols[ok]
        order = np.lexsort((j, e))[:k]
        idx[q, :len(order)] = j[order]
        out[q, :len(order)] = e[order]
    return idx, out


def band_mask(la, lb, r):
    if r == 0:
        return np.ones((la, lb), dtype=bool)
    i = np.arange(la, dtype=np.int64)[:, None]
    j = np.arange(lb, dtype=np.int64)[None, :]
    w = min(int(r), max(la, lb)) * max(la - 1, lb - 1)
    return np.abs(i * (lb - 1) - j * (la - 1)) <= w


def _dp(cost, inside, dtype):
    """D(la-1, lb-1) of the DTW recurrence over anti-diagonals, in `dtype` (one rounding per add, min exact, NaN as fmin)"""
    la, lb = cost.shape
    P = np.full((la + 1, lb + 1), np.inf, dtype=dtype)
    P[0, 0] = 0
    for d in range(la + lb - 1):
        i = np.arange(max(0, d - lb + 1), min(la, d + 1))
        j = d - i
        m = np.fmin(np.fmin(P[i, j + 1], P[i + 1, j]), P[i, j])
        v = (cost[i, j] + m).astype(dtype)
        v[~inside[i, j]] = np.inf
        P[i + 1, j + 1] = v
    return P[la, lb]


def _f32_fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def scan_cost_f32(a, b):
    """the fp32 scan's local costs [la, lb]: lane slots [-2 a~ .., 1.0 at 13, |a~|^2 at 14], stream slots [b~ .., |b~|^2 at 13]"""
    a32, b32 = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    la, lb, c = a32.shape[0], b32.shape[0], a32.shape[1]
    A = np.zeros((la, 16), dtype=np.float32)
    B = np.zeros((lb, 16), dtype=np.float32)
    A[:, :c] = -2.0 * a32
    A[:, 13] = 1.0
    A[:, 14] = (a32.astype(np.float64) ** 2).sum(axis=1).astype(np.float32)
    B[:, :c] = b32
    B[:, 13] = (b32.astype(np.float64) ** 2).sum(axis=1).astype(np.float32)
    lo = np.broadcast_to(A[:, None, 14], (la, lb)).astype(np.float32)
    hi = np.zeros((la, lb), dtype=np.float32)
    for s in range(0, 14, 2):  # the seven packed pairs (s, s + 1)
        lo = _f32_fma(A[:, None, s], B[None, :, s], lo)
        hi = _f32_fma(A[:, None, s + 1], B[None, :, s + 1], hi)
    return (lo + hi).astype(np.float32)


def scan_f32(a, b, r=0):
    la, lb = a.shape[0], b.shape[0]
    res = _dp(scan_cost_f32(a, b), band_mask(la, lb, r), np.float32)
    return float(np.float32(res) * (np.float32(1.0) / np.float32(la + lb)))


def dtw_f64(a, b, r=0):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    la, lb = a.shape[0], b.shape[0]
    cost = np.zeros((la, lb))
    for k in range(a.shape[1]):
        dl = a[:, None, k] - b[None, :, k]
        cost = cost + dl * dl
    return float(_dp(cost, band_mask(la, lb, r), np.float64) / (la + lb))


def max_norm(x):
    x32 = np.asarray(x, dtype=np.float32).astype(np.float64)
    return float(np.float32((x32 ** 2).sum(axis=1).max()))


def scan_bound(s, la, lb, na, nb):
    """E(pair) for a scan distance s of an la x lb pair; na / nb: the largest |a|^2 of the queries and |b|^2 of the shard"""
    nu = (la + lb) * U32  # gamma_{N+1}, N = la + lb - 1 path cells at most
    g = nu / (1.0 - nu)
    ec = CELL_EPS * (na + nb)
    return 1.001 * (g * abs(s) + (1.0 + g) * ec) / (1.0 - g)


def target_key(s, t, la, lb, na, nb):
    if not math.isfinite(s):
        return s
    return max(0.0, abs(s - t) - scan_bound(s, la, lb, na, nb))
