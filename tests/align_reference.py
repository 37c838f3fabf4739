"""Checkers of ss_dict_align (tests/test_align_*.py): the DTW warping path of a pair, twice.

  dtw_path       tests/cpp/dtw_path.cpp through ctypes: D with orc_dtw's operations in orc_dtw's order, then the backtrack.
                 Compiled on first use into a temporary directory (nothing is written to the tree).
  twin_dtw_path  an independent numpy restatement of the same spec (see the header of tests/cpp/dtw_path.cpp).
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "cpp", "dtw_path.cpp")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), "soundsym_align_ref_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "dtw_path_%s.so" % hashlib.sha1(src).hexdigest()[:16])
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.ref_dtw_path.restype = C.c_size_t
        L.ref_dtw_path.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        _LIB = L
    return _LIB


def dtw_path(a, b):
    """the warping path of (a, b) as uint32 [n, 2] of (i, j), ascending; empty if a side is empty or the distance is not
    finite"""
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    c = a.shape[1] if a.ndim == 2 else b.shape[1]
    la, lb = a.shape[0], b.shape[0]
    out = np.empty((max(la + lb - 1, 1), 2), dtype=np.uint32)
    n = _lib().ref_dtw_path(a.ctypes.data, la, b.ctypes.data, lb, c, out.ctypes.data)
    return out[:n].copy()


def twin_dtw_path(a, b):
    """the same recurrence written out over whole rows (local costs accumulated coefficient by coefficient, in A8's order),
    then the backtrack with NaN mapped to +inf and the first of (diag, up, left) taken on a tie"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    la, lb = a.shape[0], b.shape[0]
    empty = np.zeros((0, 2), dtype=np.uint32)
    if la == 0 or lb == 0:
        return empty
    cost = np.zeros((la, lb))
    with np.errstate(over="ignore", invalid="ignore"):  # inf / NaN costs are part of the spec
        for k in range(a.shape[1]):
            d = a[:, None, k] - b[None, :, k]
            cost = cost + d * d
    D = np.empty((la, lb))
    for i in range(la):
        for j in range(lb):
            if i == 0 and j == 0:
                m = 0.0
            elif i == 0:
                m = D[0, j - 1]
            elif j == 0:
                m = D[i - 1, 0]
            else:
                m = np.fmin(np.fmin(D[i - 1, j], D[i, j - 1]), D[i - 1, j - 1])
            D[i, j] = cost[i, j] + m
    if not np.isfinite(D[-1, -1] / (la + lb)):
        return empty
    path = [(la - 1, lb - 1)]
    i, j = la - 1, lb - 1
    while (i, j) != (0, 0):
        best, step = np.inf, None
        for di, dj in ((1, 1), (1, 0), (0, 1)):  # diag, up, left: a later one must be strictly smaller
            if i - di < 0 or j - dj < 0:
                continue
            v = D[i - di, j - dj]
            v = np.inf if np.isnan(v) else v
            if step is None or v < best:
                best, step = v, (di, dj)
        i, j = i - step[0], j - step[1]
        path.append((i, j))
    return np.array(path[::-1], dtype=np.uint32)
