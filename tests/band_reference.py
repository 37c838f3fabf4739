"""Checkers of the Sakoe-Chiba band (ss_dict_set_dtw_band, tests/test_band_*.py); spec in the header of tests/cpp/dtw_band.cpp.

  dtw_band, dtw_band_topk, dtw_band_path, in_band
                 tests/cpp/dtw_band.cpp through ctypes: D with orc_dtw's operations in orc_dtw's order, cells outside the
                 band +inf. Compiled on first use into a temporary directory (nothing is written to the tree).
  twin_dtw_band  an independent numpy restatement (band mask from the inequality, costs accumulated coefficient by
                 coefficient in A8's order).
"""
import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "cpp", "dtw_band.cpp")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), "soundsym_band_ref_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "dtw_band_%s.so" % hashlib.sha1(src).hexdigest()[:16])
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        vp, sz, u32, i = C.c_void_p, C.c_size_t, C.c_uint32, C.c_int
        L.ref_dtw_band.restype = C.c_double
        L.ref_dtw_band.argtypes = [vp, sz, vp, sz, i, u32]
        L.ref_in_band.restype = i
        L.ref_in_band.argtypes = [sz, sz, sz, sz, u32]
        L.ref_dtw_band_topk.argtypes = [vp, vp, sz, vp, vp, sz, i, i, u32, i, vp, vp]
        L.ref_dtw_band_path.restype = sz
        L.ref_dtw_band_path.argtypes = [vp, sz, vp, sz, i, u32, vp]
        _LIB = L
    return _LIB


def _f64(x):
    return np.ascontiguousarray(x, dtype=np.float64)


def _ncoeffs(a, b):
    return a.shape[1] if a.ndim == 2 else b.shape[1]


def dtw_band(a, b, r):
    a, b = _f64(a), _f64(b)
    return float(_lib().ref_dtw_band(a.ctypes.data, a.shape[0], b.ctypes.data, b.shape[0], _ncoeffs(a, b), int(r)))


def in_band(i, j, la, lb, r):
    return bool(_lib().ref_in_band(i, j, la, lb, int(r)))


def dtw_band_topk(dict_flat, dict_off, q_flat, q_off, c, k, r):
    """-> (idx u32 [nq, k], dist f64 [nq, k]), local indices"""
    d, q = _f64(dict_flat), _f64(q_flat)
    do, qo = np.ascontiguousarray(dict_off, dtype=np.uint64), np.ascontiguousarray(q_off, dtype=np.uint64)
    nq = qo.shape[0] - 1
    idx = np.empty((nq, k), dtype=np.uint32)
    dist = np.empty((nq, k), dtype=np.float64)
    _lib().ref_dtw_band_topk(d.ctypes.data, do.ctypes.data, do.shape[0] - 1, q.ctypes.data, qo.ctypes.data, nq, int(c), int(k), int(r),
                             os.cpu_count() or 1, idx.ctypes.data, dist.ctypes.data)
    return idx, dist


def dtw_band_path(a, b, r):
    """the banded warping path of (a, b) as uint32 [n, 2] of (i, j), ascending; empty if a side is empty or the distance is
    not finite"""
    a, b = _f64(a), _f64(b)
    la, lb = a.shape[0], b.shape[0]
    out = np.empty((max(la + lb - 1, 1), 2), dtype=np.uint32)
    n = _lib().ref_dtw_band_path(a.ctypes.data, la, b.ctypes.data, lb, _ncoeffs(a, b), int(r), out.ctypes.data)
    return out[:n].copy()


def band_mask(la, lb, r):
    """bool [la, lb]: the cells inside the band (all of them for r = 0)"""
    if r == 0:
        return np.ones((la, lb), dtype=bool)
    i = np.arange(la, dtype=np.int64)[:, None]
    j = np.arange(lb, dtype=np.int64)[None, :]
    w = min(int(r), max(la, lb)) * max(la - 1, lb - 1)
    return np.abs(i * (lb - 1) - j * (la - 1)) <= w


def twin_dtw_band(a, b, r):
    a, b = _f64(a), _f64(b)
    la, lb = a.shape[0], b.shape[0]
    if la == 0 or lb == 0:
        return math.inf
    cost = np.zeros((la, lb))
    with np.errstate(over="ignore", invalid="ignore"):
        for k in range(a.shape[1]):
            d = a[:, None, k] - b[None, :, k]
            cost = cost + d * d
    inside = band_mask(la, lb, r)
    D = np.full((la, lb), np.inf)
    for i in range(la):
        for j in range(lb):
            if not inside[i, j]:
                continue
            if i == 0 and j == 0:
                m = 0.0
            elif i == 0:
                m = D[0, j - 1]
            elif j == 0:
                m = D[i - 1, 0]
            else:
                m = np.fmin(np.fmin(D[i - 1, j], D[i, j - 1]), D[i - 1, j - 1])
            D[i, j] = cost[i, j] + m
    return float(D[-1, -1] / (la + lb))
