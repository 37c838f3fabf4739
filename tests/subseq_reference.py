"""Checkers of subsequence DTW (ss_dict_locate, tests/test_locate_*.py); spec A12 in the header of tests/cpp/dtw_subseq.cpp.

  subseq, subseq_matrix, subseq_topk, subseq_path, dtw_matrix
                 tests/cpp/dtw_subseq.cpp through ctypes: S and the start columns with orc_dtw's operations in orc_dtw's order,
                 the hit, the top-k by (cost, index), the backtrack of S, and A8's unnormalised D. Compiled on first use into a
                 temporary directory (nothing is written to the tree).
  twin_subseq    an independent numpy restatement (costs accumulated coefficient by coefficient in A8's order).
"""
import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "cpp", "dtw_subseq.cpp")
_LIB = None
NONE = 0xFFFFFFFF


def _lib():
    global _LIB
    if _LIB is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), "soundsym_subseq_ref_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "dtw_subseq_%s.so" % hashlib.sha1(src).hexdigest()[:16])
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        vp, sz, i = C.c_void_p, C.c_size_t, C.c_int
        L.ref_subseq.restype = i
        L.ref_subseq.argtypes = [vp, sz, vp, sz, i, vp, vp, vp, vp, vp]
        L.ref_dtw_matrix.restype = None
        L.ref_dtw_matrix.argtypes = [vp, sz, vp, sz, i, vp]
        L.ref_subseq_path.restype = sz
        L.ref_subseq_path.argtypes = [vp, sz, vp, sz, i, vp]
        L.ref_subseq_topk.restype = None
        L.ref_subseq_topk.argtypes = [vp, vp, sz, vp, vp, sz, i, i, i, vp, vp, vp, vp]
        _LIB = L
    return _LIB


def _f64(x):
    return np.ascontiguousarray(x, dtype=np.float64)


def _ncoeffs(a, b):
    return a.shape[1] if a.ndim == 2 else b.shape[1]


def subseq_matrix(a, b):
    """-> (hit (cost, start, end), S f64 [la, lb], st u32 [la, lb]); both sides non-empty"""
    a, b = _f64(a), _f64(b)
    la, lb = a.shape[0], b.shape[0]
    S = np.empty((la, lb), dtype=np.float64)
    st = np.empty((la, lb), dtype=np.uint32)
    cost, s, e = C.c_double(), C.c_uint32(), C.c_uint32()
    _lib().ref_subseq(a.ctypes.data, la, b.ctypes.data, lb, _ncoeffs(a, b), S.ctypes.data, st.ctypes.data, C.byref(cost), C.byref(s), C.byref(e))
    return (cost.value, s.value, e.value), S, st


def subseq(a, b):
    """the pair's hit -> (cost, start, end); (inf, NONE, NONE) if it has none"""
    a, b = _f64(a), _f64(b)
    cost, s, e = C.c_double(), C.c_uint32(), C.c_uint32()
    _lib().ref_subseq(a.ctypes.data, a.shape[0], b.ctypes.data, b.shape[0], _ncoeffs(a, b), None, None, C.byref(cost), C.byref(s), C.byref(e))
    return cost.value, s.value, e.value


def dtw_matrix(a, b):
    """A8's unnormalised D [la, lb] (orc_dtw's matrix)"""
    a, b = _f64(a), _f64(b)
    D = np.empty((a.shape[0], b.shape[0]), dtype=np.float64)
    _lib().ref_dtw_matrix(a.ctypes.data, a.shape[0], b.ctypes.data, b.shape[0], _ncoeffs(a, b), D.ctypes.data)
    return D


def subseq_path(a, b):
    """the backtrack of S from the hit's end to row 0 as uint32 [n, 2] of (i, j), ascending, j a column of b; empty without a hit"""
    a, b = _f64(a), _f64(b)
    la, lb = a.shape[0], b.shape[0]
    out = np.empty((max(la + lb - 1, 1), 2), dtype=np.uint32)
    n = _lib().ref_subseq_path(a.ctypes.data, la, b.ctypes.data, lb, _ncoeffs(a, b), out.ctypes.data)
    return out[:n].copy()


def subseq_topk(dict_flat, dict_off, q_flat, q_off, c, k):
    """-> (idx, start, end: u32 [nq, k], cost f64 [nq, k]), local indices"""
    d, q = _f64(dict_flat), _f64(q_flat)
    do, qo = np.ascontiguousarray(dict_off, dtype=np.uint64), np.ascontiguousarray(q_off, dtype=np.uint64)
    nq = qo.shape[0] - 1
    idx, start, end = (np.empty((nq, k), dtype=np.uint32) for _ in range(3))
    cost = np.empty((nq, k), dtype=np.float64)
    _lib().ref_subseq_topk(d.ctypes.data, do.ctypes.data, do.shape[0] - 1, q.ctypes.data, qo.ctypes.data, nq, int(c), int(k), os.cpu_count() or 1,
                           idx.ctypes.data, start.ctypes.data, end.ctypes.data, cost.ctypes.data)
    return idx, start, end, cost


def twin_subseq(a, b):
    """-> ((cost, start, end), S, st) restated in numpy; the hit is (inf, NONE, NONE) without a finite value in the last row"""
    a, b = _f64(a), _f64(b)
    la, lb = a.shape[0], b.shape[0]
    if la == 0 or lb == 0:
        return (math.inf, NONE, NONE), None, None
    cost = np.zeros((la, lb))
    with np.errstate(over="ignore", invalid="ignore"):
        for k in range(a.shape[1]):
            d = a[:, None, k] - b[None, :, k]
            cost = cost + d * d
    S = np.full((la, lb), np.inf)
    st = np.full((la, lb), NONE, dtype=np.uint32)
    S[0] = cost[0] + 0.0
    st[0] = np.arange(lb, dtype=np.uint32)
    inf = np.float64(np.inf)
    for i in range(1, la):
        for j in range(lb):
            up = S[i - 1, j]
            left = S[i, j - 1] if j else inf
            diag = S[i - 1, j - 1] if j else inf
            m = np.fmin(np.fmin(up, left), diag)
            st[i, j] = st[i - 1, j - 1] if diag == m else (st[i - 1, j] if up == m else (st[i, j - 1] if j else NONE))
            S[i, j] = cost[i, j] + m
    last = S[-1]
    fin = np.isfinite(last)
    if not fin.any():
        return (math.inf, NONE, NONE), S, st
    e = int(np.flatnonzero(last == last[fin].min())[0])
    return (float(last[e]), int(st[-1, e]), e), S, st
