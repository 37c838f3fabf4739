"""Subsequence DTW's checker (tests/cpp/dtw_subseq.cpp, spec A12 in DESIGN.md §3.1g) on the CPU: against its numpy twin bit for bit,
and the three identities DESIGN proves, by brute force against A8's D (orc_dtw's matrix), orc_dtw and the alignment's checker."""
import math

import numpy as np

import align_reference as AR
import subseq_reference as R
from oracle import oracle as O
from soundsym_b200 import synth

NONE = R.NONE


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def ragged(n, lmin, lmax, seed):
    flat, off = synth.segments(n, 13, lmin=lmin, lmax=lmax, seed=seed)
    return [flat[int(off[i]):int(off[i + 1])] for i in range(n)]


def test_checker_equals_numpy_twin_on_random_pairs():
    qs, ds = ragged(40, 1, 60, seed=11), ragged(40, 1, 60, seed=12)
    rng = np.random.default_rng(13)
    ties = [(rng.integers(0, 3, size=(la, 13)).astype(np.float64), rng.integers(0, 3, size=(lb, 13)).astype(np.float64))
            for la, lb in ((1, 1), (1, 40), (40, 1), (7, 60), (60, 7), (25, 25))]  # few distinct values: many equal costs
    for a, b in list(zip(qs, ds)) + ties:
        hit, S, st = R.subseq_matrix(a, b)
        thit, tS, tst = R.twin_subseq(a, b)
        assert np.array_equal(bits(S), bits(tS)) and np.array_equal(st, tst), (a.shape[0], b.shape[0])
        assert bits(hit[0]) == bits(thit[0]) and hit[1:] == thit[1:], (a.shape[0], b.shape[0])
        assert R.subseq(a, b) == hit


def test_identities_by_brute_force():
    """Lq, Ld <= 24, finite frames (DESIGN.md §3.1g):
    1. cost == min over s' <= e of D(q, d[s'..e]), A8's unnormalised D;
    2. cost / (Lq + e - start + 1) == orc_dtw(q, d[start..e]) bit for bit (what ss_dict_match and ss_dict_align report);
    3. the alignment's path on d[start..e] is the backtrack of S from (Lq - 1, e), columns shifted by start."""
    qs, ds = ragged(150, 1, 24, seed=21), ragged(150, 1, 24, seed=22)
    rng = np.random.default_rng(23)
    for _ in range(40):  # equal costs everywhere: the tie rules decide start and end
        la, lb = int(rng.integers(1, 25)), int(rng.integers(1, 25))
        qs.append(rng.integers(0, 2, size=(la, 13)).astype(np.float64))
        ds.append(rng.integers(0, 2, size=(lb, 13)).astype(np.float64))
    for a, b in zip(qs, ds):
        la, lb = a.shape[0], b.shape[0]
        cost, s, e = R.subseq(a, b)
        assert s <= e < lb
        best = math.inf
        for s2 in range(e + 1):
            best = min(best, R.dtw_matrix(a, b[s2:e + 1])[-1, -1])
        assert bits(cost) == bits(best), (la, lb)
        span = b[s:e + 1]
        assert bits(cost) == bits(R.dtw_matrix(a, span)[-1, -1])
        assert bits(cost / (la + e - s + 1)) == bits(O.dtw(a, span)), (la, lb, s, e)
        path = R.subseq_path(a, b)
        want = AR.dtw_path(a, span)
        assert np.array_equal(path - np.array([0, s], dtype=np.uint32), want), (la, lb, s, e)
        # the end is the smallest column of the row minimum
        last = R.subseq_matrix(a, b)[1][-1]
        assert e == int(np.flatnonzero(last == last.min())[0])


def test_one_frame_query_is_the_first_argmin_column():
    rng = np.random.default_rng(31)
    for lb in (1, 5, 33, 100):
        b = rng.integers(0, 3, size=(lb, 13)).astype(np.float64)
        a = b[lb // 2:lb // 2 + 1] + 0.5
        cost, s, e = R.subseq(a, b)
        c = ((a - b) ** 2).sum(axis=1)
        cols = np.array([R.dtw_matrix(a, b[j:j + 1])[0, 0] for j in range(lb)])
        j = int(np.argmin(cols))
        assert (s, e) == (j, j) and bits(cost) == bits(cols[j]) and np.isclose(cost, c.min())


def test_copied_query_costs_zero_at_the_smallest_zero_cost_end():
    rng = np.random.default_rng(41)
    x = rng.normal(size=(30, 13))
    b = np.concatenate([rng.normal(size=(7, 13)), x, rng.normal(size=(5, 13)), x])  # the passage occurs twice
    for s0, e0 in ((7, 36), (9, 14), (20, 20)):
        cost, s, e = R.subseq(b[s0:e0 + 1], b)
        assert (cost, s, e) == (0.0, s0, e0)
    a = x[3:9]
    cost, s, e = R.subseq(a, b)
    assert (cost, s, e) == (0.0, 10, 15)  # not the second copy, at 7 + 30 + 5 + 3


def test_nan_frames_and_empty_sides():
    rng = np.random.default_rng(51)
    a, b = rng.normal(size=(6, 13)), rng.normal(size=(20, 13))
    assert R.subseq(a[:0], b) == (math.inf, NONE, NONE) and R.subseq(a, b[:0]) == (math.inf, NONE, NONE)
    bn = b.copy()
    bn[:, 0] = np.nan
    assert R.subseq(a, bn) == (math.inf, NONE, NONE)  # no finite value in the last row
    bn = b.copy()
    bn[3:8, 2] = np.nan  # a NaN block: the hit avoids it
    hit = R.subseq(a, bn)
    assert np.isfinite(hit[0]) and (hit[1] > 7 or hit[2] < 3)
    assert hit == R.twin_subseq(a, bn)[0] and bits(hit[0]) == bits(R.twin_subseq(a, bn)[0][0])
    an = a.copy()
    an[2, 5] = np.nan  # a NaN query frame makes every path NaN
    assert R.subseq(an, b) == (math.inf, NONE, NONE)


def test_topk_equals_per_pair_hits_and_fills_past_nseg():
    d, doff = synth.segments(12, 13, lmin=1, lmax=40, seed=61)
    q, qoff = synth.segments(9, 13, lmin=1, lmax=40, seed=62)
    flat_q = [q[int(qoff[i]):int(qoff[i + 1])] for i in range(9)]
    dd = [d[int(doff[s]):int(doff[s + 1])] for s in range(12)]
    dflat = np.concatenate(dd[:5] + [d[:0]] + dd[5:])  # an empty segment at index 5 is never a hit
    doff2 = np.concatenate([doff[:6], doff[5:]]).astype(np.uint64)
    qoff2 = np.concatenate([qoff[:3], qoff[2:]]).astype(np.uint64)  # an empty query at index 2: only unfilled slots
    for k in (1, 4, 8):
        idx, start, end, cost = R.subseq_topk(dflat, doff2, q, qoff2, 13, k)
        for qi in range(10):
            if qi == 2:
                assert (idx[qi] == NONE).all() and (start[qi] == NONE).all() and (end[qi] == NONE).all() and np.isinf(cost[qi]).all()
                continue
            a = flat_q[qi - (qi > 2)]
            hits = [R.subseq(a, dflat[int(doff2[s]):int(doff2[s + 1])]) for s in range(13)]
            order = sorted((s for s in range(13) if np.isfinite(hits[s][0])), key=lambda s: (hits[s][0], s))[:k]
            assert 5 not in order and len(order) == min(k, 12)
            n = len(order)
            assert list(idx[qi, :n]) == order and (idx[qi, n:] == NONE).all()
            assert list(start[qi, :n]) == [hits[s][1] for s in order] and list(end[qi, :n]) == [hits[s][2] for s in order]
            assert np.array_equal(bits(cost[qi, :n]), bits([hits[s][0] for s in order])) and np.isinf(cost[qi, n:]).all()
        if k == 8:  # k > nseg: a dictionary of 4 segments leaves slots 4..7 unfilled
            i4, s4, e4, c4 = R.subseq_topk(dflat, doff2[:5], q, qoff2, 13, k)
            assert (i4[:, 4:] == NONE).all() and (s4[:, 4:] == NONE).all() and (e4[:, 4:] == NONE).all() and np.isinf(c4[:, 4:]).all()
            assert (i4[[0, 1, 3]][:, :4] != NONE).all()
