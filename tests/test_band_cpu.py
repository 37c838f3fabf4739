"""The Sakoe-Chiba band's checker (tests/cpp/dtw_band.cpp, spec A10 in DESIGN.md §3.1f) on the CPU: against its numpy twin bit for
bit, against orc_dtw where the band covers the whole matrix, and the two properties the spec claims (the end cell is always
reachable; r >= min(Lq-1, Ld-1) is no band at all)."""
import numpy as np
import pytest

import align_reference as AR
import band_reference as R
from oracle import oracle as O
from soundsym_b200 import synth


def bits(x):
    return np.float64(x).view(np.uint64)


def ragged(n, lmin, lmax, seed):
    flat, off = synth.segments(n, 13, lmin=lmin, lmax=lmax, seed=seed)
    return [flat[int(off[i]):int(off[i + 1])] for i in range(n)]


@pytest.mark.parametrize("r", [0, 1, 2, 3, 5, 16])
def test_checker_equals_numpy_twin_on_ragged_pairs(r):
    qs, ds = ragged(24, 1, 48, seed=11), ragged(24, 1, 48, seed=12)
    for a, b in zip(qs, ds):
        assert bits(R.dtw_band(a, b, r)) == bits(R.twin_dtw_band(a, b, r)), (a.shape[0], b.shape[0], r)


def test_checker_equals_numpy_twin_on_ties_and_extreme_shapes():
    rng = np.random.default_rng(3)
    for la, lb in ((1, 1), (1, 40), (40, 1), (2, 39), (39, 2), (7, 64), (64, 7)):
        a = rng.integers(0, 3, size=(la, 13)).astype(np.float64)  # few distinct values: many equal costs
        b = rng.integers(0, 3, size=(lb, 13)).astype(np.float64)
        for r in (1, 2, 4):
            assert bits(R.dtw_band(a, b, r)) == bits(R.twin_dtw_band(a, b, r)), (la, lb, r)


def test_end_cell_reachable_for_every_shape_up_to_40():
    """brute force over Lq, Ld <= 40 and r = 1..6: the rows' in-band intervals are contiguous, overlap row to row inside
    [0, Ld - 1], both corners are inside, and a zero-cost pair (D = 0 on every reachable cell) has a finite distance"""
    z = np.zeros((40, 1))
    for la in range(1, 41):
        for lb in range(1, 41):
            for r in range(1, 7):
                m = R.band_mask(la, lb, r)
                assert m[0, 0] and m[-1, -1], (la, lb, r)
                lo = m.argmax(axis=1)
                hi = lb - 1 - m[:, ::-1].argmax(axis=1)
                assert m.any(axis=1).all() and (m.sum(axis=1) == hi - lo + 1).all(), (la, lb, r)  # one interval per row
                assert (lo[1:] <= hi[:-1]).all(), (la, lb, r)  # consecutive rows share a column
                assert R.dtw_band(z[:la], z[:lb], r) == 0.0, (la, lb, r)


def test_mask_matches_the_checkers_predicate():
    for la, lb, r in ((5, 17, 1), (17, 5, 2), (33, 33, 3), (1, 9, 1), (9, 1, 1), (40, 3, 6)):
        m = R.band_mask(la, lb, r)
        for i in range(la):
            for j in range(lb):
                assert m[i, j] == R.in_band(i, j, la, lb, r), (la, lb, r, i, j)


def test_wide_band_and_no_band_are_orc_dtw_bit_for_bit():
    qs, ds = ragged(30, 1, 40, seed=21), ragged(30, 1, 40, seed=22)
    for a, b in zip(qs, ds):
        want = bits(O.dtw(a, b))
        assert bits(R.dtw_band(a, b, 0)) == want
        rmin = max(min(a.shape[0] - 1, b.shape[0] - 1), 1)
        for r in (rmin, rmin + 1, 2048, 0xFFFFFFFF):
            assert bits(R.dtw_band(a, b, r)) == want, (a.shape[0], b.shape[0], r)


def test_narrow_band_is_never_below_the_unbanded_distance():
    qs, ds = ragged(40, 2, 40, seed=31), ragged(40, 2, 40, seed=32)
    for a, b in zip(qs, ds):
        free = O.dtw(a, b)
        for r in (1, 2, 4):
            assert R.dtw_band(a, b, r) >= free


def test_topk_equals_per_pair_distances():
    d, doff = synth.segments(60, 13, lmin=1, lmax=40, seed=41)
    q, qoff = synth.segments(9, 13, lmin=1, lmax=40, seed=42)
    for r in (0, 1, 3):
        idx, dist = R.dtw_band_topk(d, doff, q, qoff, 13, 4, r)
        for qi in range(9):
            a = q[int(qoff[qi]):int(qoff[qi + 1])]
            all_d = np.array([R.dtw_band(a, d[int(doff[s]):int(doff[s + 1])], r) for s in range(60)])
            order = sorted(range(60), key=lambda s: (all_d[s], s))[:4]
            assert list(idx[qi]) == order, (r, qi)
            assert np.array_equal(dist[qi].view(np.uint64), all_d[order].view(np.uint64))
    oi, od = O.dtw_topk(d, doff, q, qoff, 13, 4)
    idx, dist = R.dtw_band_topk(d, doff, q, qoff, 13, 4, 0)
    assert np.array_equal(idx, oi) and np.array_equal(dist.view(np.uint64), od.view(np.uint64))


def test_banded_path_stays_in_the_band_and_is_the_unbanded_path_when_wide():
    qs, ds = ragged(30, 1, 70, seed=51), ragged(30, 1, 70, seed=52)
    for a, b in zip(qs, ds):
        la, lb = a.shape[0], b.shape[0]
        for r in (1, 2, 5):
            p = R.dtw_band_path(a, b, r)
            assert max(la, lb) <= p.shape[0] <= la + lb - 1
            assert tuple(p[0]) == (0, 0) and tuple(p[-1]) == (la - 1, lb - 1)
            steps = np.diff(p.astype(np.int64), axis=0)
            assert ((steps >= 0) & (steps <= 1)).all() and (steps.sum(axis=1) >= 1).all()
            assert all(R.in_band(int(i), int(j), la, lb, r) for i, j in p), (la, lb, r)
        assert np.array_equal(R.dtw_band_path(a, b, 0), AR.dtw_path(a, b))
        assert np.array_equal(R.dtw_band_path(a, b, max(la, lb)), AR.dtw_path(a, b))
