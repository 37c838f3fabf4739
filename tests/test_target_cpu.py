"""SS_DTW_TARGET's numpy twin (tests/target_reference.py, spec A13 in DESIGN.md §3.1h) against brute force, and the bound E(pair)
of the fp32 scan's target keys against a float32 restatement of the scan's recurrence."""
import math

import numpy as np
import pytest

import target_reference as T
from oracle import oracle as O
from soundsym_b200 import synth


def brute(D, t, k):
    nq, nseg = D.shape
    idx = np.full((nq, k), T.NONE, dtype=np.uint32)
    out = np.full((nq, k), np.inf)
    for q in range(nq):
        keys = []
        for j in range(nseg):
            e = abs(float(D[q, j]) - float(t[q]))
            if e < math.inf:
                keys.append((e, j))
        keys.sort()
        for s, (e, j) in enumerate(keys[:k]):
            idx[q, s], out[q, s] = j, e
    return idx, out


def test_twin_equals_brute_force_with_ties_negative_targets_nan_and_inf():
    rng = np.random.default_rng(5)
    D = rng.uniform(0.0, 10.0, size=(40, 300))
    D[:, ::7] = np.round(D[:, ::7])  # repeated values
    D[0, 3], D[0, 9] = np.nan, np.inf
    D[1, 5], D[1, 2], D[1, 20] = 1.0, 3.0, 3.0  # t = 2: |1 - 2| == |3 - 2|, the lowest index (2) wins
    t = rng.uniform(-5.0, 12.0, size=40)
    t[1] = 2.0
    t[2] = -3.0
    for k in (1, 3, 8):
        got = T.target_topk(D, t, k)
        want = brute(D, t, k)
        assert np.array_equal(got[0], want[0])
        assert np.array_equal(got[1].view(np.uint64), want[1].view(np.uint64))
    row = np.full((1, 6), np.nan)
    row[0, 4] = 2.5
    i, e = T.target_topk(row, [1.0], 3)
    assert list(i[0]) == [4, T.NONE, T.NONE] and e[0, 0] == 1.5 and np.all(np.isinf(e[0, 1:]))


def test_tie_between_distances_either_side_of_the_target():
    D = np.array([[5.0, 3.0, 1.0, 3.0, 1.0]])
    i, e = T.target_topk(D, [2.0], 5)
    assert list(i[0]) == [1, 2, 3, 4, 0] and list(e[0]) == [1.0, 1.0, 1.0, 1.0, 3.0]


def test_zero_targets_give_dtw_topk():
    d, doff = synth.segments(120, 13, lmin=1, lmax=40, seed=21)
    q, qoff = synth.segments(15, 13, lmin=1, lmax=40, seed=22)
    D = O.dtw_matrix(d, doff, q, qoff, 13)
    for k in (1, 8):
        oi, od = O.dtw_topk(d, doff, q, qoff, 13, k)
        for t in (None, np.zeros(15)):
            ti, te = T.target_topk(D, t, k)
            assert np.array_equal(ti, oi) and np.array_equal(te.view(np.uint64), od.view(np.uint64))


def pairs(n, lmin, lmax, seed):
    flat, off = synth.segments(2 * n, 13, lmin=lmin, lmax=lmax, seed=seed)
    segs = [flat[int(off[i]):int(off[i + 1])] for i in range(2 * n)]
    return list(zip(segs[:n], segs[n:]))


@pytest.mark.parametrize("r", [0, 3])
def test_bound_holds_on_the_float32_scan(r):
    """|scan_f32 - D| <= E(pair) for pairs of 1-400 frames and a 2 048-frame pair; prints the largest observed error as a
    fraction of the bound (the path-length term is what makes E grow with the pair)."""
    ps = pairs(24, 1, 400, seed=31 + r)
    rng = np.random.default_rng(8)
    a = rng.normal(size=(2048, 13)) * 3.0
    ps.append((a, a[::-1] + 0.05 * rng.normal(size=(2048, 13))))
    ps.append((a, a + 1e-3 * rng.normal(size=(2048, 13))))  # near-identical: the cancellation in |a|^2 + |b|^2 - 2ab
    worst = 0.0
    for a, b in ps:
        na, nb = T.max_norm(a), T.max_norm(b)
        s = T.scan_f32(a, b, r)
        D = T.dtw_f64(a, b, r)
        bound = T.scan_bound(s, a.shape[0], b.shape[0], na, nb)
        err = abs(s - D)
        assert err <= bound, (a.shape[0], b.shape[0], s, D, bound)
        worst = max(worst, err / bound)
        # the key is a lower bound on e for any target
        for t in (0.0, D, 0.5 * D, 2.0 * D + 1.0, -1.0):
            assert T.target_key(s, t, a.shape[0], b.shape[0], na, nb) <= abs(D - t)
    print("largest observed |scan - D| / E = %.3g" % worst)
    assert worst > 0.0
