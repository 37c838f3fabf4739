"""The DTW warping path (spec: tests/cpp/dtw_path.cpp, DESIGN.md §3.1e) on the CPU: the C++ checker against the independent numpy twin, hand-worked
known answers that pin the tie rule (diag, then up, then left; NaN counts as +inf), and the shape every path must have."""
import math

import numpy as np
import pytest

import align_reference as R
from oracle import oracle as O


def check_shape(path, la, lb):
    assert path.dtype == np.uint32 and path.ndim == 2 and path.shape[1] == 2
    assert tuple(path[0]) == (0, 0) and tuple(path[-1]) == (la - 1, lb - 1)
    steps = np.diff(path.astype(np.int64), axis=0)
    assert all(tuple(s) in ((1, 0), (0, 1), (1, 1)) for s in steps)
    assert max(la, lb) <= path.shape[0] <= la + lb - 1


@pytest.mark.parametrize("seed", range(6))
def test_oracle_path_equals_numpy_twin_on_random_pairs(seed):
    rng = np.random.default_rng(seed)
    for _ in range(40):
        la, lb = (int(x) for x in rng.integers(1, 71, size=2))
        c = int(rng.integers(1, 14))
        if seed % 2:  # small integer frames: many exact ties, so the rule decides most steps
            a, b = rng.integers(0, 3, size=(la, c)).astype(np.float64), rng.integers(0, 3, size=(lb, c)).astype(np.float64)
        else:
            a, b = rng.normal(size=(la, c)) * 10, rng.normal(size=(lb, c)) * 10
        p = R.dtw_path(a, b)
        assert np.array_equal(p, R.twin_dtw_path(a, b)), (la, lb, c)
        check_shape(p, la, lb)
        # the path's cost is the distance: sum of local costs along it over (La + Lb), the order of A8 up to rounding
        cost = sum(float(np.sum((a[i] - b[j]) ** 2)) for i, j in p)
        assert math.isclose(cost / (la + lb), O.dtw(a, b), rel_tol=1e-12, abs_tol=1e-12)


def test_identical_constant_sequences_take_the_diagonal_first():
    a = np.ones((4, 3))
    assert np.array_equal(R.dtw_path(a, a), [[0, 0], [1, 1], [2, 2], [3, 3]])
    # every D is 0: diag wins every tie until row 0, which only has `left`
    b = np.ones((6, 3))
    want = [[0, 0], [0, 1], [0, 2], [1, 3], [2, 4], [3, 5]]
    assert np.array_equal(R.dtw_path(a, b), want) and np.array_equal(R.twin_dtw_path(a, b), want)
    want_t = [[0, 0], [1, 0], [2, 0], [3, 1], [4, 2], [5, 3]]  # column 0 only has `up`
    assert np.array_equal(R.dtw_path(b, a), want_t) and np.array_equal(R.twin_dtw_path(b, a), want_t)


def test_three_way_tie_goes_to_diag():
    # a = [0, 1, 0], b = [0, 2]: D = [[0, 4], [1, 1], [1, 5]]; at (2, 1) up = D(1,1) = 1, left = D(2,0) = 1, diag = D(1,0) = 1
    a, b = np.array([[0.0], [1.0], [0.0]]), np.array([[0.0], [2.0]])
    assert O.dtw(a, b) == 5.0 / 5
    want = [[0, 0], [1, 0], [2, 1]]
    assert np.array_equal(R.dtw_path(a, b), want) and np.array_equal(R.twin_dtw_path(a, b), want)


def test_left_and_diag_choices():
    # a = [0, 3, 0], b = [3, 0, 0]: D = [[9, 9, 9], [9, 18, 18], [18, 9, 9]]
    a, b = np.array([[0.0], [3.0], [0.0]]), np.array([[3.0], [0.0], [0.0]])
    # at (2, 2): up = D(1,2) = 18, left = D(2,1) = 9, diag = D(1,1) = 18 -> left; at (2, 1): up = D(1,1) = 18, left = D(2,0) = 18,
    # diag = D(1,0) = 9 -> diag; at (1, 0): column 0 -> up
    want = [[0, 0], [1, 0], [2, 1], [2, 2]]
    assert np.array_equal(R.dtw_path(a, b), want) and np.array_equal(R.twin_dtw_path(a, b), want)
    # diag ties with left: a = [0, 1, 1], b = [1, 1, 0]
    a, b = np.array([[0.0], [1.0], [1.0]]), np.array([[1.0], [1.0], [0.0]])
    D = np.array([[1, 2, 2], [1, 1, 2], [1, 1, 2]], dtype=np.float64)  # hand-worked
    assert O.dtw(a, b) == D[2, 2] / 6
    # (2, 2): up = D(1,2) = 2, left = D(2,1) = 1, diag = D(1,1) = 1 -> diag; (1, 1): up = 2, left = 1, diag = 1 -> diag
    want = [[0, 0], [1, 1], [2, 2]]
    assert np.array_equal(R.dtw_path(a, b), want) and np.array_equal(R.twin_dtw_path(a, b), want)


def test_row_zero_only_has_left():
    a, b = np.zeros((1, 2)), np.arange(10.0).reshape(5, 2)
    want = [[0, j] for j in range(5)]
    assert np.array_equal(R.dtw_path(a, b), want) and np.array_equal(R.twin_dtw_path(a, b), want)
    assert np.array_equal(R.dtw_path(b, a), [[i, 0] for i in range(5)])


def test_nan_counts_as_inf_and_non_finite_distances_have_no_path():
    a = np.array([[0.0], [1.0], [2.0], [3.0]])
    b = np.array([[0.0], [1.0], [np.nan], [3.0]])
    assert not math.isfinite(O.dtw(a, b))  # a NaN frame leaves every later cell NaN or +inf
    for f in (R.dtw_path, R.twin_dtw_path):
        assert f(a, b).shape == (0, 2)
        assert f(a, np.full((3, 1), 1e200)).shape == (0, 2)  # cost overflows to inf
        assert f(np.zeros((0, 1)), b).shape == (0, 2)
        assert f(a, np.zeros((0, 1))).shape == (0, 2)
