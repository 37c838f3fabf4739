"""The numpy twin of the warped resynthesis (tests/warp_reference.py, spec A11) against a per-sample restatement of the spec,
and property P1 (a diagonal or empty path gives ss_resynth's samples) against the oracle's resynthesis. CPU only."""
import numpy as np

import warp_reference as W
from oracle import oracle as O

H = W.H


def scalar(dict_samples, dict_off, match_idx, paths, target_lens):
    """A11 one output sample at a time, with Python floats (IEEE f64, one rounding per operation)."""
    out = []
    for t, L in enumerate(int(x) for x in target_lens):
        m = int(match_idx[t])
        base, ln = int(dict_off[m]), int(dict_off[m + 1]) - int(dict_off[m])
        X = lambda p: float(dict_samples[base + p]) if p < ln else 0.0
        P = [(int(i), int(j)) for i, j in paths[t]]
        lq = P[-1][0] + 1 if P else 0

        def jb(b):
            if not P:
                return b
            if b < lq:
                return next(j for i, j in P if i == b)
            return jb(lq - 1) + (b - lq + 1)

        for n in range(L):
            b, r = divmod(n, H)
            s = jb(b) * H
            a = X(s + r)
            if b == 0 or s == jb(b - 1) * H + H:
                out.append(a)
            else:
                sp = jb(b - 1) * H
                out.append(X(sp + H + r) * ((H - r) / H) + a * (r / H))
    return np.array(out, dtype=np.float64)


def random_case(rng, nseg, nd, to_corner):
    dlens = rng.integers(0, 3000, size=nd)
    dlens[:3] = (0, 1, 5 * H)  # empty, one sample, an exact number of hops
    doff = np.zeros(nd + 1, dtype=np.uint64)
    doff[1:] = np.cumsum(dlens)
    ds = rng.normal(size=int(doff[-1]))
    tl = rng.integers(0, 3000, size=nseg).astype(np.uint64)
    tl[:4] = (0, 1, H, 3 * H + 1)
    mi = rng.integers(0, nd, size=nseg).astype(np.uint32)
    paths = []
    for t in range(nseg):
        lq = int(tl[t]) // H if rng.random() < 0.8 else int(rng.integers(0, 16))  # usually the target's frames, sometimes not
        ld = int(dlens[mi[t]]) // H if rng.random() < 0.8 else int(rng.integers(0, 16))
        paths.append(W.random_path(rng, lq, ld, to_corner, p_diag=float(rng.uniform(0.0, 1.0))))
    return ds, doff, mi, paths, tl


def test_twin_equals_the_per_sample_spec_on_random_paths():
    rng = np.random.default_rng(11)
    seen = dict(partial=0, past_end=0, vertical=0, horizontal=0)
    for to_corner in (True, False):
        ds, doff, mi, paths, tl = random_case(rng, 60, 25, to_corner)
        cells, poff = W.flatten(paths)
        got = W.resynth_warped(ds, doff, mi, cells, poff, tl)
        want = scalar(ds, doff, mi, paths, tl)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
        for t, p in enumerate(paths):
            seen["partial"] += int(tl[t]) % H != 0
            dl = int(doff[mi[t] + 1] - doff[mi[t]])
            seen["past_end"] += (int(p[-1][1]) + 1) * H > dl if len(p) else 0
            if len(p) > 1:
                d = np.diff(p.astype(np.int64), axis=0)
                seen["vertical"] += int(np.sum((d[:, 0] == 1) & (d[:, 1] == 0)))  # a source frame repeated
                seen["horizontal"] += int(np.sum((d[:, 0] == 0) & (d[:, 1] == 1)))  # source frames skipped
    assert all(v > 0 for v in seen.values()), seen
    blend = scalar(np.arange(1.0, 2 * H + 1), np.array([0, 2 * H], dtype=np.uint64), [0], [np.array([(0, 0), (1, 0)], dtype=np.uint32)], [2 * H])
    r = np.arange(H)
    assert np.array_equal(blend[H:], (r + H + 1.0) * ((H - r) / H) + (r + 1.0) * (r / H))  # block 1 repeats frame 0: c = X(H + r), a = X(r)


def test_hand_worked_blocks():
    x = np.arange(1.0, 8 * H + 1)  # X(p) = p + 1 on one sound of 8 hops
    doff = np.array([0, 8 * H], dtype=np.uint64)
    path = np.array([(0, 0), (1, 1), (1, 2), (1, 3), (2, 3)], dtype=np.uint32)  # j(0) = 0, j(1) = 1, j(2) = 3, past the path 4, 5
    L = 5 * H - 7
    got = W.resynth_warped(x, doff, [0], path, np.array([0, 5], dtype=np.uint64), [L])
    r = np.arange(H)
    want = np.concatenate([x[:H], x[H:2 * H],  # blocks 0 and 1 contiguous
                           x[2 * H:3 * H] * ((H - r) / H) + x[3 * H:4 * H] * (r / H),  # block 2 jumps from frame 1 to 3: crossfade
                           x[4 * H:5 * H], x[5 * H:6 * H - 7]])  # 3, 4 run on at unit speed; partial last block
    assert np.array_equal(got, want)
    assert np.array_equal(got, scalar(x, doff, [0], [path], [L]))


def test_diagonal_and_empty_paths_give_the_plain_resynthesis():
    """P1, bit for bit against the oracle's clone_from_dictionary + to_sound"""
    rng = np.random.default_rng(12)
    ds, doff, mi, _, tl = random_case(rng, 80, 30, True)
    paths = []
    for t in range(80):
        n = int(tl[t]) // H + int(rng.integers(-2, 3)) if t % 3 else 0  # the diagonal may be shorter or longer than the target
        paths.append(np.stack([np.arange(max(n, 0))] * 2, axis=1).astype(np.uint32))
    cells, poff = W.flatten(paths)
    got = W.resynth_warped(ds, doff, mi, cells, poff, tl)
    assert np.array_equal(got.view(np.uint64), O.resynth(ds, doff, mi, tl).view(np.uint64))
