"""ss_dict_walk_dtw (DESIGN.md §3.1i): SoundSequence::from_distances for SS_DTW_TARGET on the device. Every step must be the
nq = 1 SS_DTW_TARGET match of the previous step's segment, bit for bit. Every comparison is exact: indices with array_equal,
distances by bits, against the host loop of nq = 1 matches and against the oracle's chain (O.dtw_matrix or, under a band, the
band checker, then tests/target_reference.py)."""
import ctypes as C

import numpy as np
import pytest

import band_reference as R
import target_reference as T
from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_DTW, SS_DTW_TARGET, SS_ERR_EMPTY_DICT, SS_ERR_INVALID, SoundsymError

pytestmark = pytest.mark.gpu
NONE = 0xFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def assert_same(got, want):
    assert np.array_equal(np.asarray(got[0], dtype=np.uint32), np.asarray(want[0], dtype=np.uint32)), \
        np.argwhere(np.asarray(got[0]) != np.asarray(want[0]))[:5]
    assert np.array_equal(bits(got[1]), bits(want[1])), np.argwhere(bits(got[1]) != bits(want[1]))[:5]


def flat_of(segs, c=13):
    off = np.zeros(len(segs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([s.shape[0] for s in segs])
    flat = np.concatenate(segs, axis=0) if int(off[-1]) else np.zeros((0, c))
    return np.ascontiguousarray(flat, dtype=np.float64), off


def seg(flat, off, i):
    return flat[int(off[i]):int(off[i + 1])]


def loop_chain(dev, flat, off, start, steps, index_base=0, mode=SS_DTW_TARGET):
    """the nq = 1 loop: step t matches the segment step t - 1 returned; after a step without a result the query is empty"""
    c = flat.shape[1]
    cur, idx, dist = start, [], []
    for t in steps:
        i, d = dev.match(cur, np.array([0, cur.shape[0]], dtype=np.uint64), mode, 1, None if t is None else [t])
        idx.append(int(i[0, 0]))
        dist.append(float(d[0, 0]))
        cur = seg(flat, off, int(i[0, 0]) - index_base) if i[0, 0] != NONE else np.zeros((0, c))
    return np.array(idx, dtype=np.uint32), np.array(dist)


def oracle_chain(flat, off, start, steps, r=0):
    c = flat.shape[1]
    segs = [seg(flat, off, i) for i in range(len(off) - 1)]
    cur, idx, dist = start, [], []
    for t in steps:
        if r == 0:
            row = O.dtw_matrix(flat, off, cur, np.array([0, cur.shape[0]], dtype=np.uint64), c)
        else:
            row = np.array([[R.dtw_band(cur, b, r) for b in segs]])
        i, e = T.target_topk(row, [0.0 if t is None else t], 1)
        idx.append(int(i[0, 0]))
        dist.append(float(e[0, 0]))
        cur = segs[int(i[0, 0])] if i[0, 0] != NONE else np.zeros((0, c))
    return np.array(idx, dtype=np.uint32), np.array(dist)


def mid_targets(flat, off, start, n, seed):
    """uniform between the 10th and 90th percentile of the start's D row"""
    row = O.dtw_matrix(flat, off, start, np.array([0, start.shape[0]], dtype=np.uint64), flat.shape[1])[0]
    lo, hi = np.nanquantile(row, [0.1, 0.9])
    return np.random.default_rng(seed).uniform(lo, hi, n)


@pytest.fixture(scope="module")
def config3():
    d, doff = synth.segments(10000, 13, seed=1234)
    q, qoff = synth.segments(1000, 13, seed=5678)
    return d, doff, seg(q, qoff, 0)


def test_config3_300_steps_at_mid_targets_and_at_zero(ctx, config3):
    d, doff, start = config3
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    steps = mid_targets(d, doff, start, 300, 1)
    got = dev.walk_dtw(start, steps)
    assert_same(got, loop_chain(dev, d, doff, start, steps))
    assert_same(got, oracle_chain(d, doff, start, steps))
    # distances = NULL: t = 0 at every step, SS_DTW's nq = 1 chain
    got0 = dev.walk_dtw(start, None, 40)
    assert_same(got0, loop_chain(dev, d, doff, start, [None] * 40, mode=SS_DTW))
    assert_same(got0, oracle_chain(d, doff, start, [None] * 40))


def test_config4_64_steps(ctx):
    d, doff = synth.segments(100000, 13, seed=1234)
    q, qoff = synth.segments(8, 13, seed=5678)
    start = seg(q, qoff, 0)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    steps = mid_targets(d, doff, start, 64, 2)
    got = dev.walk_dtw(start, steps)
    assert_same(got, loop_chain(dev, d, doff, start, steps))
    assert_same(got, oracle_chain(d, doff, start, steps))


def mixed():
    """segments of 1-400 frames plus one of 2 048 (index 60)"""
    d, doff = synth.segments(120, 13, lmin=1, lmax=400, seed=41)
    segs = [seg(d, doff, i) for i in range(120)]
    long_d = np.random.default_rng(42).normal(scale=3.0, size=(2048, 13))
    return flat_of(segs[:60] + [long_d] + segs[60:]), long_d


@pytest.mark.parametrize("r", [0, 1, 3])
def test_mixed_lengths_starts_and_the_long_segment_under_a_band(ctx, r):
    (d, doff), long_d = mixed()
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    dev.set_dtw_band(r)
    rng = np.random.default_rng(43)
    for lq in (1, 32, 33, 2048):
        start = rng.normal(scale=3.0, size=(lq, 13)) if lq != 2048 else long_d + 0.01 * rng.normal(size=long_d.shape)
        # step 0 is forced onto the 2 048-frame segment: its own D as the target (e = 0); then the long segment is the query
        d_long = R.dtw_band(start, long_d, r) if r else float(O.dtw_matrix(long_d, np.array([0, 2048], dtype=np.uint64), start,
                                                                              np.array([0, lq], dtype=np.uint64), 13)[0, 0])
        steps = np.concatenate([[d_long], rng.uniform(0.0, 200.0, 4)])
        got = dev.walk_dtw(start, steps)
        assert got[0][0] == 60
        assert_same(got, loop_chain(dev, d, doff, start, steps))
        assert_same(got, oracle_chain(d, doff, start, steps, r))


def test_band_wider_than_every_pair_gives_the_unbanded_bits(ctx):
    (d, doff), long_d = mixed()
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    start = long_d[:33] + 0.5
    steps = np.linspace(0.0, 150.0, 12)
    want = dev.walk_dtw(start, steps)
    dev.set_dtw_band(2048)
    assert_same(dev.walk_dtw(start, steps), want)


def tie_dictionary():
    """start: 4 frames of zeros. A1 (4 frames, cost 1 per cell): D = 4 / 8 = 0.5; A7 (4 frames, cost 7): D = 28 / 8 = 3.5;
    B (2 frames, cost 2.25): D = 9 / 6 = 1.5 - all exact. t = 1.0 ties A1 below with B above (e = 0.5), t = 2.5 ties B below
    with A7 above (e = 1.0); the shorter B comes first in the length order but sits at the higher indices"""
    rng = np.random.default_rng(51)
    far = [rng.normal(loc=40.0, size=(n, 13)) for n in (3, 9, 4, 2, 6)]
    a1 = np.zeros((4, 13)); a1[:, 0] = 1.0
    a7 = np.zeros((4, 13)); a7[:, :4] = [2.0, 1.0, 1.0, 1.0]
    b = np.zeros((2, 13)); b[:, 0] = 1.5
    segs = [far[0], a1, far[1], a7, b, far[2], b, a1, b, a7, far[3], far[4]]
    return flat_of(segs), np.zeros((4, 13))


@pytest.mark.parametrize("index_base", [0, 1000])
def test_ties_go_to_the_lowest_index_across_the_length_order(ctx, index_base):
    (d, doff), start = tie_dictionary()
    dev = api.DeviceDictionary(ctx, d, doff, 13, index_base=index_base)
    for t, want_i, want_e in ((1.0, 1, 0.5), (2.5, 3, 1.0), (1.5, 4, 0.0)):
        idx, dist = dev.walk_dtw(start, [t])
        assert idx[0] == want_i + index_base and dist[0] == want_e
    steps = [1.0, 0.0, 3.0, 2.5, 0.2, 1.5, 9.0, 0.0]
    got = dev.walk_dtw(start, steps)
    assert_same(got, loop_chain(dev, d, doff, start, steps, index_base))
    want = oracle_chain(d, doff, start, steps)
    assert_same(got, (np.where(want[0] == NONE, NONE, want[0] + index_base).astype(np.uint32), want[1]))


def test_nan_and_empty_segments(ctx):
    d, doff = synth.segments(400, 13, lmin=0, lmax=40, seed=61)
    d = d.copy()
    d[int(doff[7]) + 1, 3] = np.nan
    d[int(doff[100]):int(doff[101])] = np.nan
    start = seg(d, doff, 7)  # a start with a NaN frame
    steps = mid_targets(d, doff, seg(d, doff, 8), 30, 3)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    got = dev.walk_dtw(start, steps)
    assert_same(got, loop_chain(dev, d, doff, start, steps))
    assert_same(got, oracle_chain(d, doff, start, steps))


def test_no_result_steps(ctx):
    d, doff = synth.segments(300, 13, seed=71)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    none = (np.full(5, NONE, dtype=np.uint32), np.full(5, np.inf))
    assert_same(dev.walk_dtw(np.zeros((0, 13)), [0.5, 1.0, 0.0, 2.0, 3.0]), none)
    assert_same(dev.walk_dtw(np.zeros((0, 13)), None, 5), none)
    empty_segs = api.DeviceDictionary(ctx, np.zeros((0, 13)), np.zeros(6, dtype=np.uint64), 13)
    assert_same(empty_segs.walk_dtw(seg(d, doff, 0), [0.5, 1.0, 0.0, 2.0, 3.0]), none)
    # only NaN segments: no step has a result either
    nan_d = np.full((int(doff[4]), 13), np.nan)
    nan_dev = api.DeviceDictionary(ctx, nan_d, doff[:5], 13)
    assert_same(nan_dev.walk_dtw(seg(d, doff, 0), [0.5, 1.0, 0.0, 2.0, 3.0]), none)


def test_dev_form_equals_host_form_and_launches_nsteps(ctx):
    import torch
    d, doff = synth.segments(3000, 13, lmin=1, lmax=60, seed=81)
    start = seg(d, doff, 11) + 0.25
    steps = mid_targets(d, doff, start, 25, 4)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    host = dev.walk_dtw(start, steps)
    sq = api.DeviceQueries(ctx, start, np.array([0, start.shape[0]], dtype=np.uint64))
    d_t = torch.from_numpy(np.ascontiguousarray(steps)).cuda()
    d_i = torch.empty(25, dtype=torch.int32, device="cuda")
    d_d = torch.empty(25, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    for ptr, want in ((d_t.data_ptr(), host), (None, dev.walk_dtw(start, None, 25))):
        n0 = ctx.launches
        ctx.check(ctx.lib.ss_dict_walk_dtw_dev(dev.h, sq.h, ptr, 25, d_i.data_ptr(), d_d.data_ptr()))
        assert ctx.launches - n0 == 25
        ctx.sync()
        assert_same((d_i.cpu().numpy().view(np.uint32), d_d.cpu().numpy()), want)
    for n in (1, 9):
        n0 = ctx.launches
        dev.walk_dtw(start, steps[:n])
        assert ctx.launches - n0 == n
    n0 = ctx.launches
    assert ctx.lib.ss_dict_walk_dtw_dev(dev.h, sq.h, None, 0, None, None) == 0
    assert dev.walk_dtw(start, [])[0].shape == (0,)
    assert ctx.launches == n0


def test_after_a_pending_dtw_match_and_interleaved_with_cosine_walks(ctx):
    import torch
    d, doff = synth.segments(4000, 13, seed=91)
    q, qoff = synth.segments(96, 13, seed=92)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    want_dtw = dev.match(q, qoff, SS_DTW, 2)
    start = seg(q, qoff, 5)
    steps = mid_targets(d, doff, start, 20, 5)
    cos_steps = np.random.default_rng(6).uniform(-0.5, 0.5, 20)
    want_walk = loop_chain(dev, d, doff, start, steps)
    want_cos = dev.walk(start, cos_steps)
    # a pending _dev SS_DTW match completes first; the ss_dict_last_* readers keep describing it
    qs = api.DeviceQueries(ctx, q, qoff)
    o_idx = torch.empty((96, 2), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((96, 2), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 2, o_idx.data_ptr(), o_dist.data_ptr()))
    got = dev.walk_dtw(start, steps)
    ctx.sync()
    assert np.array_equal(o_idx.cpu().numpy().view(np.uint32), want_dtw[0])
    assert np.array_equal(bits(o_dist.cpu().numpy()), bits(want_dtw[1]))
    assert_same(got, want_walk)
    last = (dev.last_scan_kind, dev.last_work, dev.last_uncertified, dev.last_tc_fallback, dev.last_exhaustive)
    for _ in range(2):
        assert_same(dev.walk(start, cos_steps), want_cos)
        assert_same(dev.walk_dtw(start, steps), want_walk)
    assert (dev.last_scan_kind, dev.last_work, dev.last_uncertified, dev.last_tc_fallback, dev.last_exhaustive) == last


def test_errors(ctx):
    import torch
    L = ctx.lib
    d, doff = synth.segments(200, 13, seed=5)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    start = seg(d, doff, 2)
    t = np.array([1.0, 0.5, 0.0])
    idx = np.empty(3, dtype=np.uint32)
    dist = np.empty(3, dtype=np.float64)
    P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    assert L.ss_dict_walk_dtw(None, P(start), start.shape[0], P(t), 3, P(idx), P(dist)) == SS_ERR_INVALID
    assert L.ss_dict_walk_dtw(dev.h, P(start), start.shape[0], P(t), 3, None, P(dist)) == SS_ERR_INVALID
    assert L.ss_dict_walk_dtw(dev.h, P(start), start.shape[0], P(t), 3, P(idx), None) == SS_ERR_INVALID
    assert L.ss_dict_walk_dtw(dev.h, None, 4, P(t), 3, P(idx), P(dist)) == SS_ERR_INVALID
    for bad in (np.nan, np.inf, -np.inf):
        with pytest.raises(SoundsymError) as e:
            dev.walk_dtw(start, [0.5, bad, 0.5])
        assert e.value.code == SS_ERR_INVALID
    empty = api.DeviceDictionary(ctx, np.zeros((0, 13)), np.zeros(1, dtype=np.uint64), 13)
    assert L.ss_dict_walk_dtw(empty.h, P(start), start.shape[0], P(t), 3, P(idx), P(dist)) == SS_ERR_EMPTY_DICT
    n0 = ctx.launches
    assert L.ss_dict_walk_dtw(dev.h, P(start), start.shape[0], P(t), 0, None, None) == 0
    assert ctx.launches == n0
    s12 = api.DeviceQueries(ctx, np.zeros((5, 12)), np.array([0, 5], dtype=np.uint64))
    s2 = api.DeviceQueries(ctx, d[:9], np.array([0, 4, 9], dtype=np.uint64))
    s1 = api.DeviceQueries(ctx, start, np.array([0, start.shape[0]], dtype=np.uint64))
    d_t = torch.from_numpy(t).cuda()
    d_i = torch.empty(3, dtype=torch.int32, device="cuda")
    d_d = torch.empty(3, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    assert L.ss_dict_walk_dtw_dev(dev.h, s12.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dtw_dev(dev.h, s2.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dtw_dev(dev.h, s1.h, d_t.data_ptr(), 3, None, d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dtw_dev(dev.h, None, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dtw_dev(empty.h, s1.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_EMPTY_DICT
    other = api.Context(0)
    so = api.DeviceQueries(other, start, np.array([0, start.shape[0]], dtype=np.uint64))
    assert L.ss_dict_walk_dtw_dev(dev.h, so.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    # the dictionary still walks correctly after the refusals
    assert_same(dev.walk_dtw(start, t), oracle_chain(d, doff, start, t))


def sequence_dictionary(ctx, section71, mode):
    from test_sequence_gpu import cut_offsets
    s16 = O.decode_pcm(section71["pcm"].astype(np.int32), 16)
    snd = api.Sound(s16, 44100.0, section71["mfcc"], None, section71["mfcc"].mean(axis=0), None, ctx)
    doff = cut_offsets(section71["splits_d3t4"])
    return api.SoundDictionary.from_segments(snd, section71["splits_d3t4"], ctx, mode), section71["mfcc"][: int(doff[-1])], doff


def test_python_mirror_routes_dtw_target_to_the_walk(ctx, section71, sample_excerpt, monkeypatch):
    d, dm, doff = sequence_dictionary(ctx, section71, SS_DTW_TARGET)
    qm = sample_excerpt["mfcc"]
    start_m = qm[:9]
    start = api.Sound(np.zeros(9 * 256 + 768), 44100.0, start_m, None, start_m.mean(axis=0), None, ctx)
    steps = mid_targets(dm, doff, start_m, 24, 7)
    want = oracle_chain(dm, doff, start_m, steps)
    assert_same(d._device().walk_dtw(start_m, steps), want)
    assert_same(d._device().walk_dtw(start_m, steps), loop_chain(d._device(), dm, doff, start_m, steps))
    # from_distances takes the walk (no nq = 1 match) and returns the same sounds
    n_match = []
    orig = api.DeviceDictionary.match
    monkeypatch.setattr(api.DeviceDictionary, "match", lambda self, *a, **k: n_match.append(1) or orig(self, *a, **k))
    chain = api.SoundSequence.from_distances(list(steps), start, d)
    assert not n_match
    assert [d.sounds.index(s) for s in chain.sounds()[1:]] == [int(i) for i in want[0]]
    # a step without a result raises IndexError there, as the loop's at_distance does
    with pytest.raises(IndexError):
        api.SoundSequence.from_distances([0.5, 0.5], api.Sound(np.zeros(0), 44100.0, np.zeros((0, 12)), None, np.full(12, np.nan), None, ctx), d)
    # SS_DTW keeps the loop
    d_dtw, _, _ = sequence_dictionary(ctx, section71, SS_DTW)
    chain = api.SoundSequence.from_distances([0.5, 1.0], start, d_dtw)
    assert n_match
