"""ss_dict_walk: SoundSequence::from_distances (src/sound.rs:405-417) for SS_COSINE_REF on the device. Every step must be the
bits of ss_dict_match(nq = 1, SS_COSINE_REF, targets = [distances[t]]) on the segment the previous step returned (step 0: the
start sound), and so of the CPU reference run step by step. Every comparison is exact: indices with ==, distances bit for bit."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_COSINE_REF, SS_DTW, SS_ERR_EMPTY_DICT, SS_ERR_INVALID

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def flat_of(segs, c):
    off = np.zeros(len(segs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([s.shape[0] for s in segs])
    flat = np.concatenate(segs, axis=0) if int(off[-1]) else np.zeros((0, c))
    return np.ascontiguousarray(flat, dtype=np.float64), off


def seg(flat, off, i):
    return flat[int(off[i]):int(off[i + 1])]


def oracle_chain(flat, off, c, start, steps):
    """the reference's chain, one at_distance per step"""
    idx, dist, cur = [], [], start
    for t in steps:
        oi, od = O.cosine_match(flat, off, cur, np.array([0, cur.shape[0]], dtype=np.uint64), c, np.array([t], dtype=np.float64))
        idx.append(int(oi[0]))
        dist.append(float(od[0]))
        cur = seg(flat, off, int(oi[0]))
    return np.array(idx, dtype=np.uint32), np.array(dist)


def match_chain(dev, flat, off, start, steps, base=0):
    """the host loop the walk replaces: ss_dict_match(nq = 1) per step"""
    idx, dist, cur = [], [], start
    for t in steps:
        i, d = dev.match(cur, np.array([0, cur.shape[0]], dtype=np.uint64), SS_COSINE_REF, 1, [t])
        idx.append(int(i[0, 0]))
        dist.append(float(d[0, 0]))
        cur = seg(flat, off, int(i[0, 0]) - base)
    return np.array(idx, dtype=np.uint32), np.array(dist)


def assert_same(got, want):
    gi, gd = got
    wi, wd = want
    assert np.array_equal(gi, wi), np.flatnonzero(gi != wi)[:10]
    assert np.array_equal(bits(gd), bits(wd)), np.flatnonzero(bits(gd) != bits(wd))[:10]


def cut_offsets(splits, hop=256):
    frames = (np.asarray(splits, dtype=np.uint64) // np.uint64(hop)).astype(np.uint64)
    off = np.zeros(len(frames) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(frames)
    return off


def test_walk_on_fixtures_equals_the_reference_chain(ctx, section71, sample_excerpt):
    doff, qoff = cut_offsets(section71["splits_d3t4"]), cut_offsets(sample_excerpt["splits_d3t4"])
    dm, qm = section71["mfcc"][: int(doff[-1])], sample_excerpt["mfcc"][: int(qoff[-1])]
    dev = api.DeviceDictionary(ctx, dm, doff, 12)
    start = seg(qm, qoff, 3)
    steps = [1.0, 0.0, 1e-4, -1e-4, 5e-5, float("nan"), 1.0, -2e-5, 0.5, -1.0, 2.0, 1e-4, 0.0, 3e-5, float("nan"), 0.9, -0.5, 1e-4]
    got = dev.walk(start, steps)
    assert_same(got, oracle_chain(dm, doff, 12, start, steps))
    assert_same(got, match_chain(dev, dm, doff, start, steps))
    # the Python mirror goes through the walk and returns the reference's sounds
    snd = api.Sound(np.zeros(int(doff[-1]) * 256), 44100.0, dm, None, dm.mean(axis=0), None, ctx)
    d = api.SoundDictionary.from_segments(snd, section71["splits_d3t4"], ctx, SS_COSINE_REF)
    q = api.Sound(np.zeros(start.shape[0] * 256), 44100.0, start, None, start.mean(axis=0), None, ctx)
    chain = api.SoundSequence.from_distances(steps, q, d)
    assert chain.sounds()[0] is q
    assert [d.sounds.index(s) for s in chain.sounds()[1:]] == [int(i) for i in got[0]]


@pytest.mark.parametrize("nd,nsteps", [(10000, 300), (100000, 64)])
def test_walk_equals_the_host_loop_of_nq1_matches(ctx, nd, nsteps):
    flat, off = synth.segments(nd, 13, seed=1234)
    dev = api.DeviceDictionary(ctx, flat, off)
    q, qoff = synth.segments(4, 13, seed=5678)
    rng = np.random.default_rng(nd + nsteps)
    steps = rng.uniform(-1.0, 1.0, nsteps)
    steps[::7] = 1.0
    steps[3::11] = 0.0
    steps[5::13] = np.nan
    start = seg(q, qoff, 1)
    got = dev.walk(start, steps)
    assert_same(got, match_chain(dev, flat, off, start, steps))
    assert len(set(got[0].tolist())) > 1  # the chain moves through the dictionary


def test_walk_reports_index_base_and_follows_the_local_segment(ctx):
    flat, off = synth.segments(3000, 13, seed=77)
    base = 123456
    dev = api.DeviceDictionary(ctx, flat, off, 13, index_base=base)
    steps = np.random.default_rng(3).uniform(-0.5, 0.5, 40)
    start = seg(flat, off, 17)
    got = dev.walk(start, steps)
    assert np.all(got[0] >= base)
    assert_same(got, match_chain(dev, flat, off, start, steps, base))
    wi, wd = oracle_chain(flat, off, 13, start, steps)
    assert_same((got[0] - base, got[1]), (wi, wd))


def test_walk_tie_goes_to_the_smaller_index_across_the_walk_order(ctx):
    rng = np.random.default_rng(11)
    c = 13
    segs = [rng.normal(size=(int(rng.integers(4, 33)), c)) for _ in range(20000)]
    a = rng.normal(size=(8, c))                                 # 104 values: whole chunks of 8, no tail
    segs[19000] = a                                             # short: early in the (length, index) walk order
    segs[7] = np.concatenate([a, np.zeros((24, c))])            # same sim exactly, longer, smaller index
    segs[15000] = np.concatenate([a, np.zeros((9, c))])         # same sim, larger index
    flat, off = flat_of(segs, c)
    dev = api.DeviceDictionary(ctx, flat, off)
    steps = [1.0, 1.0, 1.0, 0.0, 1.0]
    got = dev.walk(a, steps)
    assert got[0][0] == 7 and got[0][1] == 7
    assert_same(got, oracle_chain(flat, off, c, a, steps))
    assert_same(got, match_chain(dev, flat, off, a, steps))


def unit_frames(c, cols):
    v = np.zeros((2, c))
    v[0, cols[:2]] = 0.5
    v[1, cols[2:]] = 0.5                                        # |v|^2 = 4 * 0.25 = 1 exactly
    return v


def test_walk_distance_two_never_beats_the_seed(ctx):
    c = 13
    v, w = unit_frames(c, [0, 1, 3, 4]), unit_frames(c, [5, 6, 8, 9])  # sim(v, -v) = -1, sim(v, w) = 0 exactly
    lens = np.random.default_rng(5).integers(1, 9, size=5000)
    segs = [np.zeros((int(n), c)) for n in lens]                # all-zero: similarity 0/0 = NaN
    segs[4000] = -v                                             # at distance 2.0 for target 1.0 (and 3.0 for target 2.0)
    segs[2500] = w                                              # at distance 2.0 for target 2.0 (and 1.0 for target 1.0)
    flat, off = flat_of(segs, c)
    dev = api.DeviceDictionary(ctx, flat, off)
    # step 0: nothing is below 2.0, so the seed (0, 2.0) stays; step 1 queries segment 0 (all-zero): NaN against everything
    steps = [2.0, 1.0, 1.0]
    got = dev.walk(v, steps)
    assert got[0].tolist() == [0, 0, 0] and got[1].tolist() == [2.0, 2.0, 2.0]
    assert_same(got, oracle_chain(flat, off, c, v, steps))
    assert_same(got, match_chain(dev, flat, off, v, steps))
    # without w, target 1.0: -v alone at exactly 2.0 loses to the seed too
    segs[2500] = np.zeros((3, c))
    flat, off = flat_of(segs, c)
    dev = api.DeviceDictionary(ctx, flat, off)
    got = dev.walk(v, [1.0, 1.0])
    assert got[0].tolist() == [0, 0] and got[1].tolist() == [2.0, 2.0]
    assert_same(got, oracle_chain(flat, off, c, v, [1.0, 1.0]))
    assert_same(got, match_chain(dev, flat, off, v, [1.0, 1.0]))


def test_walk_after_the_seed_the_next_step_starts_from_segment_0(ctx):
    c = 13
    v = unit_frames(c, [0, 1, 3, 4])
    segs = [np.zeros((int(n), c)) for n in (3, 5, 2, 4, 6, 2, 7)]
    segs[0] = -v
    segs[3] = -v
    flat, off = flat_of(segs, c)
    dev = api.DeviceDictionary(ctx, flat, off)
    got = dev.walk(v, [1.0, 1.0, 0.0])
    # step 0: (0, 2.0); step 1 queries segment 0 = -v: sim 1, distance 0 (from v it would be 2.0 again)
    assert got[0].tolist() == [0, 0, 0] and got[1][0] == 2.0 and got[1][1] == 0.0 and got[1][2] == 1.0
    assert_same(got, oracle_chain(flat, off, c, v, [1.0, 1.0, 0.0]))
    assert_same(got, match_chain(dev, flat, off, v, [1.0, 1.0, 0.0]))


def test_walk_from_an_empty_start_sound(ctx):
    flat, off = synth.segments(500, 13, seed=9)
    dev = api.DeviceDictionary(ctx, flat, off)
    start = np.zeros((0, 13))
    steps = [1.0, 0.3, -0.2, 0.0]
    got = dev.walk(start, steps)
    assert got[0][0] == 0 and got[1][0] == 2.0  # 0/0 against everything: the fold's seed
    assert_same(got, oracle_chain(flat, off, 13, start, steps))
    assert_same(got, match_chain(dev, flat, off, start, steps))


def test_walk_with_sequences_longer_than_the_staged_query(ctx):
    rng = np.random.default_rng(21)
    c = 13
    lens = list(rng.integers(4, 401, size=300)) + [3000]
    lens[50] = 0                                               # an empty segment: NaN against everything
    segs = [rng.normal(size=(int(n), c)) for n in lens]
    rng.shuffle(segs)
    flat, off = flat_of(segs, c)
    dev = api.DeviceDictionary(ctx, flat, off)
    start = rng.normal(size=(2500, c))
    steps = rng.uniform(-0.1, 0.1, 24)
    steps[::5] = 0.0
    got = dev.walk(start, steps)
    assert_same(got, oracle_chain(flat, off, c, start, steps))
    assert_same(got, match_chain(dev, flat, off, start, steps))
    # and from the longest segment itself
    longest = int(np.argmax(np.diff(off)))
    got = dev.walk(seg(flat, off, longest), steps[:8])
    assert_same(got, oracle_chain(flat, off, c, seg(flat, off, longest), steps[:8]))


def test_walk_after_a_pending_dtw_match_and_before_a_cosine_match(ctx):
    import torch
    flat, off = synth.segments(4000, 13, seed=31)
    q, qoff = synth.segments(96, 13, seed=32)
    dev = api.DeviceDictionary(ctx, flat, off)
    want_dtw = dev.match(q, qoff, SS_DTW, 2)
    want_cos = dev.match(q, qoff, SS_COSINE_REF, 1, np.linspace(-0.5, 0.5, 96))
    steps = np.random.default_rng(4).uniform(-0.5, 0.5, 30)
    start = seg(q, qoff, 5)
    want_walk = match_chain(dev, flat, off, start, steps)
    # the walk never changes the ss_dict_last_* counters
    dev.match(q, qoff, SS_COSINE_REF, 1, np.linspace(-0.5, 0.5, 96))
    kind, work = dev.last_scan_kind, dev.last_work
    dev.walk(start, steps)
    assert (dev.last_scan_kind, dev.last_work) == (kind, work)
    qs = api.DeviceQueries(ctx, q, qoff)
    o_idx = torch.empty((96, 2), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((96, 2), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 2, o_idx.data_ptr(), o_dist.data_ptr()))
    got_walk = dev.walk(start, steps)  # completes the pending DTW match first
    ctx.check(ctx.lib.ss_dict_match_finish(dev.h))
    ctx.sync()
    assert np.array_equal(o_idx.cpu().numpy().view(np.uint32), want_dtw[0])
    assert np.array_equal(bits(o_dist.cpu().numpy()), bits(want_dtw[1]))
    assert_same(got_walk, want_walk)
    got_cos = dev.match(q, qoff, SS_COSINE_REF, 1, np.linspace(-0.5, 0.5, 96))
    assert np.array_equal(got_cos[0], want_cos[0]) and np.array_equal(bits(got_cos[1]), bits(want_cos[1]))
    # the device entry point gives the same chain
    sq = api.DeviceQueries(ctx, start, np.array([0, start.shape[0]], dtype=np.uint64))
    d_t = torch.from_numpy(np.ascontiguousarray(steps)).cuda()
    d_i = torch.empty(len(steps), dtype=torch.int32, device="cuda")
    d_d = torch.empty(len(steps), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_walk_dev(dev.h, sq.h, d_t.data_ptr(), len(steps), d_i.data_ptr(), d_d.data_ptr()))
    ctx.sync()
    assert_same((d_i.cpu().numpy().view(np.uint32), d_d.cpu().numpy()), want_walk)


def test_walk_errors(ctx):
    import torch
    L = ctx.lib
    flat, off = synth.segments(200, 13, seed=5)
    dev = api.DeviceDictionary(ctx, flat, off)
    start = seg(flat, off, 2)
    t = np.array([1.0, 0.5, 0.0])
    idx = np.empty(3, dtype=np.uint32)
    dist = np.empty(3, dtype=np.float64)
    P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    assert L.ss_dict_walk(None, P(start), start.shape[0], P(t), 3, P(idx), P(dist)) == SS_ERR_INVALID
    assert L.ss_dict_walk(dev.h, P(start), start.shape[0], P(t), 3, None, P(dist)) == SS_ERR_INVALID
    assert L.ss_dict_walk(dev.h, P(start), start.shape[0], P(t), 3, P(idx), None) == SS_ERR_INVALID
    assert L.ss_dict_walk(dev.h, None, 4, P(t), 3, P(idx), P(dist)) == SS_ERR_INVALID
    empty = api.DeviceDictionary(ctx, np.zeros((0, 13)), np.zeros(1, dtype=np.uint64), 13)
    assert L.ss_dict_walk(empty.h, P(start), start.shape[0], P(t), 3, P(idx), P(dist)) == SS_ERR_EMPTY_DICT
    with pytest.raises(api.SoundsymError):
        empty.walk(start, t)
    n0 = ctx.launches
    assert L.ss_dict_walk(dev.h, P(start), start.shape[0], P(t), 0, None, None) == 0
    assert ctx.launches == n0
    # device entry point: ncoeffs mismatch, start with nq = 2, NULL outputs, nsteps = 0
    s12 = api.DeviceQueries(ctx, np.zeros((5, 12)), np.array([0, 5], dtype=np.uint64))
    s2 = api.DeviceQueries(ctx, flat[:9], np.array([0, 4, 9], dtype=np.uint64))
    s1 = api.DeviceQueries(ctx, start, np.array([0, start.shape[0]], dtype=np.uint64))
    d_t = torch.from_numpy(t).cuda()
    d_i = torch.empty(3, dtype=torch.int32, device="cuda")
    d_d = torch.empty(3, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    assert L.ss_dict_walk_dev(dev.h, s12.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dev(dev.h, s2.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dev(dev.h, s1.h, d_t.data_ptr(), 3, None, d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dev(dev.h, None, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    assert L.ss_dict_walk_dev(empty.h, s1.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_EMPTY_DICT
    n0 = ctx.launches
    assert L.ss_dict_walk_dev(dev.h, s1.h, None, 0, None, None) == 0
    assert ctx.launches == n0
    # a different context
    other = api.Context(0)
    so = api.DeviceQueries(other, start, np.array([0, start.shape[0]], dtype=np.uint64))
    assert L.ss_dict_walk_dev(dev.h, so.h, d_t.data_ptr(), 3, d_i.data_ptr(), d_d.data_ptr()) == SS_ERR_INVALID
    # the dictionary still walks correctly after the refusals
    assert_same(dev.walk(start, t), oracle_chain(flat, off, 13, start, t))


def test_walk_launch_count_is_nsteps_plus_one(ctx):
    flat, off = synth.segments(2000, 13, seed=8)
    dev = api.DeviceDictionary(ctx, flat, off)
    start = seg(flat, off, 0)
    for n in (5, 17):
        n0 = ctx.launches
        dev.walk(start, np.linspace(-0.3, 0.3, n))
        assert ctx.launches - n0 == n + 1  # the start query's norm, then one launch per step


def test_from_distances_keeps_the_loop_for_dtw_and_an_empty_chain_builds_nothing(ctx):
    flat, off = synth.segments(300, 12, seed=12)
    snd = api.Sound(np.zeros(int(off[-1]) * 256), 44100.0, flat, None, flat.mean(axis=0), None, ctx)
    splits = (np.diff(off).astype(np.int64) * 256).tolist()
    d = api.SoundDictionary.from_segments(snd, splits, ctx, SS_DTW)
    start = d.sounds[4]
    chain = api.SoundSequence.from_distances([0.5, -0.5, 1.0], start, d)
    cur, want = start, []
    for t in (0.5, -0.5, 1.0):
        cur = d.at_distance(t, cur)
        want.append(cur)
    assert all(a is b for a, b in zip(chain.sounds()[1:], want))
    # an empty chain returns [start] without a device dictionary, even over an empty dictionary
    e = api.SoundDictionary(ctx, SS_COSINE_REF)
    assert [s is start for s in api.SoundSequence.from_distances([], start, e).sounds()] == [True]
    assert e._dev is None
    with pytest.raises(api.SoundsymError):
        api.SoundSequence.from_distances([1.0], start, e)
