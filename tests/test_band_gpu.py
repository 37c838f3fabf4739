"""ss_dict_set_dtw_band: SS_DTW matches and ss_dict_align under a Sakoe-Chiba band (spec A10, DESIGN.md §3.1f), on the device.
Every comparison is exact: indices with array_equal, distances by bits, against the banded checker tests/cpp/dtw_band.cpp."""
import numpy as np
import pytest

import band_reference as R
from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_COSINE_REF, SS_DTW

pytestmark = pytest.mark.gpu
NONE = 0xFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def check(idx, dist, oidx, odist):
    assert np.array_equal(idx, oidx), np.argwhere(idx != oidx)[:5]
    assert np.array_equal(bits(dist), bits(odist))


def flat_of(segs, c=13):
    off = np.zeros(len(segs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([s.shape[0] for s in segs])
    flat = np.concatenate(segs, axis=0) if int(off[-1]) else np.zeros((0, c))
    return np.ascontiguousarray(flat, dtype=np.float64), off


@pytest.fixture(scope="module")
def config3():
    d, doff = synth.segments(10000, 13, seed=1234)
    q, qoff = synth.segments(1000, 13, seed=5678)
    return d, doff, q, qoff


@pytest.mark.parametrize("r", [1, 3, 8])
def test_config3_every_query_every_first_stage(ctx, config3, r):
    d, doff, q, qoff = config3
    oidx, odist = R.dtw_band_topk(d, doff, q, qoff, 13, 8, r)
    if r == 1:  # the band changes the answer of this workload
        free_idx, _ = R.dtw_band_topk(d, doff, q, qoff, 13, 1, 0)  # (r = 0 is orc_dtw: tests/test_band_cpu.py)
        assert np.sum(free_idx[:, 0] != oidx[:, 0]) > 0
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    dev.set_dtw_band(r)
    assert dev.dtw_band == r
    for first_stage in range(4):
        dev.set_scan(first_stage)
        for k in (1, 8):
            idx, dist = dev.match(q, qoff, SS_DTW, k)
            check(idx, dist, oidx[:, :k], odist[:, :k])
            assert dev.last_uncertified == 0, (first_stage, k)


@pytest.mark.parametrize("r", [1, 16])
def test_mixed_lengths_1_to_400(ctx, r):
    d, doff = synth.segments(300, 13, lmin=1, lmax=400, seed=61)
    q, qoff = synth.segments(40, 13, lmin=1, lmax=400, seed=62)
    oidx, odist = R.dtw_band_topk(d, doff, q, qoff, 13, 2, r)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    dev.set_dtw_band(r)
    idx, dist = dev.match(q, qoff, SS_DTW, 2)
    check(idx, dist, oidx, odist)
    assert dev.last_uncertified == 0


@pytest.mark.parametrize("r", [1, 16])
def test_2048_frame_pair(ctx, r):
    rng = np.random.default_rng(7)
    dsegs = [rng.normal(size=(2048, 13)), rng.normal(size=(2048, 13)) + 0.5, rng.normal(size=(700, 13))]
    a = dsegs[0] + 0.1 * rng.normal(size=(2048, 13))
    d, doff = flat_of(dsegs)
    q, qoff = flat_of([np.roll(a, 3 * r, axis=0)])  # a shift the band only partly allows
    oidx, odist = R.dtw_band_topk(d, doff, q, qoff, 13, 3, r)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    dev.set_dtw_band(r)
    idx, dist = dev.match(q, qoff, SS_DTW, 3)
    check(idx, dist, oidx, odist)
    paths, pdist = dev.align(q, qoff, idx[:, 0])
    assert np.array_equal(paths[0], R.dtw_band_path(q, d[int(doff[idx[0, 0]]):int(doff[idx[0, 0] + 1])], r))
    assert np.array_equal(bits(pdist), bits(dist[:, 0]))


def near_duplicates(seg_len, seed):
    rng = np.random.default_rng(seed)
    base, boff = synth.segments(64, 13, lmin=seg_len // 2, lmax=seg_len, seed=seed)
    seg = base[int(boff[3]):int(boff[4])]
    L = len(seg)
    copies = [seg + rng.normal(size=seg.shape) * 1e-4 for _ in range(40)] + [seg.copy(), seg.copy()]
    d = np.concatenate([base] + copies)
    doff = np.concatenate([boff, boff[-1] + np.uint64(L) * np.arange(1, len(copies) + 1, dtype=np.uint64)]).astype(np.uint64)
    q = np.concatenate([seg, base[int(boff[10]):int(boff[11])]])
    qoff = np.array([0, L, L + int(boff[11] - boff[10])], dtype=np.uint64)
    return d, doff, q, qoff


@pytest.mark.parametrize("seg_len,first_stages", [(32, (3, 2)), (60, (3,))])
def test_near_duplicates_drive_the_banded_exhaustive_stage(ctx, seg_len, first_stages):
    d, doff, q, qoff = near_duplicates(seg_len, seed=9)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    for r in (1, 2):
        oidx, odist = R.dtw_band_topk(d, doff, q, qoff, 13, 4, r)
        dev.set_dtw_band(r)
        for first_stage in first_stages:
            dev.set_scan(first_stage)
            idx, dist = dev.match(q, qoff, SS_DTW, 4)
            check(idx, dist, oidx, odist)
            assert dist[0, 0] == 0.0 and dev.last_exhaustive >= 1 and dev.last_uncertified == 0, (r, first_stage)


def test_wide_band_and_band_zero_reproduce_the_unbanded_match(ctx):
    d, doff = synth.segments(2000, 13, lmin=1, lmax=90, seed=71)
    q, qoff = synth.segments(200, 13, lmin=1, lmax=90, seed=72)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    free_idx, free_dist = dev.match(q, qoff, SS_DTW, 4)
    oidx, odist = O.dtw_topk(d, doff, q, qoff, 13, 4)
    check(free_idx, free_dist, oidx, odist)
    dev.set_dtw_band(2)
    bidx, bdist = dev.match(q, qoff, SS_DTW, 4)
    check(bidx, bdist, *R.dtw_band_topk(d, doff, q, qoff, 13, 4, 2))
    assert not np.array_equal(bits(bdist), bits(free_dist))
    for r in (2048, 0):
        dev.set_dtw_band(r)
        idx, dist = dev.match(q, qoff, SS_DTW, 4)
        check(idx, dist, free_idx, free_dist)
        paths, pdist = dev.align(q, qoff, idx[:, 0])
        assert np.array_equal(bits(pdist), bits(dist[:, 0]))


def check_band_paths(paths, pdist, dflat, doff, qflat, qoff, idx, r):
    for p in range(len(paths)):
        a = qflat[int(qoff[p]):int(qoff[p + 1])]
        b = dflat[int(doff[idx[p]]):int(doff[idx[p] + 1])]
        want = R.dtw_band_path(a, b, r)
        assert np.array_equal(paths[p], want), (p, a.shape[0], b.shape[0])
        assert all(R.in_band(int(i), int(j), a.shape[0], b.shape[0], r) for i, j in paths[p])
        e = R.dtw_band(a, b, r)
        assert bits(pdist[p]) == bits(e if np.isfinite(e) else np.inf), p


@pytest.mark.parametrize("r", [1, 4])
def test_align_with_a_band(ctx, r):
    d, doff = synth.segments(400, 13, lmin=1, lmax=140, seed=81)
    q, qoff = synth.segments(120, 13, lmin=1, lmax=140, seed=82)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    dev.set_dtw_band(r)
    idx, mdist = dev.match(q, qoff, SS_DTW, 1)
    paths, pdist = dev.align(q, qoff, idx[:, 0])
    assert np.array_equal(bits(pdist), bits(mdist[:, 0]))
    check_band_paths(paths, pdist, d, doff, q, qoff, idx[:, 0], r)
    fixed = np.arange(120, dtype=np.uint32) * 3 % 400  # pairs the match did not choose, short and long mixed
    paths, pdist = dev.align(q, qoff, fixed)
    check_band_paths(paths, pdist, d, doff, q, qoff, fixed, r)


def test_align_with_a_band_spanning_two_direction_waves(ctx):
    """300 queries of 2 048 frames against a dictionary whose longest segment is 2 048 frames: two direction waves"""
    rng = np.random.default_rng(5)
    dsegs = [rng.normal(size=(n, 13)) for n in (40, 2048, 33, 17)]
    dflat, doff = flat_of(dsegs)
    dev = api.DeviceDictionary(ctx, dflat, doff, 13)
    dev.set_dtw_band(3)
    nq = 300
    qflat = rng.normal(size=(nq * 2048, 13))
    qoff = np.arange(nq + 1, dtype=np.uint64) * 2048
    idx = np.array([1 if p in (3, 150, 299) else [0, 2, 3][p % 3] for p in range(nq)], dtype=np.uint32)
    n0 = ctx.launches
    paths, pdist = dev.align(qflat, qoff, idx)
    assert ctx.launches - n0 == 5
    sel = [0, 1, 2, 3, 150, 298, 299]
    check_band_paths([paths[p] for p in sel], pdist[sel], dflat, doff, np.concatenate([qflat[2048 * p:2048 * (p + 1)] for p in sel]),
                     np.arange(len(sel) + 1, dtype=np.uint64) * 2048, idx[sel], 3)


def test_cosine_match_and_walk_ignore_the_band(ctx):
    d, doff = synth.segments(3000, 13, seed=91)
    q, qoff = synth.segments(100, 13, seed=92)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    targets = np.linspace(0.0, 1.0, 100)
    ci, cd = dev.match(q, qoff, SS_COSINE_REF, 1, targets)
    wi, wd = dev.walk(q[:int(qoff[1])], targets[:20])
    dev.set_dtw_band(1)
    ci2, cd2 = dev.match(q, qoff, SS_COSINE_REF, 1, targets)
    wi2, wd2 = dev.walk(q[:int(qoff[1])], targets[:20])
    check(ci2, cd2, ci, cd)
    check(wi2, wd2, wi, wd)


def test_band_set_between_match_dev_and_finish_leaves_that_match_unbanded(ctx, config3):
    import torch
    d, doff, q, qoff = config3
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    o_idx = torch.empty((1000, 1), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((1000, 1), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 1, o_idx.data_ptr(), o_dist.data_ptr()))
    dev.set_dtw_band(1)  # completes the pending match first, under radius 0
    ctx.sync()
    oidx, odist = R.dtw_band_topk(d, doff, q, qoff, 13, 1, 0)
    check(o_idx.cpu().numpy().view(np.uint32), o_dist.cpu().numpy(), oidx, odist)
    assert dev.dtw_band == 1
    idx, dist = dev.match(q, qoff, SS_DTW, 1)
    check(idx, dist, *R.dtw_band_topk(d, doff, q, qoff, 13, 1, 1))


def test_python_sound_dictionary_keeps_its_band_across_add_segments(ctx):
    rng = np.random.default_rng(10)
    segs = [rng.normal(size=(n, 12)) * 3 for n in rng.integers(1, 60, size=50)]
    qsegs = [rng.normal(size=(n, 12)) * 3 for n in rng.integers(1, 60, size=12)]
    snd = lambda s: api.Sound(np.zeros(1024 + 256 * max(s.shape[0] - 1, 0)), 44100.0, s, 0.0, s.mean(axis=0), None, ctx)
    sd = api.SoundDictionary(ctx, SS_DTW, dtw_band=2)
    sd.sounds = [snd(s) for s in segs[:30]]
    qsnd = [snd(s) for s in qsegs]
    qflat, qoff = flat_of(qsegs, 12)
    idx, dist = sd.match_indices(qsnd, k=2)
    dflat, doff = flat_of(segs[:30], 12)
    check(idx, dist, *R.dtw_band_topk(dflat, doff, qflat, qoff, 12, 2, 2))
    sd.sounds += [snd(s) for s in segs[30:]]
    sd._dev = None  # what add_segments does: the next call builds a new device dictionary
    idx, dist = sd.match_indices(qsnd, k=2)
    dflat, doff = flat_of(segs, 12)
    check(idx, dist, *R.dtw_band_topk(dflat, doff, qflat, qoff, 12, 2, 2))
    paths, pdist = sd.align(qsnd, idx[:, 0])
    check_band_paths(paths, pdist, dflat, doff, qflat, qoff, idx[:, 0], 2)


def test_sharded_equals_one_gpu(ctx):
    import torch
    n = min(torch.cuda.device_count(), 8)
    if n < 2:
        pytest.skip("needs 2 GPUs")
    d, doff = synth.segments(4000, 13, lmin=1, lmax=60, seed=101)
    q, qoff = synth.segments(300, 13, lmin=1, lmax=60, seed=102)
    one = api.DeviceDictionary(ctx, d, doff, 13)
    one.set_dtw_band(2)
    want = one.match(q, qoff, SS_DTW, 4)
    ctxs = [ctx] + [api.Context(i) for i in range(1, n)]
    sd = api.ShardedDictionary(ctxs, d, doff, 13)
    sd.set_dtw_band(2)
    check(*sd.match(q, qoff, SS_DTW, 4), *want)
