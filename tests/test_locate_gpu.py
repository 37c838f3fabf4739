"""ss_dict_locate: subsequence DTW (spec A12, DESIGN.md §3.1g) on the device. Every comparison is exact: indices, starts and ends
with array_equal, costs by bits, against the checker tests/cpp/dtw_subseq.cpp."""
import numpy as np
import pytest

import subseq_reference as R
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_COSINE_REF, SS_DTW

pytestmark = pytest.mark.gpu
NONE = 0xFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def check(got, want, index_base=0):
    idx, start, end, cost = got
    widx, wstart, wend, wcost = want
    widx = np.where(widx == NONE, NONE, widx.astype(np.uint64) + index_base).astype(np.uint32)
    assert np.array_equal(idx, widx), np.argwhere(idx != widx)[:5]
    assert np.array_equal(start, wstart), np.argwhere(start != wstart)[:5]
    assert np.array_equal(end, wend), np.argwhere(end != wend)[:5]
    assert np.array_equal(bits(cost), bits(wcost))


def flat_of(segs, c=13):
    off = np.zeros(len(segs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([s.shape[0] for s in segs])
    flat = np.concatenate(segs, axis=0) if int(off[-1]) else np.zeros((0, c))
    return np.ascontiguousarray(flat, dtype=np.float64), off


def launches(nq, nseg):
    b = max(1, min(nq, (1 << 24) // nseg))
    return 3 * -(-nq // b) if nq else 0


@pytest.fixture(scope="module")
def config3():
    d, doff = synth.segments(10000, 13, seed=1234)
    q, qoff = synth.segments(1000, 13, seed=5678)
    q, qoff = q[:int(qoff[200])], qoff[:201]  # 200 of its queries
    return d, doff, q, qoff, R.subseq_topk(d, doff, q, qoff, 13, 8)


@pytest.mark.parametrize("k", [1, 8])
def test_config3(ctx, config3, k):
    d, doff, q, qoff, want = config3
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    check(dev.locate(q, qoff, k), [w[:, :k] for w in want])


def test_mixed_lengths_1_to_400_and_2048_frame_queries(ctx):
    d, doff = synth.segments(150, 13, lmin=1, lmax=400, seed=61)
    q, qoff = synth.segments(30, 13, lmin=1, lmax=400, seed=62)
    rng = np.random.default_rng(63)
    long_q = [rng.normal(size=(2048, 13)) * 5, d[int(doff[7]):int(doff[7]) + 300].repeat(7, axis=0)[:2048]]
    q, qoff = flat_of([q[int(qoff[i]):int(qoff[i + 1])] for i in range(30)] + long_q)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    check(dev.locate(q, qoff, 3), R.subseq_topk(d, doff, q, qoff, 13, 3))


def test_queries_longer_than_every_segment(ctx):
    d, doff = synth.segments(500, 13, lmin=1, lmax=32, seed=71)
    q, qoff = synth.segments(40, 13, lmin=33, lmax=120, seed=72)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    got = dev.locate(q, qoff, 4)
    check(got, R.subseq_topk(d, doff, q, qoff, 13, 4))
    assert (got[0] != NONE).all()


def test_queries_cut_from_long_dictionary_sounds_are_found_at_cost_zero(ctx, config3):
    d = config3[0]
    sounds = [d[5100 * i:5100 * i + 5000 + 37 * i] for i in range(4)]  # config-3 segments concatenated, ~5 000 frames each, disjoint
    dflat, doff = flat_of(sounds)
    rng = np.random.default_rng(81)
    cuts = []
    for _ in range(24):
        s = int(rng.integers(0, 4))
        n = int(rng.integers(1, 300))
        a = int(rng.integers(0, sounds[s].shape[0] - n + 1))
        cuts.append((s, a, a + n - 1))
    q, qoff = flat_of([sounds[s][a:e + 1] for s, a, e in cuts])
    dev = api.DeviceDictionary(ctx, dflat, doff, 13)
    idx, start, end, cost = got = dev.locate(q, qoff, 2)
    assert [(int(idx[p, 0]), int(start[p, 0]), int(end[p, 0])) for p in range(24)] == cuts
    assert (cost[:, 0] == 0.0).all()
    check(got, R.subseq_topk(dflat, doff, q, qoff, 13, 2))


def test_index_base(ctx, config3):
    d, doff, q, qoff, want = config3
    dev = api.DeviceDictionary(ctx, d, doff, 13, index_base=123456)
    check(dev.locate(q[:int(qoff[50])], qoff[:51], 8), [w[:50] for w in want], index_base=123456)


def test_locate_dev_equals_host_form_and_documented_launch_count(ctx):
    """100 000 segments: batches of 167 queries, so 400 queries take three batches"""
    import torch
    d, doff = synth.segments(100000, 13, lmin=1, lmax=3, seed=91)
    q, qoff = synth.segments(400, 13, lmin=1, lmax=6, seed=92)
    qoff[57:] -= qoff[57] - qoff[56]  # query 56 is empty
    q = q[:int(qoff[-1])]
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    host = dev.locate(q, qoff, 5)
    check(host, R.subseq_topk(d, doff, q, qoff, 13, 5))
    assert (host[0][56] == NONE).all()
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    o = [torch.full((400, 5), 7, dtype=torch.int32, device="cuda") for _ in range(3)] + [torch.empty((400, 5), dtype=torch.float64, device="cuda")]
    torch.cuda.synchronize()
    n0 = ctx.launches
    ctx.check(ctx.lib.ss_dict_locate_dev(dev.h, qs.h, 5, *[t.data_ptr() for t in o]))
    assert ctx.launches - n0 == launches(400, 100000) == 9
    ctx.sync()
    got = [t.cpu().numpy() for t in o]
    check([g.view(np.uint32) for g in got[:3]] + [got[3]], host)
    # NULL start / end / cost, and nq = 0
    ctx.check(ctx.lib.ss_dict_locate_dev(dev.h, qs.h, 5, o[0].data_ptr(), None, None, None))
    ctx.sync()
    assert np.array_equal(o[0].cpu().numpy().view(np.uint32), host[0])
    empty = api.DeviceQueries(ctx, np.zeros((0, 13)), np.zeros(1, dtype=np.uint64), 13)
    n0 = ctx.launches
    ctx.check(ctx.lib.ss_dict_locate_dev(dev.h, empty.h, 5, None, None, None, None))
    assert ctx.launches == n0


def test_located_spans_are_what_match_and_align_report(ctx, config3):
    """identity 2 and 3 on the device: cost / (Lq + end - start + 1) is ss_dict_match's and ss_dict_align's distance of the
    query against a segment made of frames start..end, and the alignment's path there is the backtrack of S"""
    d, doff, q, qoff, want = config3
    idx, start, end, cost = [w[:, 0] for w in want]
    spans = [d[int(doff[idx[p]]) + int(start[p]):int(doff[idx[p]]) + int(end[p]) + 1] for p in range(200)]
    sflat, soff = flat_of(spans)
    dev = api.DeviceDictionary(ctx, sflat, soff, 13)
    lq = np.diff(qoff).astype(np.int64)
    norm = cost / (lq + end.astype(np.int64) - start.astype(np.int64) + 1)
    paths, pdist = dev.align(q, qoff, np.arange(200, dtype=np.uint32))
    assert np.array_equal(bits(pdist), bits(norm))
    for p in range(200):
        a = q[int(qoff[p]):int(qoff[p + 1])]
        want_path = R.subseq_path(a, d[int(doff[idx[p]]):int(doff[idx[p] + 1])]) - np.array([0, start[p]], dtype=np.uint32)
        assert np.array_equal(paths[p], want_path), p
    for p in range(0, 200, 25):  # ss_dict_match against a dictionary of that one span
        one = api.DeviceDictionary(ctx, spans[p], np.array([0, spans[p].shape[0]], dtype=np.uint64), 13)
        mi, md = one.match(q[int(qoff[p]):int(qoff[p + 1])], np.array([0, lq[p]], dtype=np.uint64), SS_DTW, 1)
        assert mi[0, 0] == 0 and bits(md[0, 0]) == bits(norm[p]), p


def test_band_and_pending_match_and_last_readers_are_unaffected(ctx, config3):
    import torch
    d, doff, q, qoff, want = config3
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    midx, mdist = dev.match(q, qoff, SS_DTW, 4)
    readers = (dev.last_work, dev.last_scan_kind, dev.last_uncertified, dev.last_tc_fallback, dev.last_exhaustive)
    cidx, cdist = dev.match(q, qoff, SS_COSINE_REF, 1)
    creaders = (dev.last_work, dev.last_scan_kind)
    check(dev.locate(q, qoff, 8), want)
    assert (dev.last_work, dev.last_scan_kind) == creaders
    dev.set_dtw_band(1)  # the band does not apply to locate
    check(dev.locate(q, qoff, 8), want)
    dev.set_dtw_band(0)
    # an asynchronous SS_DTW match, then locate: the match completes first, with its own results
    o_idx = torch.empty((200, 4), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((200, 4), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 4, o_idx.data_ptr(), o_dist.data_ptr()))
    check(dev.locate(q, qoff, 8), want)
    ctx.sync()
    assert np.array_equal(o_idx.cpu().numpy().view(np.uint32), midx) and np.array_equal(bits(o_dist.cpu().numpy()), bits(mdist))
    assert (dev.last_work, dev.last_scan_kind, dev.last_uncertified, dev.last_tc_fallback, dev.last_exhaustive) == readers
    # later matches are unchanged
    i2, d2 = dev.match(q, qoff, SS_DTW, 4)
    assert np.array_equal(i2, midx) and np.array_equal(bits(d2), bits(mdist))
    c2, cd2 = dev.match(q, qoff, SS_COSINE_REF, 1)
    assert np.array_equal(c2, cidx) and np.array_equal(bits(cd2), bits(cdist))


def test_errors(ctx):
    from soundsym_b200._lib import SS_ERR_EMPTY_DICT, SS_ERR_INVALID, SoundsymError
    d, doff = synth.segments(20, 13, seed=3)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    for k in (0, 9):
        with pytest.raises(SoundsymError) as e:
            dev.locate(d[:10], np.array([0, 10], dtype=np.uint64), k)
        assert e.value.code == SS_ERR_INVALID and "k must be" in e.value.message
    assert ctx.lib.ss_dict_locate(dev.h, None, None, 1, 1, None, None, None, None) == SS_ERR_INVALID
    empty = api.DeviceDictionary(ctx, np.zeros((0, 13)), np.zeros(1, dtype=np.uint64), 13)
    with pytest.raises(SoundsymError) as e:
        empty.locate(d[:10], np.array([0, 10], dtype=np.uint64))
    assert e.value.code == SS_ERR_EMPTY_DICT
    idx, start, end, cost = dev.locate(np.zeros((0, 13)), np.zeros(1, dtype=np.uint64), 2)
    assert idx.shape == (0, 2)


def test_python_sound_dictionary_locate(ctx):
    rng = np.random.default_rng(10)
    segs = [rng.normal(size=(n, 12)) * 3 for n in rng.integers(1, 300, size=20)]
    qsegs = [segs[3][10:50], segs[11][:1], rng.normal(size=(40, 12)) * 3, segs[0][:0]]
    snd = lambda s: api.Sound(np.zeros(1024 + 256 * max(s.shape[0] - 1, 0)), 44100.0, s, 0.0, s.mean(axis=0) if len(s) else None, None, ctx)
    sd = api.SoundDictionary(ctx, SS_COSINE_REF, dtw_band=2)
    sd.sounds = [snd(s) for s in segs]
    got = sd.locate([snd(s) for s in qsegs], k=2)
    dflat, doff = flat_of(segs, 12)
    qflat, qoff = flat_of(qsegs, 12)
    check(got, R.subseq_topk(dflat, doff, qflat, qoff, 12, 2))
    assert (got[0][0, 0], got[1][0, 0], got[2][0, 0], got[3][0, 0]) == (3, 10, 49, 0.0)
    assert (got[0][3] == NONE).all()


def test_cpp_mirror_locate(tmp_path, section71):
    """the C++ mirror (include/soundsym.hpp SoundDictionary::locate) on the examples/matcher.rs flow: a directory of long cuts of
    the recording as the dictionary, query files cut from them at whole hops; equal to the Python mirror, which shares nothing
    with it above the C ABI, and every query found where it was cut"""
    import os
    from test_cpp_host_gpu import run, write_wav
    pcm = section71["pcm"]
    ddir, qdir = tmp_path / "dict", tmp_path / "queries"
    ddir.mkdir(), qdir.mkdir()
    bounds = [0, 150000, 320000, len(pcm)]
    for i in range(3):
        write_wav(str(ddir / ("d%d.wav" % i)), pcm[bounds[i]:bounds[i + 1]], 16)
    rng = np.random.default_rng(4)
    cut = []
    for i in range(5):
        s = int(rng.integers(0, 3))
        frame = int(rng.integers(0, 200))
        n = int(rng.integers(3000, 20000))
        write_wav(str(qdir / ("q%d.wav" % i)), pcm[bounds[s] + 256 * frame:bounds[s] + 256 * frame + n], 16)
        cut.append((s, frame))
    rc, r = run(["--matcher", str(ddir), str(qdir), "--locate"])
    assert rc == 0, r
    ctx = api.Context(0)
    d = api.SoundDictionary.from_path(str(ddir), ctx)
    q = api.SoundDictionary.from_path(str(qdir), ctx)
    idx, start, end, cost = d.locate(q.sounds, k=1)
    want = [[s.name, d.sounds[int(idx[p, 0])].name, int(start[p, 0]), int(end[p, 0]), float(cost[p, 0])] for p, s in enumerate(q.sounds)]
    assert r["located"] == want
    for p, (s, frame) in enumerate(cut):
        assert (int(idx[p, 0]), int(start[p, 0]), int(end[p, 0]), cost[p, 0]) == (s, frame, frame + q.sounds[p].num_frames() - 1, 0.0)
    assert sorted(os.listdir(qdir)) == ["q%d.wav" % i for i in range(5)]
