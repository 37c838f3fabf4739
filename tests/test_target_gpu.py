"""SS_DTW_TARGET (spec A13, DESIGN.md §3.1h) on the device: the k best (|D - t|, index) per query. Every comparison is exact:
indices with array_equal, distances by bits, against the numpy twin (tests/target_reference.py) built on the oracle's dtw_matrix
and, under a band, on the band checker (tests/cpp/dtw_band.cpp)."""
import numpy as np
import pytest

import band_reference as R
import target_reference as T
from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_DTW, SS_DTW_TARGET, SoundsymError

from test_cpp_host_gpu import run, write_model, write_wav
from test_sequence_gpu import cut_offsets

pytestmark = pytest.mark.gpu
NONE = 0xFFFFFFFF


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def check(got, want, index_base=0):
    (idx, dist), (widx, wdist) = got, want
    widx = np.where(widx == NONE, NONE, widx.astype(np.uint64) + index_base).astype(np.uint32)
    assert np.array_equal(idx, widx), np.argwhere(idx != widx)[:5]
    assert np.array_equal(bits(dist), bits(wdist)), np.argwhere(bits(dist) != bits(wdist))[:5]


def flat_of(segs, c=13):
    off = np.zeros(len(segs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([s.shape[0] for s in segs])
    flat = np.concatenate(segs, axis=0) if int(off[-1]) else np.zeros((0, c))
    return np.ascontiguousarray(flat, dtype=np.float64), off


def split(flat, off):
    return [flat[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)]


def band_matrix(d, doff, q, qoff, r):
    ds, qs = split(d, doff), split(q, qoff)
    return np.array([[R.dtw_band(a, b, r) for b in ds] for a in qs])


@pytest.fixture(scope="module")
def config3():
    d, doff = synth.segments(10000, 13, seed=1234)
    q, qoff = synth.segments(1000, 13, seed=5678)
    return d, doff, q, qoff, O.dtw_matrix(d, doff, q, qoff, 13)


def quantile_targets(D, p):
    lo, hi = np.nanmin(D, axis=1), np.nanmax(D, axis=1)
    if p == "below":
        return lo - 1.0
    if p == "above":
        return hi + 1.0
    return np.nanquantile(D, p, axis=1)


@pytest.mark.parametrize("p", ["below", 0.0, 0.01, 0.5, 0.9, 1.0, "above"])
def test_config3_targets_at_quantiles(ctx, config3, p):
    d, doff, q, qoff, D = config3
    t = quantile_targets(D, p)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    for k in (1, 8):
        check(dev.match(q, qoff, SS_DTW_TARGET, k, t), T.target_topk(D, t, k))
        assert dev.last_uncertified == 0 and dev.last_scan_kind == 3


def test_null_and_zero_targets_equal_ss_dtw(ctx, config3):
    d, doff, q, qoff, _ = config3
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    for k in (1, 8):
        want = dev.match(q, qoff, SS_DTW, k)
        for t in (None, np.zeros(len(qoff) - 1)):
            got = dev.match(q, qoff, SS_DTW_TARGET, k, t)
            assert np.array_equal(got[0], want[0]) and np.array_equal(bits(got[1]), bits(want[1]))


def test_ss_dtw_still_ignores_targets(ctx, config3):
    d, doff, q, qoff, D = config3
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    a = dev.match(q, qoff, SS_DTW, 4)
    b = dev.match(q, qoff, SS_DTW, 4, quantile_targets(D, 0.5))
    assert np.array_equal(a[0], b[0]) and np.array_equal(bits(a[1]), bits(b[1]))


def mixed():
    d, doff = synth.segments(300, 13, lmin=1, lmax=400, seed=61)
    q, qoff = synth.segments(40, 13, lmin=1, lmax=400, seed=62)
    rng = np.random.default_rng(63)
    long_d = rng.normal(size=(2048, 13))
    ds = split(d, doff) + [long_d, long_d[::-1] + 0.3]
    qs = split(q, qoff) + [long_d + 0.05 * rng.normal(size=(2048, 13))]
    d, doff = flat_of(ds)
    q, qoff = flat_of(qs)
    return d, doff, q, qoff


@pytest.mark.parametrize("r", [0, 1, 3])
def test_mixed_lengths_and_2048_frames_banded(ctx, r):
    d, doff, q, qoff = mixed()
    D = O.dtw_matrix(d, doff, q, qoff, 13) if r == 0 else band_matrix(d, doff, q, qoff, r)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    dev.set_dtw_band(r)
    for p in (0.0, 0.3, 0.7, "above"):
        t = quantile_targets(D, p)
        for k in (1, 3):
            check(dev.match(q, qoff, SS_DTW_TARGET, k, t), T.target_topk(D, t, k))
            assert dev.last_uncertified == 0


def test_near_duplicates_around_the_target_go_exhaustive(ctx):
    rng = np.random.default_rng(71)
    base = rng.normal(size=(40, 13))
    dups = [base + 1e-9 * rng.normal(size=base.shape) for _ in range(64)]
    others, ooff = synth.segments(200, 13, lmin=20, lmax=60, seed=72)
    d, doff = flat_of(split(others, ooff)[:100] + dups + split(others, ooff)[100:])
    q, qoff = flat_of([base[::-1].copy(), rng.normal(size=(45, 13))])
    D = O.dtw_matrix(d, doff, q, qoff, 13)
    t = D[:, 150]  # a duplicate's distance: dozens of pairs within the scan's error of the target
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    for k in (1, 8):
        check(dev.match(q, qoff, SS_DTW_TARGET, k, t), T.target_topk(D, t, k))
        assert dev.last_exhaustive > 0 and dev.last_uncertified == 0


def test_four_shards_merged_equal_one_dictionary(ctx):
    import torch
    d, doff = synth.segments(900, 13, lmin=1, lmax=60, seed=81)
    q, qoff = synth.segments(40, 13, lmin=1, lmax=60, seed=82)
    D = O.dtw_matrix(d, doff, q, qoff, 13)
    t = quantile_targets(D, 0.4)
    k = 4
    whole = api.DeviceDictionary(ctx, d, doff, 13).match(q, qoff, SS_DTW_TARGET, k, t)
    check(whole, T.target_topk(D, t, k))
    cuts = [0, 200, 450, 700, 900]
    li, ld = [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        i, dd = api.DeviceDictionary(ctx, d, doff[a:b + 1], 13, index_base=a).match(q, qoff, SS_DTW_TARGET, k, t)
        li.append(i)
        ld.append(dd)
    gi = torch.from_numpy(np.stack(li).astype(np.int64)).to(torch.int32).cuda()
    gd = torch.from_numpy(np.stack(ld)).cuda()
    oi = torch.empty((40, k), dtype=torch.int32, device="cuda")
    od = torch.empty((40, k), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_topk_merge_dev(ctx.h, gi.data_ptr(), gd.data_ptr(), 4, 40, k, oi.data_ptr(), od.data_ptr()))
    ctx.sync()
    assert np.array_equal(oi.cpu().numpy().astype(np.uint32), whole[0]) and np.array_equal(bits(od.cpu().numpy()), bits(whole[1]))
    if torch.cuda.device_count() > 1:
        n = min(torch.cuda.device_count(), 4)
        ctxs = [ctx] + [api.Context(i) for i in range(1, n)]
        sd = api.ShardedDictionary(ctxs, d, doff, 13)
        got = sd.match(q, qoff, SS_DTW_TARGET, k, t)
        assert np.array_equal(got[0], whole[0]) and np.array_equal(bits(got[1]), bits(whole[1]))


def test_dev_form_equals_host_form(ctx):
    import torch
    d, doff = synth.segments(2000, 13, lmin=1, lmax=80, seed=91)
    q, qoff = synth.segments(100, 13, lmin=1, lmax=80, seed=92)
    D = O.dtw_matrix(d, doff, q, qoff, 13)
    t = quantile_targets(D, 0.6)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    host = dev.match(q, qoff, SS_DTW_TARGET, 3, t)
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    td = torch.from_numpy(t).cuda()
    o_idx = torch.empty((100, 3), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((100, 3), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, SS_DTW_TARGET, td.data_ptr(), 3, o_idx.data_ptr(), o_dist.data_ptr()))
    ctx.check(ctx.lib.ss_dict_match_finish(dev.h))
    ctx.sync()
    assert np.array_equal(o_idx.cpu().numpy().astype(np.uint32), host[0]) and np.array_equal(bits(o_dist.cpu().numpy()), bits(host[1]))
    check(host, T.target_topk(D, t, 3))


def test_errors(ctx):
    d, doff = synth.segments(50, 13, seed=101)
    q, qoff = synth.segments(3, 13, seed=102)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    for bad in (np.nan, np.inf, -np.inf):
        with pytest.raises(SoundsymError) as e:
            dev.match(q, qoff, SS_DTW_TARGET, 1, [0.5, bad, 0.5])
        assert e.value.code == -1
    for k in (0, 9):
        with pytest.raises(SoundsymError) as e:
            dev.match(q, qoff, SS_DTW_TARGET, k, [0.5, 0.5, 0.5])
        assert e.value.code == -1
    empty = api.DeviceDictionary(ctx, np.zeros((0, 13)), np.zeros(1, dtype=np.uint64), 13)
    with pytest.raises(SoundsymError) as e:
        empty.match(q, qoff, SS_DTW_TARGET, 1, [0.5, 0.5, 0.5])
    assert e.value.code == -5
    # the dictionary still works after the refusals
    D = O.dtw_matrix(d, doff, q, qoff, 13)
    check(dev.match(q, qoff, SS_DTW_TARGET, 2, [0.5, 1.0, 2.0]), T.target_topk(D, [0.5, 1.0, 2.0], 2))


def sequence_fixture(ctx, section71, sample_excerpt):
    s16 = O.decode_pcm(section71["pcm"].astype(np.int32), 16)
    snd = api.Sound(s16, 44100.0, section71["mfcc"], None, section71["mfcc"].mean(axis=0), None, ctx)
    d = api.SoundDictionary.from_segments(snd, section71["splits_d3t4"], ctx, SS_DTW_TARGET)
    tgt = O.decode_pcm(sample_excerpt["pcm"], 24)
    tsnd = api.Sound(tgt, 44100.0, sample_excerpt["mfcc"], None, sample_excerpt["mfcc"].mean(axis=0), None, ctx)
    qd = api.SoundDictionary.from_segments(tsnd, sample_excerpt["splits_d3t4"], ctx, SS_DTW_TARGET)
    doff, qoff = cut_offsets(section71["splits_d3t4"]), cut_offsets(sample_excerpt["splits_d3t4"])
    dm, qm = section71["mfcc"][: int(doff[-1])], sample_excerpt["mfcc"][: int(qoff[-1])]
    return d, qd, dm, doff, qm, qoff


def chain_want(dm, doff, first, steps):
    cur, want = first, []
    for step in steps:
        row = O.dtw_matrix(dm, doff, cur, np.array([0, cur.shape[0]], dtype=np.uint64), 12)
        i, _ = T.target_topk(row, [step], 1)
        want.append(int(i[0, 0]))
        cur = dm[int(doff[i[0, 0]]):int(doff[i[0, 0] + 1])]
    return want


def test_python_mirror_morph_to_at_distance_from_distances(ctx, section71, sample_excerpt):
    d, qd, dm, doff, qm, qoff = sequence_fixture(ctx, section71, sample_excerpt)
    D = O.dtw_matrix(dm, doff, qm, qoff, 12)
    near = np.nanmin(D, axis=1)
    n = len(qoff) - 1
    distances = np.linspace(near.min(), 2.0 * near.max(), n)
    seq = api.SoundSequence(qd.sounds, ctx)
    oidx, _ = T.target_topk(D, distances, 1)
    assert [d.sounds.index(s) for s in seq.morph_to(distances, d).sounds()] == [int(i) for i in oidx[:, 0]]
    for j in (0, n // 2, n - 1):
        assert d.at_distance(float(distances[j]), qd.sounds[j]) is d.sounds[int(oidx[j, 0])]
    zi, _ = O.dtw_topk(dm, doff, qm, qoff, 12, 1)
    assert d.match_sound(qd.sounds[3]) is d.sounds[int(zi[3, 0])]  # match_sound is at_distance(0.0) in this mode
    steps = list(np.linspace(near.min(), near.max(), 5))
    chain = api.SoundSequence.from_distances(steps, qd.sounds[0], d)
    want = chain_want(dm, doff, qm[int(qoff[0]):int(qoff[1])], steps)
    assert [d.sounds.index(s) for s in chain.sounds()[1:]] == want


def test_cpp_mirror_dtw_target_morph(tmp_path, section71, sample_excerpt):
    src, tgt, mdl = (str(tmp_path / n) for n in ("source.wav", "target.wav", "model.bin"))
    write_wav(src, section71["pcm"], 16)
    write_wav(tgt, sample_excerpt["pcm"], 24)
    write_model(mdl, section71)
    rc, r = run(["-s", src, "-t", tgt, "-m", mdl, "--dtw-target", "--morph", "--chain", "6"])
    assert rc == 0
    doff, qoff = cut_offsets(section71["splits_d3t4"]), cut_offsets(sample_excerpt["splits_d3t4"])
    dm, qm = section71["mfcc"][: int(doff[-1])], sample_excerpt["mfcc"][: int(qoff[-1])]
    D = O.dtw_matrix(dm, doff, qm, qoff, 12)
    near = np.nanmin(D, axis=1)
    n = len(qoff) - 1
    want_t = [near.min() + (2.0 * near.max() - near.min()) * i / max(n - 1, 1) for i in range(n)]
    assert np.allclose(r["targets"], want_t, rtol=1e-12, atol=0)  # (the example analyses the wav files itself)
    oidx, _ = T.target_topk(D, np.array(r["targets"]), 1)
    assert r["morph"] == [int(i) for i in oidx[:, 0]]
    assert r["chain"] == chain_want(dm, doff, qm[int(qoff[0]):int(qoff[1])], r["steps"])
