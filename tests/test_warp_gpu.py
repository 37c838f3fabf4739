"""ss_resynth_warped (spec A11, DESIGN.md §3.5) on the device: resynthesis along the DTW warping path. Every comparison is exact
(array_equal on the f64 samples) against the numpy twin tests/warp_reference.py, which tests/test_warp_cpu.py checks against a
per-sample restatement of the spec."""
import ctypes as C

import numpy as np
import pytest

import warp_reference as W
from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_COSINE_REF, SS_DTW, SS_ERR_EMPTY_DICT, SS_ERR_INVALID, SoundsymError

from test_cpp_host_gpu import run, write_model, write_wav

pytestmark = pytest.mark.gpu
H = W.H


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def cuts(ctx, sound, splits):
    """reconstruction.rs:77-81: segment i takes splits[i] samples and splits[i] / HOP MFCC rows of `sound`"""
    segs, spos, fpos = [], 0, 0
    for sp in (int(x) for x in splits):
        m = sound.mfcc_arrays()[fpos:fpos + sp // H]
        segs.append(api.Sound(sound.samples()[spos:spos + sp], sound.sample_rate(), m, None, m.mean(axis=0) if len(m) else np.full(12, np.nan),
                              None, ctx))
        spos += sp
        fpos += sp // H
    return segs


def dict_arrays(dictionary):
    doff = np.zeros(len(dictionary.sounds) + 1, dtype=np.uint64)
    doff[1:] = np.cumsum([len(s.samples()) for s in dictionary.sounds])
    return np.concatenate([s.samples() for s in dictionary.sounds]), doff


@pytest.fixture(scope="module")
def config1(ctx, section71, sample_excerpt):
    """the config-1 fixtures: Section_7_1 cut at its depth-3 / threshold-4 splits as the dictionary source, the sample.wav
    excerpt cut at its own splits as the target"""
    src = api.Sound(O.decode_pcm(section71["pcm"].astype(np.int32), 16), 44100.0, section71["mfcc"], None, section71["mfcc"].mean(axis=0), None, ctx)
    tgt = api.Sound(O.decode_pcm(sample_excerpt["pcm"], 24), 44100.0, sample_excerpt["mfcc"], None, sample_excerpt["mfcc"].mean(axis=0), None, ctx)
    return src, section71["splits_d3t4"], cuts(ctx, tgt, sample_excerpt["splits_d3t4"])


def check_flow(ctx, dictionary, segs):
    """clone_from_dictionary(warp=True) against the twin applied to that call's own indices and paths"""
    seq = api.SoundSequence(segs, ctx)
    out = seq.clone_from_dictionary(dictionary, warp=True)
    idx = dictionary.match_indices(segs)[0][:, 0]
    paths, _ = dictionary.align(segs, idx)
    cells, poff = W.flatten(paths)
    ds, doff = dict_arrays(dictionary)
    tl = np.array([len(s.samples()) for s in segs], dtype=np.uint64)
    want = W.resynth_warped(ds, doff, idx, cells, poff, tl)
    got = out.to_sound().samples()
    assert np.array_equal(got, want)
    assert np.array_equal(np.concatenate([s.samples() for s in out.sounds()]), want)
    return out, idx, paths, want


@pytest.mark.parametrize("mode,band", [(SS_DTW, 0), (SS_DTW, 3), (SS_COSINE_REF, 0)])
def test_config1_flow_equals_the_twin(ctx, config1, mode, band):
    src, splits, segs = config1
    d = api.SoundDictionary.from_segments(src, splits, ctx, mode)
    d.dtw_band = band
    out, idx, paths, want = check_flow(ctx, d, segs)
    plain = api.SoundSequence(segs, ctx).clone_from_dictionary(d).to_sound().samples()
    assert not np.array_equal(plain, want)  # the paths move samples on this data
    straight = [t for t, p in enumerate(paths) if len(p) and np.all(p[:, 0] == p[:, 1])]
    tl = np.cumsum([0] + [len(s.samples()) for s in segs])
    for t in straight:  # P1 per segment: a diagonal path gives the plain resynthesis
        assert np.array_equal(want[tl[t]:tl[t + 1]], plain[tl[t]:tl[t + 1]])
    for t in list(range(0, len(segs), max(len(segs) // 8, 1))):  # the batched analysis of the output segments
        mfcc, mp, mean = ctx.analyze(out.sounds()[t].samples())
        s = out.sounds()[t]
        assert np.array_equal(s.mfcc_arrays(), mfcc) and s.max_power() == mp
        assert np.allclose(s.mean_mfccs(), mean, rtol=1e-12, atol=1e-12, equal_nan=True)  # the batch sums rows in another order


def test_own_segments_give_back_the_target(ctx):
    """P1 end to end: every segment matches itself along the diagonal, so the output is the target, as with warp=False"""
    audio = synth.audio(12.0, seed=5)
    snd = api.Sound.from_samples(audio, 44100.0, ctx=ctx)
    rng = np.random.default_rng(6)
    splits = []
    while sum(splits) < len(audio) - 6000:
        splits.append(int(rng.integers(300, 6000)))
    d = api.SoundDictionary.from_segments(snd, splits, ctx, SS_DTW)
    idx = d.match_indices(d.sounds)[0][:, 0]
    assert np.array_equal(idx, np.arange(len(splits)))
    warped = api.SoundSequence(d.sounds, ctx).clone_from_dictionary(d, warp=True).to_sound().samples()
    plain = api.SoundSequence(d.sounds, ctx).clone_from_dictionary(d).to_sound().samples()
    assert np.array_equal(warped, audio[:sum(splits)]) and np.array_equal(warped, plain)


def random_inputs(rng, nseg=240, nd=60):
    dlens = rng.integers(0, 4000, size=nd)
    dlens[:2] = (0, 7)
    doff = np.zeros(nd + 1, dtype=np.uint64)
    doff[1:] = np.cumsum(dlens)
    ds = rng.normal(size=int(doff[-1]))
    tl = rng.integers(0, 3001, size=nseg)
    tl[tl % H == 0] += 1  # never a whole number of hops, except the empty segments below
    tl[:3] = (0, 1, 255)
    mi = rng.integers(0, nd, size=nseg).astype(np.uint32)
    paths = [W.random_path(rng, int(tl[t]) // H + int(rng.integers(0, 3)), int(dlens[mi[t]]) // H + int(rng.integers(0, 3)), t % 4 != 3,
                           float(rng.uniform(0.1, 0.9))) for t in range(nseg)]
    return ds, doff, mi, paths, tl.astype(np.uint64)


def test_random_valid_paths_equal_the_twin(ctx):
    rng = np.random.default_rng(21)
    ds, doff, mi, paths, tl = random_inputs(rng)
    cells, poff = W.flatten(paths)
    dl = np.diff(doff)[mi]
    assert np.any(dl < tl) and np.any(dl > tl)  # dictionary sounds both shorter and longer than their targets
    n0 = ctx.launches
    got = ctx.resynth_warped(ds, doff, mi, cells, poff, tl)
    assert ctx.launches - n0 == 1
    assert np.array_equal(got, W.resynth_warped(ds, doff, mi, cells, poff, tl))


def test_errors_and_launch_count(ctx):
    rng = np.random.default_rng(22)
    ds, doff, mi, paths, tl = random_inputs(rng, nseg=20, nd=10)
    cells, poff = W.flatten(paths)
    L = ctx.lib

    def call(ds=ds, doff=doff, mi=mi, cells=cells, poff=poff, tl=tl, nd=10, nseg=20, out=True):
        o = np.empty(max(int(np.sum(tl)) if tl is not None else 0, 1))
        p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        return L.ss_resynth_warped(ctx.h, p(ds), p(doff), nd, p(mi), p(cells), p(poff), p(tl), nseg, p(o) if out else None)

    n0 = ctx.launches
    assert call(nseg=0) == 0 and ctx.launches == n0  # nseg == 0: nothing to do, nothing launched
    assert call(tl=np.zeros(20, dtype=np.uint64)) == 0 and ctx.launches == n0  # no output samples: no launch
    for kw in (dict(doff=None), dict(mi=None), dict(poff=None), dict(tl=None), dict(out=False)):
        assert call(**kw) == SS_ERR_INVALID, kw
    assert call(cells=None) == SS_ERR_INVALID and "paths is NULL" in L.ss_last_error(ctx.h).decode()
    assert call(nd=0) == SS_ERR_EMPTY_DICT
    bad = mi.copy()
    bad[5] = 10
    assert call(mi=bad) == SS_ERR_INVALID and "match_idx[5]" in L.ss_last_error(ctx.h).decode()
    k = next(t for t in range(20) if poff[t + 1] - poff[t] >= 3)
    bad = poff.copy()
    bad[5] = poff[6] + 1
    assert call(poff=bad) == SS_ERR_INVALID and "not monotone at 5" in L.ss_last_error(ctx.h).decode()
    assert call(poff=(poff + 1).astype(np.uint64)) == SS_ERR_INVALID  # offsets must start at 0
    e = int(poff[k])
    for cell, what in (((0, 1), "start at (0, 0)"), ((1, 0), "start at (0, 0)")):
        c = cells.copy()
        c[e] = cell
        assert call(cells=c) == SS_ERR_INVALID and what in L.ss_last_error(ctx.h).decode()
    for step in ((2, 0), (0, 2), (0, 0), (2, 2)):  # only (1, 0), (0, 1), (1, 1) are steps
        c = cells.copy()
        c[e + 2] = c[e + 1] + np.array(step, dtype=np.uint32)
        assert call(cells=c) == SS_ERR_INVALID, step
        assert "is not (1, 0), (0, 1) or (1, 1)" in L.ss_last_error(ctx.h).decode()
    assert ctx.launches == n0
    assert call() == 0 and ctx.launches == n0 + 1
    with pytest.raises(SoundsymError):
        ctx.resynth_warped(ds, doff, mi, cells, poff[:-1], tl)


def test_cpp_mirror_reconstruction_dtw_warp(ctx, tmp_path, section71, sample_excerpt):
    """examples/reconstruction.cpp --dtw --warp writes the samples the Python mirror computes for the same flow"""
    src, tgt, mdl, out = (str(tmp_path / n) for n in ("source.wav", "target.wav", "model.bin", "out.wav"))
    write_wav(src, section71["pcm"], 16)
    write_wav(tgt, sample_excerpt["pcm"], 24)
    write_model(mdl, section71)
    rc, r = run(["-s", src, "-t", tgt, "-o", out, "-m", mdl, "--dtw", "--warp"])
    assert rc == 0, r
    model = (section71["gmm_means"], section71["gmm_covs"], section71["gmm_weights"])
    s = api.Sound.from_samples(O.decode_pcm(section71["pcm"].astype(np.int32), 16), 44100.0, ctx=ctx)
    part = api.Partitioner(s, ctx).set_threshold(4).set_depth(3)
    part.train(model)
    d = api.SoundDictionary.from_segments(s, part.partition(), ctx, SS_DTW)
    t = api.Sound.from_samples(O.decode_pcm(sample_excerpt["pcm"], 24), 44100.0, ctx=ctx)
    part.sound = t
    segs = cuts(ctx, t, part.partition())
    got, idx, _, _ = check_flow(ctx, d, segs)
    samples = got.to_sound().samples()
    assert r["idx"] == [int(i) for i in idx] and r["out_samples"] == len(samples)
    assert r["out_sum"] == float(np.cumsum(samples)[-1])  # the C++ sum runs in sample order
    mine = str(tmp_path / "python.wav")
    api._write_wav_i32(mine, samples, 44100.0)
    assert open(out, "rb").read() == open(mine, "rb").read()


def test_config5_scale_one_hour(ctx):
    """config 5: an hour of synthetic audio, source = first half, target = second half, cosine matcher, warped resynthesis"""
    audio = synth.audio(3600.0, seed=42)
    half = (len(audio) // 2 // H) * H
    src = api.Sound.from_samples(audio[:half], 44100.0, ctx=ctx)
    part = api.Partitioner(src, ctx).set_threshold(4).set_depth(3)
    part.train(seed=3)
    d = api.SoundDictionary.from_segments(src, part.partition(), ctx, SS_COSINE_REF)
    tgt = api.Sound.from_samples(audio[half:], 44100.0, ctx=ctx)
    part.sound = tgt
    segs = cuts(ctx, tgt, part.partition())
    assert len(segs) > 5000
    seq = api.SoundSequence(segs, ctx).clone_from_dictionary(d, warp=True)
    got = seq.to_sound().samples()
    idx = d.match_indices(segs)[0][:, 0]
    paths, _ = d.align(segs, idx)
    ds, doff = dict_arrays(d)
    tl = np.array([len(s.samples()) for s in segs], dtype=np.uint64)
    ooff = np.concatenate([[0], np.cumsum(tl)]).astype(np.int64)
    step = 500  # the twin in slices of segments, to bound its memory
    for a in range(0, len(segs), step):
        b = min(a + step, len(segs))
        cells, poff = W.flatten(paths[a:b])
        assert np.array_equal(got[ooff[a]:ooff[b]], W.resynth_warped(ds, doff, idx[a:b], cells, poff, tl[a:b])), a
