"""ss_dict_align: the DTW warping path (spec: tests/cpp/dtw_path.cpp, DESIGN.md §3.1e) on the device. Every comparison is exact: paths
with array_equal against the C++ checker tests/cpp/dtw_path.cpp, distances bit for bit against ss_dict_match's SS_DTW distance and the oracle's orc_dtw."""
import os
import subprocess

import numpy as np
import pytest

import align_reference as R
from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_COSINE_REF, SS_DTW, SS_ERR_INVALID

pytestmark = pytest.mark.gpu
NONE = 0xFFFFFFFF
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def check_against_oracle(paths, dist, dflat, doff, qflat, qoff, idx, base=0):
    for p in range(len(paths)):
        q = seg(qflat, qoff, p)
        if int(idx[p]) == NONE:
            assert paths[p].shape == (0, 2) and bits(dist[p]) == bits(np.inf), p
            continue
        d = seg(dflat, doff, int(idx[p]) - base)
        want = R.dtw_path(q, d)
        assert np.array_equal(paths[p], want), (p, q.shape[0], d.shape[0])
        e = O.dtw(q, d) if q.shape[0] and d.shape[0] else np.inf
        assert bits(dist[p]) == bits(e if np.isfinite(e) else np.inf), (p, dist[p], e)


def test_config3_every_query_against_its_match_and_a_fixed_segment(ctx):
    d, doff = synth.segments(10000, 13, seed=1234)
    q, qoff = synth.segments(1000, 13, seed=5678)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    idx, mdist = dev.match(q, qoff, SS_DTW, 1)
    idx = idx[:, 0]
    paths, dist = dev.align(q, qoff, idx)
    assert np.array_equal(bits(dist), bits(mdist[:, 0]))
    check_against_oracle(paths, dist, d, doff, q, qoff, idx)
    other = np.full(1000, 7, dtype=np.uint32)
    paths, dist = dev.align(q, qoff, other)
    check_against_oracle(paths, dist, d, doff, q, qoff, other)


def long_case(rng, c=13):
    lens = [1, 2, 31, 32, 33, 63, 64, 65, 96, 100, 128, 129, 200, 257, 400] + [int(x) for x in rng.integers(1, 401, size=25)]
    segs = [rng.normal(size=(n, c)) * 5 for n in lens]
    return segs, lens


def test_long_pairs_straddling_strip_and_row_block_edges(ctx):
    rng = np.random.default_rng(3)
    dsegs, dl = long_case(rng)
    qsegs, ql = long_case(rng)
    dflat, doff = flat_of(dsegs, 13)
    # every query against a shorter, a longer and an equal-class segment: both sides cross 32 / 33 / 64 / 65
    pairs = [(qi, di) for qi in range(len(qsegs)) for di in rng.choice(len(dsegs), size=3, replace=False)]
    pairs += [(qi, qi) for qi in range(len(qsegs))]
    qs = [qsegs[a] for a, _ in pairs]
    idx = np.array([b for _, b in pairs], dtype=np.uint32)
    qflat, qoff = flat_of(qs, 13)
    dev = api.DeviceDictionary(ctx, dflat, doff, 13)
    paths, dist = dev.align(qflat, qoff, idx)
    check_against_oracle(paths, dist, dflat, doff, qflat, qoff, idx)
    assert any(int(qoff[p + 1] - qoff[p]) > int(doff[i + 1] - doff[i]) for p, i in enumerate(idx))
    assert any(int(qoff[p + 1] - qoff[p]) < int(doff[i + 1] - doff[i]) for p, i in enumerate(idx))


def test_2048_by_2048(ctx):
    rng = np.random.default_rng(4)
    a, b = rng.normal(size=(2048, 13)), rng.normal(size=(2048, 13))
    dflat, doff = flat_of([rng.normal(size=(5, 13)), b], 13)
    dev = api.DeviceDictionary(ctx, dflat, doff, 13)
    qflat, qoff = flat_of([a, b[:700]], 13)
    paths, dist = dev.align(qflat, qoff, np.array([1, 1], dtype=np.uint32))
    check_against_oracle(paths, dist, dflat, doff, qflat, qoff, [1, 1])


def test_direction_storage_spanning_two_waves(ctx):
    """300 queries of 2 048 frames against a dictionary whose longest segment is 2 048 frames: the host-known bound is 1 MB of
    directions per pair, so the 256 MB budget takes two waves (launches: align + 2 waves + scan + compact)."""
    rng = np.random.default_rng(5)
    dsegs = [rng.normal(size=(n, 13)) for n in (40, 2048, 33, 17)]
    dflat, doff = flat_of(dsegs, 13)
    dev = api.DeviceDictionary(ctx, dflat, doff, 13)
    nq = 300
    qflat = rng.normal(size=(nq * 2048, 13))
    qoff = np.arange(nq + 1, dtype=np.uint64) * 2048
    idx = np.array([1 if p in (3, 299) else [0, 2, 3][p % 3] for p in range(nq)], dtype=np.uint32)
    n0 = ctx.launches
    paths, dist = dev.align(qflat, qoff, idx)
    assert ctx.launches - n0 == 5
    check_against_oracle(paths, dist, dflat, doff, qflat, qoff, idx)


def test_ties_decide_the_path(ctx):
    rng = np.random.default_rng(6)
    base = rng.integers(0, 2, size=(6, 13)).astype(np.float64)
    dsegs = [np.repeat(base[:3], 4, axis=0), np.ones((20, 13)), np.ones((45, 13)), np.repeat(base, 7, axis=0)]
    qsegs = [np.ones((9, 13)), np.ones((32, 13)), np.ones((50, 13)), np.repeat(base[:4], 3, axis=0), np.repeat(base, 9, axis=0),
             rng.integers(0, 2, size=(30, 13)).astype(np.float64)]
    dflat, doff = flat_of(dsegs, 13)
    pairs = [(qi, di) for qi in range(len(qsegs)) for di in range(len(dsegs))]
    qflat, qoff = flat_of([qsegs[a] for a, _ in pairs], 13)
    idx = np.array([b for _, b in pairs], dtype=np.uint32)
    dev = api.DeviceDictionary(ctx, dflat, doff, 13)
    paths, dist = dev.align(qflat, qoff, idx)
    check_against_oracle(paths, dist, dflat, doff, qflat, qoff, idx)


def test_empty_none_nan_and_index_base(ctx):
    rng = np.random.default_rng(7)
    dsegs = [rng.normal(size=(n, 12)) for n in (5, 0, 40, 12)]
    dsegs[3][4, 2] = np.nan
    dflat, doff = flat_of(dsegs, 12)
    qsegs = [rng.normal(size=(n, 12)) for n in (0, 7, 7, 7, 36, 7, 3)]
    qsegs[5][1, 0] = np.nan
    qflat, qoff = flat_of(qsegs, 12)
    for base in (0, 1000):
        dev = api.DeviceDictionary(ctx, dflat, doff, 12, index_base=base)
        idx = np.array([0, NONE, 1, 3, 2, 0, 2], dtype=np.uint32)
        gidx = np.where(idx == NONE, idx, idx + base).astype(np.uint32)
        paths, dist = dev.align(qflat, qoff, gidx)
        check_against_oracle(paths, dist, dflat, doff, qflat, qoff, gidx, base)
        for p in (0, 1, 2, 3, 5):  # empty query, 0xFFFFFFFF, empty segment, NaN in the segment, NaN in the query
            assert paths[p].shape == (0, 2) and np.isinf(dist[p])
        assert paths[4].shape[0] >= 40 and np.isfinite(dist[6])


def test_invalid_index_and_capacity(ctx):
    rng = np.random.default_rng(8)
    dflat, doff = flat_of([rng.normal(size=(n, 12)) for n in (5, 9)], 12)
    qflat, qoff = flat_of([rng.normal(size=(n, 12)) for n in (4, 6)], 12)
    dev = api.DeviceDictionary(ctx, dflat, doff, 12, index_base=10)
    L = ctx.lib
    path = np.empty((64, 2), dtype=np.uint32)
    poff = np.empty(3, dtype=np.uint64)
    dist = np.empty(2)

    def call(idx, cap):
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        return L.ss_dict_align(dev.h, qflat.ctypes.data, qoff.ctypes.data, 2, idx.ctypes.data, path.ctypes.data, cap, poff.ctypes.data,
                               dist.ctypes.data)

    assert call([10, 12], 64) == SS_ERR_INVALID  # local index 2 of 2 segments
    assert call([9, 11], 64) == SS_ERR_INVALID   # below index_base
    need = (4 + 5 - 1) + (6 + 9 - 1)
    assert call([10, 11], need - 1) == SS_ERR_INVALID
    assert call([10, 11], need) == 0
    assert call([NONE, 11], 6 + 9 - 1) == 0 and int(poff[1]) == 0
    import torch
    qs = api.DeviceQueries(ctx, qflat, qoff, 12)
    d_idx = torch.tensor([10, 11], dtype=torch.int32, device="cuda")
    d_path = torch.empty((64, 2), dtype=torch.int32, device="cuda")
    d_off = torch.empty(3, dtype=torch.int64, device="cuda")
    d_dist = torch.empty(2, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    need_dev = (4 + 9 - 1) + (6 + 9 - 1)
    args = lambda cap: (dev.h, qs.h, d_idx.data_ptr(), d_path.data_ptr(), cap, d_off.data_ptr(), d_dist.data_ptr())
    assert L.ss_dict_align_dev(*args(need_dev - 1)) == SS_ERR_INVALID
    assert L.ss_dict_align_dev(*args(need_dev)) == 0
    ctx.sync()
    d_idx[1] = 13  # out of range: only the device sees it -> empty path, NaN
    torch.cuda.synchronize()
    assert L.ss_dict_align_dev(*args(need_dev)) == 0
    ctx.sync()
    o = d_off.cpu().numpy()
    assert o[2] == o[1] and np.isnan(d_dist.cpu().numpy()[1])


def dev_align(ctx, dev, qs, nq, d_idx, cap):
    import torch
    d_path = torch.empty((max(cap, 1), 2), dtype=torch.int32, device="cuda")
    d_off = torch.empty(nq + 1, dtype=torch.int64, device="cuda")
    d_dist = torch.empty(nq, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    n0 = ctx.launches
    ctx.check(ctx.lib.ss_dict_align_dev(dev.h, qs.h, d_idx.data_ptr(), d_path.data_ptr(), cap, d_off.data_ptr(), d_dist.data_ptr()))
    launches = ctx.launches - n0
    ctx.sync()
    o = d_off.cpu().numpy().view(np.uint64)
    pth = d_path.cpu().numpy().view(np.uint32)
    return [pth[int(o[p]):int(o[p + 1])] for p in range(nq)], d_dist.cpu().numpy(), launches


def test_dev_call_equals_host_call_and_chains_after_match_dev(ctx):
    import torch
    d, doff = synth.segments(10000, 13, seed=1234)
    q, qoff = synth.segments(1000, 13, seed=5678)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    idx, mdist = dev.match(q, qoff, SS_DTW, 1)
    hp, hd = dev.align(q, qoff, idx[:, 0])
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    cap = int(np.sum(np.diff(qoff).astype(np.int64) + dev.max_len - 1))
    d_idx = torch.from_numpy(idx[:, 0].astype(np.int32)).cuda()
    dp, dd, launches = dev_align(ctx, dev, qs, 1000, d_idx, cap)
    assert launches == 3
    assert all(np.array_equal(a, b) for a, b in zip(dp, hp)) and np.array_equal(bits(dd), bits(hd))
    # chained: the match's device output feeds the align with no synchronisation in between
    o_idx = torch.empty((1000, 1), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((1000, 1), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 1, o_idx.data_ptr(), o_dist.data_ptr()))
    dp2, dd2, launches2 = dev_align(ctx, dev, qs, 1000, o_idx, cap)
    assert launches2 == 3
    assert np.array_equal(o_idx.cpu().numpy().view(np.uint32)[:, 0], idx[:, 0])
    assert all(np.array_equal(a, b) for a, b in zip(dp2, hp)) and np.array_equal(bits(dd2), bits(mdist[:, 0]))


def test_align_leaves_the_match_counters_alone(ctx):
    import torch
    d, doff = synth.segments(3000, 13, seed=11)
    q, qoff = synth.segments(300, 13, seed=12)
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    idx, _ = dev.match(q, qoff, SS_DTW, 1)
    counters = lambda: (dev.last_scan_kind, dev.last_work, dev.last_uncertified, dev.last_tc_fallback, dev.last_exhaustive)
    want = counters()
    dev.align(q, qoff, idx[:, 0])
    assert counters() == want
    # a pending asynchronous DTW match completes before the align runs
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    o_idx = torch.empty((300, 1), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((300, 1), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 1, o_idx.data_ptr(), o_dist.data_ptr()))
    paths, dist = dev.align(q, qoff, idx[:, 0])
    ctx.sync()
    assert np.array_equal(o_idx.cpu().numpy().view(np.uint32), idx)
    assert counters() == want
    check_against_oracle(paths, dist, d, doff, q, qoff, idx[:, 0])
    # the mode of the last match does not matter
    ci, _ = dev.match(q, qoff, SS_COSINE_REF, 1)
    paths, dist = dev.align(q, qoff, ci[:, 0])
    check_against_oracle(paths, dist, d, doff, q, qoff, ci[:, 0])


def sounds_of(ctx, segs):
    return [api.Sound(np.zeros(1024 + 256 * max(s.shape[0] - 1, 0)), 44100.0, s, 0.0, s.mean(axis=0) if s.shape[0] else np.full(12, np.nan), None, ctx)
            for s in segs]


def test_python_sound_dictionary_align(ctx):
    rng = np.random.default_rng(9)
    dsegs = [rng.normal(size=(n, 12)) * 3 for n in rng.integers(1, 80, size=60)]
    qsegs = [rng.normal(size=(n, 12)) * 3 for n in rng.integers(1, 80, size=25)]
    sd = api.SoundDictionary(ctx, SS_DTW)
    sd.sounds = sounds_of(ctx, dsegs)
    qsnd = sounds_of(ctx, qsegs)
    idx, _ = sd.match_indices(qsnd)
    paths, dist = sd.align(qsnd, idx[:, 0])
    dflat, doff = flat_of(dsegs, 12)
    qflat, qoff = flat_of(qsegs, 12)
    check_against_oracle(paths, dist, dflat, doff, qflat, qoff, idx[:, 0])


DRIVER = r"""
#include <cstdio>
#include <cstring>
#include <fstream>
#include "soundsym.hpp"
using namespace soundsym;
// reads: nd, nq, then per sound its frame count and frames x 12 doubles (dictionary first); prints the top-1 indices, the
// align distances (as bits) and the paths as one JSON line
static std::vector<std::shared_ptr<Sound>> read_sounds(std::ifstream& f, uint64_t n) {
    std::vector<std::shared_ptr<Sound>> out;
    for (uint64_t i = 0; i < n; i++) {
        uint64_t frames = 0;
        f.read((char*)&frames, 8);
        std::vector<double> m(frames * NCOEFFS);
        f.read((char*)m.data(), m.size() * 8);
        out.push_back(std::make_shared<Sound>(Sound::from_samples(std::vector<double>(1024 + 256 * (frames ? frames - 1 : 0), 0.0), 44100.0, m)));
    }
    return out;
}
int main(int argc, char** argv) {
    std::ifstream f(argv[1], std::ios::binary);
    uint64_t nd = 0, nq = 0;
    f.read((char*)&nd, 8);
    f.read((char*)&nq, 8);
    SoundDictionary dict;
    dict.mode = SS_DTW;
    dict.sounds = read_sounds(f, nd);
    auto q = read_sounds(f, nq);
    std::vector<uint32_t> idx;
    std::vector<double> dist;
    dict.match_indices(q, {}, 1, &idx, &dist);
    std::vector<std::vector<std::pair<uint32_t, uint32_t>>> paths;
    std::vector<double> adist;
    dict.align(q, idx, &paths, &adist);
    printf("{\"idx\": [");
    for (size_t p = 0; p < nq; p++) printf("%s%u", p ? ", " : "", idx[p]);
    printf("], \"dist_bits\": [");
    for (size_t p = 0; p < nq; p++) {
        uint64_t b;
        memcpy(&b, &adist[p], 8);
        printf("%s\"%llu\"", p ? ", " : "", (unsigned long long)b);
    }
    printf("], \"paths\": [");
    for (size_t p = 0; p < nq; p++) {
        printf("%s[", p ? ", " : "");
        for (size_t e = 0; e < paths[p].size(); e++) printf("%s%u, %u", e ? ", " : "", paths[p][e].first, paths[p][e].second);
        printf("]");
    }
    printf("]}\n");
    return 0;
}
"""


def test_cpp_sound_dictionary_align(ctx, tmp_path):
    import json
    rng = np.random.default_rng(10)
    dsegs = [rng.normal(size=(n, 12)) * 3 for n in rng.integers(1, 70, size=40)]
    qsegs = [rng.normal(size=(n, 12)) * 3 for n in rng.integers(1, 70, size=15)]
    src, exe, inp = tmp_path / "align_driver.cpp", str(tmp_path / "align_driver"), tmp_path / "in.bin"
    src.write_text(DRIVER)
    lib = os.path.join(ROOT, "soundsym_b200")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I" + os.path.join(ROOT, "include"), str(src), "-o", exe, "-L" + lib,
                           "-lsoundsym_b200", "-Wl,-rpath," + lib])
    with open(inp, "wb") as f:
        f.write(np.array([len(dsegs), len(qsegs)], dtype="<u8").tobytes())
        for s in dsegs + qsegs:
            f.write(np.array([s.shape[0]], dtype="<u8").tobytes() + np.ascontiguousarray(s, dtype="<f8").tobytes())
    out = subprocess.run([exe, str(inp)], capture_output=True, text=True, timeout=300, check=True).stdout
    r = json.loads(out.strip().splitlines()[-1])
    dflat, doff = flat_of(dsegs, 12)
    qflat, qoff = flat_of(qsegs, 12)
    idx = np.array(r["idx"], dtype=np.uint32)
    want_idx, _ = O.dtw_topk(dflat, doff, qflat, qoff, 12, 1)
    assert np.array_equal(idx, want_idx[:, 0])
    paths = [np.array(p, dtype=np.uint32).reshape(-1, 2) for p in r["paths"]]
    dist = np.array([int(b) for b in r["dist_bits"]], dtype=np.uint64).view(np.float64)
    check_against_oracle(paths, dist, dflat, doff, qflat, qoff, idx)
