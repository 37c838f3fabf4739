"""GPU parity tests of the matcher subsystem (SURVEY.md §8a rows 14-16, 20): CUDA path through the C ABI vs the oracle."""
import numpy as np
import pytest

from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_COSINE_REF, SS_DTW, SoundsymError

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def cut(mfcc, seg_lens_samples, hop=256):
    frames = (np.asarray(seg_lens_samples, dtype=np.uint64) // np.uint64(hop)).astype(np.uint64)
    off = np.zeros(len(frames) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(frames)
    return mfcc[: int(off[-1])], off


def check_dtw(idx, dist, oidx, odist, k):
    """indices bit-exact; distances are produced by the f64 refine kernel with the oracle's arithmetic -> 1e-12
    (the north-star bar is 1e-4 relative)."""
    assert idx.shape == oidx.shape
    fin = np.isfinite(odist)
    assert np.array_equal(np.isfinite(dist), fin)
    assert np.allclose(dist[fin], odist[fin], rtol=1e-12, atol=0)
    assert np.array_equal(idx, oidx)


def test_dtw_synthetic_small_vs_oracle_and_golden(ctx, synthetic_small):
    d, doff = synth.segments(600, 13, seed=1234)
    q, qoff = synth.segments(48, 13, seed=5678)
    dev = api.DeviceDictionary(ctx, d, doff)
    for k in (1, 4, 8):
        idx, dist = dev.match(q, qoff, SS_DTW, k)
        oidx, odist = O.dtw_topk(d, doff, q, qoff, 13, k)
        check_dtw(idx, dist, oidx, odist, k)
        assert dev.last_uncertified == 0
        assert dev.last_work == int(doff[-1]) * int(qoff[-1])
    idx, dist = dev.match(q, qoff, SS_DTW, 4)
    assert np.array_equal(idx, synthetic_small["dtw_idx"])
    assert np.allclose(dist, synthetic_small["dtw_dist"], rtol=1e-12, atol=0)


def test_dtw_config1_real_segments_long_strips(ctx, section71, sample_excerpt):
    """config 1: queries = segments of sample.wav, dictionary = segments of Section_7_1.wav (C = 12, segments up to 83
    frames -> multi-strip path, queries up to 385 frames)."""
    d, doff = cut(section71["mfcc"], section71["splits_d3t4"])
    q, qoff = cut(sample_excerpt["mfcc"], sample_excerpt["splits_d3t4"])
    dev = api.DeviceDictionary(ctx, d, doff)
    idx, dist = dev.match(q, qoff, SS_DTW, 4)
    check_dtw(idx, dist, sample_excerpt["dtw_idx"], sample_excerpt["dtw_dist"], 4)
    # real segments take the tensor-core path too: 32-column strips + streamed query rows (dtw_h2.cu, k_dtw_scan_h2_long)
    assert dev.last_scan_kind == 1, "config 1 did not run the packed-half tensor-core scan (kind %d)" % dev.last_scan_kind
    assert dev.last_uncertified == 0
    print("\nconfig 1: %d of %d queries left the first tensor-core pass, %d reached the exhaustive stage"
          % (dev.last_tc_fallback, len(qoff) - 1, dev.last_exhaustive))
    dev.set_scan(2)  # and the fp32 CUDA-core scan (the path these fixtures took before) still agrees
    idx2, dist2 = dev.match(q, qoff, SS_DTW, 4)
    assert dev.last_scan_kind == 3
    check_dtw(idx2, dist2, sample_excerpt["dtw_idx"], sample_excerpt["dtw_dist"], 4)


def test_cosine_ref_config1_bit_exact(ctx, section71, sample_excerpt):
    d, doff = cut(section71["mfcc"], section71["splits_d3t4"])
    q, qoff = cut(sample_excerpt["mfcc"], sample_excerpt["splits_d3t4"])
    dev = api.DeviceDictionary(ctx, d, doff)
    idx, dist = dev.match(q, qoff, SS_COSINE_REF, 1)
    assert np.array_equal(idx[:, 0], sample_excerpt["cos_idx"])
    assert np.array_equal(dist[:, 0], sample_excerpt["cos_dist"])  # bit-exact f64


def test_cosine_ref_synthetic_and_targets(ctx, synthetic_small):
    d, doff = synth.segments(600, 13, seed=1234)
    q, qoff = synth.segments(48, 13, seed=5678)
    dev = api.DeviceDictionary(ctx, d, doff)
    idx, dist = dev.match(q, qoff, SS_COSINE_REF, 1)
    assert np.array_equal(idx[:, 0], synthetic_small["cos_idx"]) and np.array_equal(dist[:, 0], synthetic_small["cos_dist"])
    targets = np.linspace(-1e-4, 1e-4, 48)  # at_distance(target != 1), src/sound.rs:351
    idx, dist = dev.match(q, qoff, SS_COSINE_REF, 1, targets)
    oidx, odist = O.cosine_match(d, doff, q, qoff, 13, targets)
    assert np.array_equal(idx[:, 0], oidx) and np.array_equal(dist[:, 0], odist)
    assert dev.last_work == sum(min(int(a), int(b)) for a in np.diff(qoff) for b in np.diff(doff)) * 13


def test_ties_and_self_match(ctx):
    d, doff = synth.segments(200, 12, seed=3)
    # duplicate segment 17 at the end: a query equal to it must report 17 first (lowest index), then the copy
    seg = d[int(doff[17]):int(doff[18])]
    d2 = np.concatenate([d, seg])
    doff2 = np.concatenate([doff, [doff[-1] + np.uint64(len(seg))]]).astype(np.uint64)
    dev = api.DeviceDictionary(ctx, d2, doff2)
    idx, dist = dev.match(seg, np.array([0, len(seg)], dtype=np.uint64), SS_DTW, 3)
    assert list(idx[0, :2]) == [17, 200] and dist[0, 0] == 0.0 and dist[0, 1] == 0.0
    oidx, odist = O.dtw_topk(d2, doff2, seg, np.array([0, len(seg)], dtype=np.uint64), 12, 3)
    check_dtw(idx, dist, oidx, odist, 3)
    cidx, cdist = dev.match(seg, np.array([0, len(seg)], dtype=np.uint64), SS_COSINE_REF, 1)
    oc, od = O.cosine_match(d2, doff2, seg, np.array([0, len(seg)], dtype=np.uint64), 12)
    assert cidx[0, 0] == oc[0] and cdist[0, 0] == od[0]


def test_cosine_ref_first_minimum_wins_whatever_the_scan_order(ctx):
    """The cosine scan walks the dictionary by (length, index), not by index: equal distances must still go to the
    lowest index (the reference's strict '<' fold in index order, src/sound.rs:361-366), across staged groups and slices."""
    rng = np.random.default_rng(5)
    # every segment is orthogonal to the query -> sim = 0, |sim - 1| = 1 for all of them: index 0 (a LONG segment, last in
    # the scan order) must win; then a dictionary where only a few mixed-length segments tie at the minimum
    lens = np.array([9, 1, 2, 1, 7, 3, 1, 2, 2, 5, 1, 40, 1, 1, 6], dtype=np.uint64)
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    d = np.zeros((int(off[-1]), 2))
    d[:, 1] = rng.uniform(1.0, 3.0, size=len(d))
    q = np.zeros((3, 2))
    q[:, 0] = [1.0, 2.0, 0.5]
    qoff = np.array([0, 1, 3], dtype=np.uint64)
    dev = api.DeviceDictionary(ctx, d, off)
    idx, dist = dev.match(q, qoff, SS_COSINE_REF, 1)
    oidx, odist = O.cosine_match(d, off, q, qoff, 2)
    assert np.array_equal(idx[:, 0], oidx) and np.array_equal(dist[:, 0], odist) and list(idx[:, 0]) == [0, 0]
    for n in (37, 1000, 5003):  # many staged groups / several slices: copies of one segment under different indices
        dd, doff = synth.segments(n, 13, seed=n)
        qq, qo = synth.segments(40, 13, seed=n + 1)
        lens = np.diff(doff).astype(np.int64)
        copies = rng.choice(n, size=n // 3, replace=False)
        src = copies[rng.permutation(len(copies))]
        for a, b in zip(copies, src):  # overwrite segment a with (a prefix / tiling of) segment b
            la, lb = int(lens[a]), int(lens[b])
            rows = dd[int(doff[b]):int(doff[b]) + lb]
            dd[int(doff[a]):int(doff[a]) + la] = np.resize(rows, (la, 13))
        dev = api.DeviceDictionary(ctx, dd, doff)
        idx, dist = dev.match(qq, qo, SS_COSINE_REF, 1)
        oidx, odist = O.cosine_match(dd, doff, qq, qo, 13)
        assert np.array_equal(idx[:, 0], oidx) and np.array_equal(dist[:, 0], odist)
        # a query that IS a dictionary segment several times over
        s0 = int(src[0])
        qseg = dd[int(doff[s0]):int(doff[s0 + 1])]
        i1, d1 = dev.match(qseg, np.array([0, len(qseg)], dtype=np.uint64), SS_COSINE_REF, 1)
        o1, od1 = O.cosine_match(dd, doff, qseg, np.array([0, len(qseg)], dtype=np.uint64), 13)
        assert i1[0, 0] == o1[0] and d1[0, 0] == od1[0]


def test_cosine_ref_paired_and_single_query_groups(ctx):
    """The cosine scan gives a warp two query groups of one length wherever a length has two (2 queries x 4 segments per
    thread) and the odd group of a length to a warp of its own, in one launch: every mix of the two, against dictionaries
    whose staged groups of four are uniform, mixed, and longer than the staging buffer (39 frames at C = 13) - bit-exact
    (src/sound.rs:23-38, 351-370), with per-query targets."""
    rng = np.random.default_rng(77)

    def make(lens, c):
        lens = np.asarray(lens, dtype=np.uint64)
        off = np.zeros(len(lens) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        return rng.normal(size=(int(off[-1]), c)), off

    dict_lens = {
        "uniform": np.repeat([5, 17, 32], 40),                                    # staged fours of one length
        "mixed": rng.integers(1, 39, size=203),                                   # nearly every staged four is mixed
        "long": np.concatenate([rng.integers(40, 90, size=21), [3, 12, 39, 40]]),  # beyond the staging buffer (+ boundary)
    }
    query_lens = {
        "pairs only": np.repeat([6, 20], 64),                       # 2 + 2 groups -> two paired items
        "singles only": np.arange(1, 34),                           # 33 lengths, one group each
        "pairs + odd group + partial lanes": np.concatenate([np.repeat(9, 32 * 3 + 5), np.repeat(31, 70), [2, 2, 50, 64]]),
    }
    for dname, dl in dict_lens.items():
        d, doff = make(dl, 13)
        dev = api.DeviceDictionary(ctx, d, doff)
        for qname, ql in query_lens.items():
            q, qoff = make(rng.permutation(ql), 13)
            oidx, odist = O.cosine_match(d, doff, q, qoff, 13)
            idx, dist = dev.match(q, qoff, SS_COSINE_REF, 1)
            assert np.array_equal(idx[:, 0], oidx) and np.array_equal(dist[:, 0], odist), (dname, qname)
            targets = rng.uniform(-1.0, 1.0, size=len(ql))
            ot, odt = O.cosine_match(d, doff, q, qoff, 13, targets=targets)
            it, dt = dev.match(q, qoff, SS_COSINE_REF, 1, targets=targets)
            assert np.array_equal(it[:, 0], ot) and np.array_equal(dt[:, 0], odt), (dname, qname, "targets")


def test_ragged_edge_cases(ctx):
    rng = np.random.default_rng(11)
    # lengths 1, 0 (empty), 33, 64, 65, 200 on both sides
    lens = np.array([1, 0, 33, 64, 65, 200, 2, 31, 32], dtype=np.uint64)
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    d = rng.normal(size=(int(off[-1]), 13)) * 5
    q = rng.normal(size=(int(off[-1]), 13)) * 5
    dev = api.DeviceDictionary(ctx, d, off)
    idx, dist = dev.match(q, off, SS_DTW, 8)
    oidx, odist = O.dtw_topk(d, off, q, off, 13, 8)
    check_dtw(idx, dist, oidx, odist, 8)
    assert np.all(idx[1] == 0xFFFFFFFF) and np.all(np.isinf(dist[1]))  # empty query matches nothing
    cidx, cdist = dev.match(q, off, SS_COSINE_REF, 1)
    oc, od = O.cosine_match(d, off, q, off, 13)
    assert np.array_equal(cidx[:, 0], oc) and np.array_equal(cdist[:, 0], od)
    # zero queries
    idx, dist = dev.match(np.zeros((0, 13)), np.zeros(1, dtype=np.uint64), SS_DTW, 2)
    assert idx.shape == (0, 2)


def test_index_base_and_topk_merge_across_shards(ctx):
    """dictionary split into 3 shards with global index bases; merged top-k must equal the single-shard answer
    (SURVEY.md §8e: results identical for 1/2/4/8 shards)."""
    import ctypes as C
    import torch
    d, doff = synth.segments(900, 13, seed=21)
    q, qoff = synth.segments(40, 13, seed=22)
    k = 4
    whole = api.DeviceDictionary(ctx, d, doff)
    widx, wdist = whole.match(q, qoff, SS_DTW, k)
    cuts = [0, 250, 610, 900]
    li, ld = [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        sh = api.DeviceDictionary(ctx, d, doff[a:b + 1], index_base=a)
        i, dd = sh.match(q, qoff, SS_DTW, k)
        li.append(i)
        ld.append(dd)
    gi = torch.from_numpy(np.stack(li).astype(np.int64)).to(torch.uint32 if hasattr(torch, "uint32") else torch.int32).cuda()
    gd = torch.from_numpy(np.stack(ld)).cuda()
    oi = torch.empty((40, k), dtype=gi.dtype, device="cuda")
    od = torch.empty((40, k), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.ss_topk_merge_dev(ctx.h, gi.data_ptr(), gd.data_ptr(), 3, 40, k, oi.data_ptr(), od.data_ptr()))
    ctx.sync()
    assert np.array_equal(oi.cpu().numpy().astype(np.uint32), widx) and np.array_equal(od.cpu().numpy(), wdist)


def test_error_behaviour(ctx):
    d, doff = synth.segments(10, 13, seed=1)
    with pytest.raises(SoundsymError) as e:
        api.DeviceDictionary(ctx, d, doff, ncoeffs=14)
    assert e.value.code == -1
    empty = api.DeviceDictionary(ctx, np.zeros((0, 13)), np.zeros(1, dtype=np.uint64))
    with pytest.raises(SoundsymError) as e:  # the reference panics on sounds[0] of an empty dictionary (src/sound.rs:369)
        empty.match(d, doff, SS_DTW, 1)
    assert e.value.code == -5
    dev = api.DeviceDictionary(ctx, d, doff)
    with pytest.raises(SoundsymError):
        dev.match(d, doff, SS_DTW, 9)
    with pytest.raises(SoundsymError):
        dev.match(d, doff, SS_COSINE_REF, 2)
    with pytest.raises(SoundsymError):
        dev.match(d, np.array([0, 5, 3], dtype=np.uint64), SS_DTW, 1)


def test_tensor_core_scan_fallback_on_near_duplicates(ctx):
    """A dictionary with many near-identical segments: more than KP candidates sit inside the fp16 scan's error bound,
    so the certification must refuse them and the fp32 scan must re-run those queries; results stay exact and ties still
    resolve to the lowest index."""
    rng = np.random.default_rng(5)
    base, boff = synth.segments(64, 13, seed=9)
    seg = base[int(boff[3]):int(boff[4])]
    L = len(seg)
    copies = [seg + rng.normal(size=seg.shape) * 1e-4 for _ in range(40)] + [seg.copy(), seg.copy()]
    d = np.concatenate([base] + copies)
    doff = np.concatenate([boff, boff[-1] + np.uint64(L) * np.arange(1, len(copies) + 1, dtype=np.uint64)]).astype(np.uint64)
    q = np.concatenate([seg, base[int(boff[10]):int(boff[11])]])
    qoff = np.array([0, L, L + int(boff[11] - boff[10])], dtype=np.uint64)
    dev = api.DeviceDictionary(ctx, d, doff)
    oidx, odist = O.dtw_topk(d, doff, q, qoff, 13, 4)
    # default flow: the packed-half scan's second chance walks the per-slice candidate lists (here: the whole dictionary, no
    # slice list is full), refines all 43 near-identical segments in f64 and certifies - no later stage runs
    idx, dist = dev.match(q, qoff, SS_DTW, 4)
    check_dtw(idx, dist, oidx, odist, 4)
    assert list(idx[0, :3]) == [3, 104, 105] and dist[0, 0] == 0.0  # the original and its two exact copies, lowest index first
    assert dev.last_tc_fallback == 0 and dev.last_exhaustive == 0 and dev.last_uncertified == 0
    # without the second chance (ss_dict_set_scan 3) the later stages are driven: 43 segments within 1e-7 of each other, neither
    # scan can certify query 0 -> exhaustive f64 stage; nothing stays uncertified
    dev.set_scan(3)
    idx, dist = dev.match(q, qoff, SS_DTW, 4)
    check_dtw(idx, dist, oidx, odist, 4)
    assert list(idx[0, :3]) == [3, 104, 105] and dist[0, 0] == 0.0
    assert dev.last_tc_fallback >= 1 and dev.last_exhaustive >= 1 and dev.last_uncertified == 0
    # from the other first stages: fp32-DP tensor-core scan -> fp32 CUDA-core scan -> exhaustive, and fp32 CUDA-core scan ->
    # exhaustive; here neither scan certifies either query of the batch
    for first_stage, scan_kind, tc_fallback, exhaustive in ((1, 2, 2, 2), (2, 3, 0, 2)):
        dev.set_scan(first_stage)
        idx, dist = dev.match(q, qoff, SS_DTW, 4)
        check_dtw(idx, dist, oidx, odist, 4)
        assert list(idx[0, :3]) == [3, 104, 105] and dist[0, 0] == 0.0
        assert dev.last_scan_kind == scan_kind
        assert (dev.last_tc_fallback, dev.last_exhaustive, dev.last_uncertified) == (tc_fallback, exhaustive, 0)


def test_fp32_scan_forced_matches_tensor_core_scan(ctx):
    """One 33-frame segment in the dictionary (far from everything: never a candidate) rules out the fp32-DP tensor-core
    scan and moves the packed-half scan to its strip kernel; on otherwise identical data the results must not change.
    (ss_dict_set_scan(2) forces the fp32 CUDA-core scan itself: see the config-1 and config-3 tests.)"""
    d, doff = synth.segments(300, 13, seed=31)
    q, qoff = synth.segments(70, 13, seed=32)
    tc = api.DeviceDictionary(ctx, d, doff)
    i1, d1 = tc.match(q, qoff, SS_DTW, 4)
    long_seg = np.random.default_rng(1).normal(size=(33, 13)) * 50 + 500  # far from everything: never a candidate
    d2 = np.concatenate([d, long_seg])
    doff2 = np.concatenate([doff, [doff[-1] + np.uint64(33)]]).astype(np.uint64)
    fp = api.DeviceDictionary(ctx, d2, doff2)
    i2, dd2 = fp.match(q, qoff, SS_DTW, 4)
    assert np.array_equal(i1, i2) and np.array_equal(d1, dd2)
    assert fp.last_tc_fallback == 0


def test_tc_scan_declines_loud_queries_and_rekeys_query_blocks_per_dictionary(ctx):
    """(1) The tensor-core scan carries |a|^2 / s in one fp16 slot: queries far louder than the dictionary would overflow
    it, so they must take the fp32 scan and still come out exact. (2) The fp16 query blocks are centred on the dictionary's
    mean frame and scaled by its s: one resident query batch matched against two different dictionaries must be rebuilt
    for the second one."""
    import torch
    d, doff = synth.segments(300, 13, seed=41)
    q, qoff = synth.segments(40, 13, seed=42)
    dev = api.DeviceDictionary(ctx, d, doff)
    loud = q * 400.0
    idx, dist = dev.match(loud, qoff, SS_DTW, 2)
    oidx, odist = O.dtw_topk(d, doff, loud, qoff, 13, 2)
    check_dtw(idx, dist, oidx, odist, 2)
    assert dev.last_uncertified == 0
    d2 = d * 0.5 + 37.5  # another mean frame, another norm scale
    dev2 = api.DeviceDictionary(ctx, d2, doff)
    qs = api.DeviceQueries(ctx, q, qoff)
    nq = len(qoff) - 1
    o_idx = torch.empty((nq, 2), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((nq, 2), dtype=torch.float64, device="cuda")
    for dd, dv in ((d, dev), (d2, dev2), (d, dev)):
        ctx.check(ctx.lib.ss_dict_match_dev(dv.h, qs.h, SS_DTW, None, 2, o_idx.data_ptr(), o_dist.data_ptr()))
        ctx.check(ctx.lib.ss_dict_match_finish(dv.h))  # the device results are final after the fallback decision
        ctx.sync()
        oidx, odist = O.dtw_topk(dd, doff, q, qoff, 13, 2)
        check_dtw(o_idx.cpu().numpy().astype(np.uint32), o_dist.cpu().numpy(), oidx, odist, 2)
        assert dv.last_uncertified == 0
        # (against d2 the queries sit far from the dictionary's mean frame: the packed-half filter's range is exceeded for
        # most pairs and it hands those queries on; against d it certifies them itself)
        if dv is dev:
            assert dv.last_tc_fallback == 0
