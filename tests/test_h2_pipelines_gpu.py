"""The two-pipeline packed-half scan (dtw_h2.cu k_dtw_scan_h2_2p): pipeline p of a CTA takes tiles p, p + 2, .. of its slice.

With one group of queries the scan cuts the dictionary into about one slice per SM (148 on a B200), so the dictionary size
sets the tiles per slice: 4 segments of 17..32 frames are one slice of one tile (pipeline 1 has nothing to do), ~1 200 make
slices of about two tiles and ~1 800 slices of about three (pipeline 0 has one tile more), and tiles of different lengths mix
slices of 1, 2 and 3 tiles. Segments of 9..16 frames are the NB = 2 kind, which runs the same kernel.

Every case checks the matcher's indices and distances against the f64 oracle, and every raw scan value of
ss_dict_debug_h2_scan against the rounded-frame DTW bound the certification rests on (as in test_parity_large_gpu.py).
"""
import numpy as np
import pytest

from oracle import oracle as O
from soundsym_b200 import api, synth
from soundsym_b200._lib import SS_DTW

pytestmark = pytest.mark.gpu

C = 13


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0)


def rounded_operands(x, mu):
    """the scan's fp16 operands as f64: fp16(fp32(x - mu)), exactly k_h2_dict_tiles / k_tc_query_tiles' conversion"""
    return (x - mu).astype(np.float32).astype(np.float16).astype(np.float64)


@pytest.mark.parametrize("nd,lmin,lmax,nq", [
    (4, 24, 24, 100),       # one slice of one tile
    (8, 17, 32, 100),       # one tile per slice, two kinds of column count
    (1184, 24, 24, 100),    # slices of two equal tiles
    (1776, 24, 24, 100),    # slices of three equal tiles
    (1500, 17, 32, 300),    # unequal tiles: slices of 1, 2 and 3 tiles; three query groups
    (1500, 9, 32, 128),     # NB = 1 and NB = 2 kinds (the last kind gets slices of half the cost)
])
def test_two_pipeline_scan_exact_and_a_lower_bound(ctx, nd, lmin, lmax, nq):
    d, doff = synth.segments(nd, C, lmin=lmin, lmax=lmax, seed=4321 + nd)
    q, qoff = synth.segments(nq, C, lmin=4, lmax=32, seed=8765 + nd)
    O.set_threads(O.hardware_threads())
    dev = api.DeviceDictionary(ctx, d, doff)
    for k in (1, 2):
        idx, dist = dev.match(q, qoff, SS_DTW, k)
        oidx, odist = O.dtw_topk(d, doff, q, qoff, C, k)
        assert np.array_equal(idx, oidx), "indices differ from the f64 oracle at %s" % (np.argwhere(idx != oidx)[:5].tolist(),)
        assert np.allclose(dist, odist, rtol=1e-12, atol=0)
    scan, mu, scale, S = dev.debug_h2_scan(q, qoff)
    assert scan.shape == (nq, nd) and not np.any(np.isnan(scan))
    dr, qr = rounded_operands(d, mu[:C]), rounded_operands(q, mu[:C])
    ref = O.dtw_matrix(dr, doff, qr, qoff, C)
    lq = (qoff[1:] - qoff[:-1]).astype(np.float64)[:, None]
    ld = (doff[1:] - doff[:-1]).astype(np.float64)[None, :]
    u = 2.0 ** -11
    eta = (13.0 * float(np.max(np.abs(dr))) + 4.0) * 2.0 ** -24 / S
    fin = np.isfinite(scan)
    assert fin.any()
    lower = (scan.astype(np.float64) - eta) * (1.0 + u) ** -(lq + ld + 2.0)
    assert np.max(lower[fin] / ref[fin]) <= 1.0, "the packed-half scan's certified lower bound exceeds the rounded-frame DTW"
    assert (scan.astype(np.float64)[fin] / ref[fin] - 1.0).min() >= -0.05
    # a pair may only read +inf if its path sum really is beyond the fp16 range
    npath = lq + ld + 0 * ref
    assert np.all((ref * npath * S * (1.0 + u) ** (npath + 2.0))[~fin] >= 65504.0 * 0.999)
