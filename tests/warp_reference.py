"""numpy twin of the warped resynthesis (ss_resynth_warped, spec A11 in DESIGN.md §3.5 and include/soundsym_b200.h).

A11, with H = SS_HOP = 256. Target segment t has L_t samples, is matched to dictionary sound m = match_idx[t] of len_m samples,
and has the warping path P_t: (i, j) cells in forward order, as ss_dict_align writes them. X(p) = sample p of sound m for
p < len_m, else 0.0.
  - Blocks: the output of segment t is G = ceil(L_t / H) blocks; block b holds samples n = b H + r, 0 <= r < min(H, L_t - b H).
  - Source frame: for a non-empty path, Lq = 1 + the i of its last cell; j(b) = the j of the first cell of row b for b < Lq,
    j(b) = j(Lq - 1) + (b - Lq + 1) for b >= Lq. For an empty path, j(b) = b. s_b = j(b) H.
  - Samples: a = X(s_b + r). out = a if b = 0 or s_b = s_{b-1} + H; otherwise out = c (H - r) / H + a r / H with
    c = X(s_{b-1} + H + r). The weights are exact dyadic numbers; two products and a sum, each rounded to nearest (no FMA).
  - Segments are concatenated in order.
numpy does not contract a product and a sum into an FMA, so this twin is exact.

  resynth_warped   the twin, vectorised over all segments (fit for an hour of audio)
  random_path      a random valid path from (0, 0) (optionally ending at (Lq - 1, Ld - 1), as a DTW path does)
  flatten          list of [n, 2] paths -> (cells uint32 [N, 2], offsets uint64 [nseg + 1])
"""
import numpy as np

H = 256


def flatten(paths):
    off = np.zeros(len(paths) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([p.shape[0] for p in paths])
    cells = np.concatenate([np.asarray(p, dtype=np.uint32).reshape(-1, 2) for p in paths]) if int(off[-1]) else np.zeros((0, 2), dtype=np.uint32)
    return np.ascontiguousarray(cells, dtype=np.uint32), off


def random_path(rng, lq, ld, to_corner=True, p_diag=0.4):
    """(0, 0) then steps (1, 0), (0, 1), (1, 1); to_corner: ends at (lq - 1, ld - 1) without leaving the lq x ld matrix. Otherwise
    any number of steps in [0, lq + ld), free to leave it (lq, ld then only set the length)."""
    if lq == 0 or ld == 0:
        return np.zeros((0, 2), dtype=np.uint32)
    i = j = 0
    cells = [(0, 0)]
    if to_corner:
        while (i, j) != (lq - 1, ld - 1):
            if i == lq - 1:
                j += 1
            elif j == ld - 1:
                i += 1
            else:
                u = rng.random()
                if u < p_diag:
                    i, j = i + 1, j + 1
                elif u < (1 + p_diag) / 2:
                    i += 1
                else:
                    j += 1
            cells.append((i, j))
    else:
        for _ in range(int(rng.integers(0, lq + ld))):
            step = [(1, 1), (1, 0), (0, 1)][int(rng.integers(0, 3))]
            i, j = i + step[0], j + step[1]
            cells.append((i, j))
    return np.array(cells, dtype=np.uint32)


def resynth_warped(dict_samples, dict_off, match_idx, cells, path_off, target_lens):
    ds = np.ascontiguousarray(dict_samples, dtype=np.float64)
    doff = np.asarray(dict_off, dtype=np.int64)
    mi = np.asarray(match_idx, dtype=np.int64)
    cells = np.asarray(cells, dtype=np.int64).reshape(-1, 2)
    poff = np.asarray(path_off, dtype=np.int64)
    L = np.asarray(target_lens, dtype=np.int64)
    nseg = L.shape[0]
    total = int(L.sum())
    if total == 0:
        return np.zeros(0)
    # ---- per block: source frame j(b) -------------------------------------------------------------------------------------
    G = (L + H - 1) // H
    nblk = int(G.sum())
    bseg = np.repeat(np.arange(nseg), G)
    bstart = np.zeros(nseg + 1, dtype=np.int64)
    bstart[1:] = np.cumsum(G)
    b = np.arange(nblk, dtype=np.int64) - bstart[bseg]
    cseg = np.repeat(np.arange(nseg), np.diff(poff))
    first = np.ones(cells.shape[0], dtype=bool)  # a cell starts a row iff it is its path's first cell or its i differs from the previous
    first[1:] = (cells[1:, 0] != cells[:-1, 0]) | (cseg[1:] != cseg[:-1])
    row_j = cells[first, 1]  # per segment, rows 0 .. Lq-1 in order
    lq = np.bincount(cseg[first], minlength=nseg).astype(np.int64)
    roff = np.zeros(nseg + 1, dtype=np.int64)
    roff[1:] = np.cumsum(lq)
    lqb = lq[bseg]
    row = np.minimum(b, np.maximum(lqb - 1, 0))
    j = b.copy()  # empty path: the diagonal
    has = lqb > 0
    j[has] = row_j[roff[bseg][has] + row[has]] + (b[has] - row[has])
    s = j * H
    prev = np.zeros_like(s)  # s_{b-1}; only read where b > 0
    prev[1:] = s[:-1]
    contig = (b == 0) | (s == prev + H)
    # ---- per sample -----------------------------------------------------------------------------------------------------
    blen = np.minimum(H, L[bseg] - b * H)
    blk = np.repeat(np.arange(nblk), blen)
    ostart = np.zeros(nblk + 1, dtype=np.int64)
    ostart[1:] = np.cumsum(blen)
    r = np.arange(total, dtype=np.int64) - ostart[blk]
    m = mi[bseg][blk]
    base, ln = doff[m], doff[m + 1] - doff[m]
    a = _x(ds, base, ln, s[blk] + r)
    out = a.copy()
    cf = ~contig[blk]
    if np.any(cf):
        rc = r[cf]
        c = _x(ds, base[cf], ln[cf], prev[blk][cf] + H + rc)
        out[cf] = c * ((H - rc).astype(np.float64) / H) + a[cf] * (rc.astype(np.float64) / H)
    return out


def _x(ds, base, ln, p):
    """X(p): sample p of the matched sound, 0.0 at or past its end"""
    ok = p < ln
    if not ds.shape[0]:
        return np.zeros(p.shape[0])
    return np.where(ok, ds[np.where(ok, base + p, 0)], 0.0)
