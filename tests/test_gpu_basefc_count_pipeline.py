"""k_basefc_count's tile pipeline when the warps of a CTA do not wait for each other at tile ends: a warp that runs
out of chunks in tile k goes on to tile k+1 while others still count tile k, and the duplicate filter, the chunk
counter and the index stage of a tile are reused two (live) tiles later.  Against the CPU oracle entry by entry.

One batch serves the three cases; its layout is checked through the mirror in count_layout.py:
- skewed tiles: the 32-record chunks of a tile alternate between records with 20-entry stabbing lists (an eighth
  of them with stored CIGARs) and records that the flag filter drops, so the warps that draw them end the tile far
  apart; every seventh tile is almost empty, so that fast warps reach the next tile early;
- stale-filter aliasing: every live tile has its own features (jmin = 22 t) and one read over its local features 0
  and 1 with the same UMI and cell, so that every tile puts the same filter keys in -- naming different features.
  A filter that still held the keys of an earlier tile would drop that read's pairs, whichever tiles a CTA gets;
- short runs: dead one- to three-record tiles (a contig without features) between live ones, and epochs of 1, 2
  and 3 tiles (CTAs with one tile each) or of 2 and 3 tiles per CTA of the full grid."""

import numpy as np
import pytest

import count_layout as cl
from recsets import D, I, M
from test_gpu_basefc_count_edges import MODES, Batch, Conf, check, umis

N_CELLS = 24
N_LIVE = 1300
N_LOCAL = 22                     # features per live tile: the two alias features and 20 long ones
ALIAS_COL = 7
CIG = [(M, 25), (D, 2), (M, 20), (I, 3), (M, 13)]           # 60 reference bases
GRID = 148 * 4


def heavy(t, c):
    """chunk c of live tile t holds counted records"""
    return t % 7 != 3 and (c + t) % 2 == 0


def pipeline_batch():
    rng = np.random.RandomState(31)
    B = Batch()
    u = umis(41)
    for t in range(N_LIVE):
        base = 2000 * t
        B.feat(0, base, base + 40)                        # local features 0 and 1: the alias keys
        B.feat(0, base + 30, base + 60)
        for i in range(20):                               # local features 2 .. 21 cover every other read
            B.feat(0, base + 90 + i, base + 900 + i)
        i = np.arange(3, 1024)
        pos = np.concatenate([[base, base + 25, base + 25], base + 100 + (i - 3) * 600 // 1021])
        ops = [None] * 3 + [CIG if k % 8 == 0 else None for k in range(len(i))]
        flag = np.array([4, 0, 0] + [0 if heavy(t, k // 32) else 4 for k in i])
        col = np.concatenate([[0, ALIAS_COL, ALIAS_COL], rng.randint(0, N_CELLS, len(i))])
        umi = np.concatenate([u[:1], u[:1], u[:1], u[1 + rng.randint(0, 40, len(i))]])
        B.run(0, pos, pos + np.where(np.arange(1024) < 3, 10, 60), ops, col=col, umi=umi, flag=flag)
        for q in range([0, 1, 0, 2, 1, 0, 3][t % 7]):     # dead tiles between the live ones
            m = 1 + (t + q) % 3
            p = np.sort(rng.randint(0, 5000, m))
            B.run(1, p, p + 60, col=rng.randint(0, N_CELLS, m), umi=u[1 + rng.randint(0, 40, m)])
    return B


@pytest.fixture(scope="module")
def pipeline():
    B = pipeline_batch()
    return B, B.reads(N_CELLS)


def test_pipeline_layout(pipeline):
    B, reads = pipeline
    ix, descs = B.layout(reads)
    live = [d for d in descs if d.live]
    assert len(live) == N_LIVE and len(descs) - N_LIVE > N_LIVE // 2
    gaps, run = set(), 0
    for d in descs:
        if d.live:
            gaps.add(run)
            run = 0
        else:
            run += 1
            assert 1 <= d.n_rec <= 3
    assert gaps == {0, 1, 2, 3}
    # every live tile: its own features, numbered from jmin = 22 t, staged boundaries and CIGAR words
    assert [d.jmin for d in live] == list(range(0, N_LOCAL * N_LIVE, N_LOCAL))
    assert all(d.n_rec == 1024 and d.staged and d.cig_staged for d in live)
    pe, flag = reads.pos_end, np.array(B.flag)
    cb = cl.col_bits(N_CELLS)
    ku = cl.umi_compact(umis(41)[0])
    keys = set()
    for t, d in enumerate(live):
        hits = [[j - d.jmin for j in range(d.jmin, d.jmin + N_LOCAL)
                 if ix.sf_beg[j] < pe[i, 1] and ix.sf_end[j] > pe[i, 0]] for i in (d.rec_beg + 1, d.rec_beg + 600)]
        assert hits == [[0, 1], list(range(2, N_LOCAL))]
        # the alias read's filter keys: the same in every tile, for features of that tile only
        keys |= {ku | (jl << cb) | ALIAS_COL for jl in hits[0]}
        assert ix.sf_row[d.jmin] == N_LOCAL * t
    assert len(keys) == 2 and all(k >> cb & ((1 << (24 - cb)) - 1) < cl.filter_bound(N_CELLS) for k in keys)
    # skew: counted and dropped chunks alternate inside a tile
    for t in (0, 1, 2, 3):
        d = live[t]
        per_chunk = [(flag[d.rec_beg + 32 * c:d.rec_beg + 32 * c + 32] == 0).sum() for c in range(32)]
        assert [n > 2 for n in per_chunk] == [heavy(t, c) for c in range(32)]
    assert sum(heavy(3, c) for c in range(32)) == 0 and sum(heavy(0, c) for c in range(32)) == 16


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["seg", "sets"])
@pytest.mark.parametrize("tiles", [None, "1", "2", "3", str(2 * GRID), str(3 * GRID)])
def test_pipeline(gpu_ctx, monkeypatch, pipeline, mode, tiles):
    B, reads = pipeline
    env = dict(MODES[mode])
    if tiles:
        env["XG_EPOCH_TILES"] = tiles
    exp = check(gpu_ctx, monkeypatch, reads, B.gid, B.beg, B.end, N_CELLS, Conf(), env, min_nnz=N_LIVE * 100)
    row, col, val = exp
    alias = (row % N_LOCAL < 2) & (row < N_LOCAL * N_LIVE)
    # the alias read counts once for each of its two features in every live tile
    assert alias.sum() == 2 * N_LIVE and (col[alias] == ALIAS_COL).all() and (val[alias] == 1).all()
