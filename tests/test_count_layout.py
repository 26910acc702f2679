"""The layout mirror (count_layout.py) that the tests of k_basefc_count rely on, checked by brute force on random
feature sets with nested, duplicated, empty, touching and unfetchable intervals: every stabbing list is the set of
features covering its segment, a read finds exactly the features it overlaps through the index, and no read of a
tile overlaps a feature below the tile's jmin."""

import numpy as np
import pytest

import count_layout as cl
from recsets import build, cell_keys, umi_keys


def random_case(seed):
    rng = np.random.RandomState(seed)
    n_gid = int(rng.randint(1, 5))
    L = int(rng.choice([300, 3000, 40000]))
    nf = int(rng.randint(1, 120))
    gid = rng.randint(-1, n_gid + 1, nf)
    beg = rng.randint(-5, L, nf)
    end = beg + rng.randint(-3, L // 3 + 2, nf)
    k = nf // 4
    beg[:k] = beg[k:2 * k]                                    # duplicated and nested
    end[:k] = np.maximum(end[k:2 * k] - rng.randint(0, 3, k), beg[:k])
    gid[:k] = gid[k:2 * k]
    t = nf // 8
    beg[2 * k:2 * k + t] = end[k:k + t]                       # touching
    gid[2 * k:2 * k + t] = gid[k:k + t]
    runs, pos, n = [], [], 0
    for r in range(int(rng.randint(1, 5))):
        m = int(rng.choice([1, 40, 1024, 1500, 3000]))
        pos.append(np.sort(rng.randint(0, L, m)))
        runs.append((r, int(rng.randint(-1, n_gid + 1)), n, n + m))
        n += m
    pos = np.concatenate(pos)
    end_r = pos + rng.randint(1, 300, n)
    reads = build(pos, cell_keys(1)[0], umi_keys(1)[0], runs, end=end_r)
    return reads, gid, beg, end, n_gid


def overlapping(ix, g, pos, end):
    j0, j1 = ix.sf_goff[g], ix.sf_goff[g + 1]
    return {j for j in range(j0, j1) if ix.sf_beg[j] < end and ix.sf_end[j] > pos}


@pytest.mark.parametrize("seed", range(12))
def test_stabbing_lists_cover_their_segments(seed):
    reads, gid, beg, end, n_gid = random_case(seed)
    ix = cl.Index(gid, beg, end, n_gid)
    valid = [(g, b, e) for g, b, e in zip(gid, beg, end) if 0 <= g < n_gid and b >= 0 and e > b]
    assert len(ix.sf_row) == len(valid)
    for g in range(n_gid):
        for k in range(ix.bnd_goff[g], ix.bnd_goff[g + 1] - 1):
            for p in (ix.bnd[k], ix.bnd[k + 1] - 1):
                cover = {j for j in range(ix.sf_goff[g], ix.sf_goff[g + 1]) if ix.sf_beg[j] <= p < ix.sf_end[j]}
                assert set(ix.stabbing(k).tolist()) == cover
        for k in range(ix.bnd_goff[g], ix.bnd_goff[g + 1]):
            starts = {j for j in range(ix.sf_goff[g], ix.sf_goff[g + 1]) if ix.sf_beg[j] == ix.bnd[k]}
            assert set(range(ix.fb[k], ix.fb[k + 1])) == starts


def check_tiles(seed):
    """every read of every tile against brute force; returns the number of live tiles"""
    reads, gid, beg, end, n_gid = random_case(seed)
    ix = cl.Index(gid, beg, end, n_gid)
    pe = reads.pos_end
    n_live = 0
    for d in cl.tile_descs(reads, ix):
        recs = range(d.rec_beg, d.rec_beg + d.n_rec)
        want = [overlapping(ix, d.gid, pe[i, 0], pe[i, 1]) if 0 <= d.gid < n_gid else set() for i in recs]
        if not d.live:
            assert not any(want)
            continue
        n_live += 1
        assert d.bx <= d.by and (d.by == d.b1 or ix.bnd[d.by] >= d.max_end)
        for i, w in zip(recs, want):
            assert all(j >= d.jmin for j in w)
            # count_record: the stabbing list of the segment holding pos, then the features beginning at a
            # boundary in (pos, end) -- from ub up to the tile's by
            ub = cl.first_bnd_above(ix, d, pe[i, 0])
            assert d.bx <= ub <= d.by
            got = set(ix.stabbing(ub - 1).tolist()) if ub > d.b0 else set()
            for kb in range(ub, d.by):
                if ix.bnd[kb] >= pe[i, 1]:
                    break
                got |= set(range(ix.fb[kb], ix.fb[kb + 1]))
            assert got == w
    return n_live


def test_reads_find_their_features_above_jmin():
    assert sum(check_tiles(s) for s in range(12)) > 10
