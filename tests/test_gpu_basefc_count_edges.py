"""k_basefc_count at each of its internal switches, on both sides of the value where it flips, against the CPU
oracle entry by entry: the staged boundary slice (SB_MAX, by its alignment) and its branch-free search (nb <= 8),
the staged stabbing entries (STAB_CAP), the staged CIGAR words (CIG_CAP, by the alignment of c_lo, >= 255-op
records at the tile's ends), the include table in shared or global memory (INCL_CAP), the warp's pair stage
(WPAIR_CAP) and its two direct paths, the bound of the tile-local duplicate filter and its clearing from tile to
tile, the persistent CTAs' pipeline over live and dead tiles, and the read-level edges of the feature lookup.

Every case checks through the layout mirror (count_layout.py) that its input reaches the value it is named for.
Each case runs with segments (the default), with every feature a set (XG_SEG_MAX=0, filter on) and with the
filter off (XG_SEG_MODE=0); cases that depend on the CIGAR ranges also run through the streamed call."""

import numpy as np
import pytest

import count_layout as cl
from recsets import D, I, M, N, S, build, cell_keys, umi_keys
from xcltk_b200 import engine

MODES = {"seg": {}, "sets": {"XG_SEG_MAX": "0"}, "nofilter": {"XG_SEG_MODE": "0"}}


class Conf(object):
    min_mapq, min_len, min_include = 20, 1, 0.5
    incl_flag, excl_flag, no_orphan = 0, 772, False

    def __init__(self, barcodes=True, **kw):
        self.barcodes = barcodes
        self.__dict__.update(kw)

    def use_barcodes(self):
        return self.barcodes

    def use_umi(self):
        return True


class Batch(object):
    """Runs appended one after another; one run per (contig, BAM), features per contig."""

    def __init__(self):
        self.runs, self.gid, self.beg, self.end = [], [], [], []
        self.pos, self.rend, self.ops, self.col, self.umi, self.flag, self.mapq = [], [], [], [], [], [], []

    def feat(self, g, b, e):
        self.gid.append(g)
        self.beg.append(int(b))
        self.end.append(int(e))

    def run(self, g, pos, end=None, ops=None, col=0, umi=None, flag=0, mapq=60, bam=0):
        """ops: one [(op, len)] or None per read; end: needed for the reads without a CIGAR"""
        n = len(pos)
        ops = list(ops) if ops is not None else [None] * n
        end = np.asarray(end if end is not None else np.zeros(n), dtype=np.int64)
        rend = [int(p) + max(sum(l for o, l in op if o in (M, D, N)), 1) if op is not None else int(e)
                for p, e, op in zip(pos, end, ops)]
        assert list(pos) == sorted(pos)
        k0 = len(self.pos)
        self.runs.append((bam, g, k0, k0 + n))
        self.pos += [int(p) for p in pos]
        self.rend += rend
        self.ops += ops
        for lst, v in ((self.col, col), (self.umi, umi), (self.flag, flag), (self.mapq, mapq)):
            lst += [int(x) for x in np.broadcast_to(np.asarray(v, dtype=np.uint64), (n,))]

    def reads(self, n_cols):
        ck = cell_keys(n_cols)
        ops = self.ops if any(o is not None for o in self.ops) else None
        return build(np.array(self.pos), ck[np.array(self.col)], np.array(self.umi, dtype=np.uint64), self.runs,
                     end=np.array(self.rend), ops=ops, flag=np.array(self.flag), mapq=np.array(self.mapq))

    def layout(self, reads):
        n_gid = max(r[1] for r in self.runs) + 1
        ix = cl.Index(self.gid, self.beg, self.end, n_gid)
        return ix, cl.tile_descs(reads, ix)


def umis(n, salt=0):
    return umi_keys(n, salt=salt).astype(np.uint64)


def check(ctx, monkeypatch, reads, gid, beg, end, n_cols, conf, env, host=False, min_nnz=1):
    """basefc == oracle.basefc, entry by entry"""
    from oracle import oracle
    gid, beg, end = (np.asarray(a, dtype=np.int32) for a in (gid, beg, end))
    ck = cell_keys(n_cols) if conf.use_barcodes() else None
    with monkeypatch.context() as mp:
        for k, v in env.items():
            mp.setenv(k, v)
        p = engine.make_params(conf, reads.max_aln_len, True)
        d = ctx.upload(reads)
        try:
            if host:
                h = d.download()
                try:
                    got = [np.asarray(x) for x in ctx.basefc_host(h, gid, beg, end, ck, n_cols, p)[:3]]
                finally:
                    h.close()
            else:
                got = [np.asarray(x) for x in ctx.basefc(d, gid, beg, end, ck, n_cols, p)[:3]]
        finally:
            d.close()
    exp = oracle.basefc(reads, gid, beg, end, ck, n_cols, oracle.params(conf), 8)
    assert len(exp[2]) >= min_nnz
    for a, b in zip(got, exp):
        assert np.array_equal(a, b), env
    return exp


def cigar_ops(k, rng):
    """k CIGAR ops: M blocks of 2..6 separated by I 1, D 1..2 and now and then N 20"""
    ops = []
    for q in range(k):
        if q % 2 == 0 or q == k - 1:
            ops.append((M, int(rng.randint(2, 7))))
        else:
            ops.append([(I, 1), (D, int(rng.randint(1, 3))), (N, 20)][int(rng.randint(0, 3))])
    return ops


# ---------------------------------------------------------------------------------------------- 1. boundary slice
N_CELLS = 24


def boundary_batch():
    """One contig per tile.  Features [b_k, b_k+3) on a grid of boundaries 10 apart, so that every boundary but the
    first three ends a feature and every one but the last three begins one.  Tiles: by - (bx & ~3) = 127, 128, 129
    for every bx % 4 (first read on bx, max end on by); nb = by - bx = 8 and 9; a tile before the contig's first
    boundary that ends on it (nb = 0) and one that crosses it."""
    rng = np.random.RandomState(11)
    B = Batch()
    u = umis(40)
    n_bnd = 0                                        # boundaries of the contigs so far (global index of b0)

    def contig(g, n_feat, base=1000):
        for k in range(n_feat):
            B.feat(g, base + 10 * k, base + 10 * (k + 3))
        return [base + 10 * k for k in range(n_feat + 3)]

    def reads_between(g, lo, hi):
        """reads of 25 b from lo to hi, every third one a CIGAR of the same span; the first starts on lo and
        the last ends on hi; one read in four starts on a boundary"""
        pos = sorted(set(list(range(lo, hi - 25, 4)) + list(range(lo, hi - 25, 10)) + list(range(lo + 5, hi - 25, 10)) +
                         [hi - 25]))
        ops = [[(M, 10), (D, 2), (M, 13)] if k % 3 == 0 else None for k in range(len(pos))]
        B.run(g, pos, np.array(pos) + 25, ops, col=rng.randint(0, N_CELLS, len(pos)),
              umi=u[rng.randint(0, len(u), len(pos))])

    g = 0
    targets = [(r, dd) for dd in (127, 128, 129) for r in range(4)] + [("nb", 8), ("nb", 9)]
    for r, dd in targets:
        if r == "nb":
            bl = 5
            by_l = bl + dd
        else:
            bl = 4 + (r - n_bnd) % 4                  # (n_bnd + bl) % 4 == r
            by_l = ((n_bnd + bl) & ~3) + dd - n_bnd
        b = contig(g, by_l + 4)
        reads_between(g, b[bl], b[by_l])
        n_bnd += len(b)
        g += 1
    b = contig(g, 20)                                 # before the first boundary, ending on it: nb == 0
    B.run(g, [900, 950, 975], [950, 1000, 1000], col=[1, 2, 3], umi=u[:3])
    n_bnd += len(b)
    g += 1
    b = contig(g, 20)                                 # first read before the first boundary
    reads_between(g, 940, b[6])
    return B


def test_boundary_slice_layout():
    B = boundary_batch()
    ix, descs = B.layout(B.reads(N_CELLS))
    live = [d for d in descs if d.live]
    assert len(live) == len(descs)
    slices = {(d.bx % 4, d.by - (d.bx & ~3)) for d in live}
    assert {(r, dd) for r in range(4) for dd in (127, 128, 129)} <= slices
    assert {0, 8, 9} <= {d.by - d.bx for d in live}
    assert [d.staged for d in live if d.by - (d.bx & ~3) in (128, 129)].count(False) == 4
    assert any(d.first_pos < ix.bnd[d.b0] < d.max_end for d in live)
    pe = B.reads(N_CELLS).pos_end
    for d in live:
        if d.by - d.bx in (8, 9, 127, 128, 129):
            assert d.first_pos == ix.bnd[d.bx] and d.max_end == ix.bnd[d.by]
            recs = pe[d.rec_beg:d.rec_beg + d.n_rec]
            assert np.isin(recs[:, 0], ix.bnd).sum() > 5 and np.isin(recs[:, 1], ix.bnd).sum() > 5


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("incl", [0, 0.4])
def test_boundary_slice(gpu_ctx, monkeypatch, mode, incl):
    B = boundary_batch()
    check(gpu_ctx, monkeypatch, B.reads(N_CELLS), B.gid, B.beg, B.end, N_CELLS, Conf(min_include=incl),
          MODES[mode], min_nnz=500)


# ------------------------------------------------------------------------------------------- 2. stabbing slice
def stabbing_batch():
    """One tile per contig over two segments [1000, 1500) and [1500, 2000): a features cover both, b only the
    first, so st_n = 2a + b = 127, 128, 129 with the boundaries staged."""
    rng = np.random.RandomState(12)
    B = Batch()
    u = umis(60)
    for g, (a, b) in enumerate([(60, 7), (60, 8), (60, 9), (40, 49)]):
        for k in range(a):
            B.feat(g, 1000, 2000)
        for k in range(b):
            B.feat(g, 1000, 1500)
        pos = np.sort(rng.randint(1000, 1950, 300))
        pos[0] = 1000
        ln = rng.randint(20, 50, 300)
        ops = [[(M, int(x) // 2), (N, 3), (M, int(x) - int(x) // 2)] if k % 4 == 0 else None for k, x in enumerate(ln)]
        B.run(g, pos, np.minimum(pos + ln, 2000), ops, col=rng.randint(0, N_CELLS, 300), umi=u[rng.randint(0, 60, 300)])
    return B


def test_stabbing_slice_layout():
    B = stabbing_batch()
    _, descs = B.layout(B.reads(N_CELLS))
    assert [(d.st_n, d.staged, d.stab_staged) for d in descs] == \
        [(127, True, True), (128, True, True), (129, True, False), (129, True, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_stabbing_slice(gpu_ctx, monkeypatch, mode):
    B = stabbing_batch()
    check(gpu_ctx, monkeypatch, B.reads(N_CELLS), B.gid, B.beg, B.end, N_CELLS, Conf(), MODES[mode], min_nnz=1000)


# --------------------------------------------------------------------------------------------- 3. CIGAR slice
def cigar_batch():
    """The batch's first record has 255 ops (c_lo = 0).  Tiles with c_hi - c_al = 1023, 1024, 1025 for every
    c_lo % 4, each behind a pad run on a contig without features that sets the alignment; tiles whose first or
    last record has 254, 255 or 256 ops.  Reads without a CIGAR are mixed in everywhere."""
    rng = np.random.RandomState(13)
    B = Batch()
    u = umis(50)
    n_g = 20
    for g in range(n_g):
        for b, e in ((0, 6000), (500, 1500), (1000, 2600), (1400, 1410), (2000, 9000), (700, 701)):
            B.feat(g, b, e)
    words = [0]                                       # CIGAR words so far

    def add(g, ops_list):
        pos, ends, k = [], [], 0
        p = 0
        for o in ops_list:
            p += int(rng.randint(0, 5))
            pos.append(p)
            ends.append(p + 40)
            if o is not None:
                words[0] += len(o) + (1 if len(o) >= 255 else 0)
        n = len(pos)
        B.run(g, pos, ends, ops_list, col=rng.randint(0, N_CELLS, n), umi=u[rng.randint(0, len(u), n)])

    def fill(first, n_words, last=None):
        """first record, then records of 1..12 ops (some without a CIGAR) up to n_words words after
        the first record's op words, last record included"""
        out, left = [first], n_words - len(first) - (len(last) + (len(last) >= 255) if last is not None else 0)
        while left > 0:
            if rng.rand() < 0.25:
                out.append(None)
            k = min(int(rng.randint(1, 13)), left)
            out.append(cigar_ops(k, rng))
            left -= k
        if last is not None:
            out.append(last)
        return out

    add(0, [cigar_ops(255, rng), None, cigar_ops(5, rng)])
    g = 0
    for r in range(4):
        for t in (1023, 1024, 1025):
            pad = (r - words[0] + 1) % 4 or 4
            add(n_g, [cigar_ops(pad, rng)])          # contig n_g has no features: a dead tile
            # c_lo = words - 1 (first record below 255 ops), c_hi - c_al = n + 1 + r
            add(g, fill(cigar_ops(9, rng), t - 1 - r))
            g += 1
    for k in (254, 255, 256):
        add(g, fill(cigar_ops(k, rng), 700 + k))
        add(g + 1, fill(cigar_ops(3, rng), 300 + k, last=cigar_ops(k, rng)))
        g += 2
    return B


def test_cigar_slice_layout():
    B = cigar_batch()
    reads = B.reads(N_CELLS)
    _, descs = B.layout(reads)
    cig_off = reads._arrays["cig_off"]
    assert cig_off[0] == 1 and descs[0].c_lo == 0 and reads.fmq[0] >> 24 == 255 and descs[0].live
    live = [d for d in descs if d.live]
    assert {(r, t) for r in range(4) for t in (1023, 1024, 1025)} <= {(d.c_lo % 4, d.c_hi - d.c_al) for d in live}
    assert sum(d.cig_staged for d in live) > 8 and sum(not d.cig_staged for d in live) >= 4
    ncw = reads.fmq >> 24
    cigar = reads._arrays["cigar"]
    n_ops = [int(cigar[cig_off[i] - 1]) if ncw[i] == 255 else int(ncw[i]) for i in range(reads.n)]
    firsts = {n_ops[d.rec_beg] for d in live}
    lasts = {n_ops[d.rec_beg + d.n_rec - 1] for d in live}
    assert {254, 255, 256} <= firsts and {254, 255, 256} <= lasts
    assert all(0 in n_ops[d.rec_beg:d.rec_beg + d.n_rec] for d in live)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES) + ["streamed"])
def test_cigar_slice(gpu_ctx, monkeypatch, mode):
    B = cigar_batch()
    check(gpu_ctx, monkeypatch, B.reads(N_CELLS), B.gid, B.beg, B.end, N_CELLS, Conf(),
          MODES.get(mode, {}), host=mode == "streamed", min_nnz=200)


# ------------------------------------------------------------------------------------------- 4. include table
ALNS = (255, 256, 257, 260, 300)                      # 300: the batch's max_aln_len, the table's last entry
FRACS = (0.1 + 0.2, 1 / 3, 0.95)


def include_batch():
    """Per aligned length n: a read without a CIGAR and a read [S 3, M, I 2, M, S 2] of the same span; features
    that they overlap by m = need - 1, need, need + 1 bases for every fraction's threshold need(n)."""
    B = Batch()
    pos, end, ops = [], [], []
    for k, n in enumerate(ALNS):
        p = 1000 + 2000 * k
        ms = set()
        for f in FRACS:
            tab, _ = engine.include_threshold(f, max(ALNS))
            ms |= {int(tab[n]) - 1, int(tab[n]), int(tab[n]) + 1}
        for m in sorted(x for x in ms if 0 < x <= n):
            B.feat(0, p + n - m, p + n + 50)
        pos += [p, p]
        end += [p + n, p + n]
        ops += [None, [(S, 3), (M, n // 2), (I, 2), (M, n - n // 2), (S, 2)]]
    B.run(0, pos, end, ops, col=np.arange(len(pos)) % 4, umi=umis(len(pos)))
    return B


def test_include_table_layout():
    B = include_batch()
    reads = B.reads(8)
    assert reads.max_aln_len == max(ALNS)
    for f in FRACS:
        tab, _ = engine.include_threshold(f, reads.max_aln_len)
        assert len(tab) == reads.max_aln_len + 1 and cl.INCL_CAP in ALNS and cl.INCL_CAP - 1 in ALNS
        # the global table's entries differ from their predecessors where the test reads them
        assert any(tab[n] != tab[n - 1] for n in ALNS if n >= cl.INCL_CAP)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["seg", "sets"])
@pytest.mark.parametrize("frac,min_len", [(f, 1) for f in FRACS] + [(1 / 3, n) for n in (255, 256, 257)])
def test_include_table(gpu_ctx, monkeypatch, mode, frac, min_len):
    B = include_batch()
    check(gpu_ctx, monkeypatch, B.reads(8), B.gid, B.beg, B.end, 8, Conf(min_include=frac, min_len=min_len),
          MODES[mode], min_nnz=10)


# ----------------------------------------------------------------------------------------------- 5. pair stage
PAIR_K = (1, 2, 3, 4, 5)


def pair_batch():
    """Contig k - 1: 256 reads (8 full chunks), each overlapping exactly k features, every UMI distinct:
    32 k pairs per record step.  Contig 5: every read overlaps 3 features with 256 candidates and 2 with 128."""
    rng = np.random.RandomState(15)
    B = Batch()
    u = umis(256 * (len(PAIR_K) + 1))
    for g, k in enumerate(PAIR_K):
        for q in range(k):
            B.feat(g, 0, 100000 + q)
        pos = 1000 + np.arange(256)
        B.run(g, pos, pos + 50, col=rng.randint(0, N_CELLS, 256), umi=u[256 * g:256 * (g + 1)])
    g = len(PAIR_K)
    pos = 1000 + 10 * np.arange(256)
    for q in range(3):
        B.feat(g, 0, 100000 + q)
    for q in range(2):
        B.feat(g, 0, pos[127] + 1 + q)
        B.feat(g, pos[128] - q, 100000)
    B.run(g, pos, pos + 5, col=rng.randint(0, N_CELLS, 256), umi=u[256 * g:])
    return B


def test_pair_stage_layout():
    B = pair_batch()
    reads = B.reads(N_CELLS)
    ix, descs = B.layout(reads)
    pe = reads.pos_end
    for d in descs:
        assert d.n_rec == 256
        per = {len([j for j in range(ix.sf_goff[d.gid], ix.sf_goff[d.gid + 1])
                    if ix.sf_beg[j] < pe[i, 1] and ix.sf_end[j] > pe[i, 0]]) for i in range(d.rec_beg, d.rec_beg + 256)}
        assert per == {PAIR_K[d.gid] if d.gid < len(PAIR_K) else 5}
    assert {32 * k for k in PAIR_K} == {32, 64, cl.WPAIR_CAP, 128, 160}
    g = len(PAIR_K)                                   # the mixed contig: 150 lies between the candidate counts
    cand = [int(((pe[:, 0] < ix.sf_end[j]) & (pe[:, 1] > ix.sf_beg[j]))[reads.runs[g][2]:reads.runs[g][3]].sum())
            for j in range(ix.sf_goff[g], ix.sf_goff[g + 1])]
    assert sorted(cand) == [128] * 4 + [256] * 3


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES) + ["mixed"])
def test_pair_stage(gpu_ctx, monkeypatch, mode):
    B = pair_batch()
    env = MODES.get(mode, {"XG_SEG_MAX": "150"})
    check(gpu_ctx, monkeypatch, B.reads(N_CELLS), B.gid, B.beg, B.end, N_CELLS, Conf(), env, min_nnz=500)


# ---------------------------------------------------------------------------------- 6. duplicate filter bound
def filter_batch(n_cols):
    """Contig 0: features F_0 .. F_bound+1, 20 b apart, and one tile: reads B_i on F_0 (= jmin) with UMI
    u_i + 2^24 (packed) or interned id + 1, reads A'_i on F_bound-1 (twice each), reads A_i on F_bound with UMI u_i
    -- A_i's filter key equals B_i's if the bound were one larger -- with reads the MAPQ filter drops in between,
    so that the B_i are seen well before the A_i.  Contig 1: 40 distinct UMIs whose keys share one filter slot,
    each read twice in turns."""
    rng = np.random.RandomState(16)
    bound = cl.filter_bound(n_cols)
    B = Batch()
    for i in range(bound + 2):
        B.feat(0, 100 + 20 * i, 110 + 20 * i)
    n = 128
    packed = umis(n, salt=5)
    interned = (np.uint64(1) << np.uint64(63)) | (np.uint64(1000) + np.uint64(2) * np.arange(n, dtype=np.uint64))
    ua = np.concatenate([packed, interned])
    ub = np.concatenate([packed + np.uint64(1 << 24), interned + np.uint64(1)])
    cols = rng.randint(0, n_cols, 2 * n)
    cols[:4] = n_cols - 1
    fa = 100 + 20 * bound
    fa1 = fa - 20
    B.run(0, [100] * (2 * n) + [105] * 384 + [fa1] * n + [fa] * (2 * n),
          [110] * (2 * n) + [106] * 384 + [fa1 + 10] * n + [fa + 10] * (2 * n),
          col=np.concatenate([cols, np.zeros(384, int), cols[:n // 2], cols[:n // 2], cols]),
          umi=np.concatenate([ub, np.full(384, ua[0]), ua[:n // 2], ua[:n // 2], ua]),
          mapq=np.concatenate([np.full(2 * n, 60), np.zeros(384), np.full(3 * n, 60)]))
    # contig 1: keys umi | col that share one slot (local feature 0)
    B.feat(1, 0, 1000)
    cand = umis(200000, salt=77)
    col = n_cols - 2
    slot = cl.filter_slot(cand | np.uint64(col))
    same = cand[slot == np.bincount(slot).argmax()][:40]
    B.run(1, [10] * 80, [60] * 80, col=col, umi=np.concatenate([same, same]))
    return B, bound, ua, ub, cols, same, col


@pytest.mark.parametrize("n_cols", [(1 << 17) + 1, 1 << 18, 1 << 19])
def test_filter_bound_layout(n_cols):
    B, bound, ua, ub, cols, same, col = filter_batch(n_cols)
    assert (cl.col_bits(n_cols), bound) == {(1 << 17) + 1: (18, 64), 1 << 18: (18, 64), 1 << 19: (19, 32)}[n_cols]
    ix, descs = B.layout(B.reads(n_cols))
    d = descs[0]
    assert d.jmin == 0 and ix.sf_beg[bound] == 100 + 20 * bound and d.n_rec == 1024 and len(descs) == 2
    cb = cl.col_bits(n_cols)
    for a, b, c in zip(ua, ub, cols):
        ka = cl.umi_compact(a) | (bound << cb) | int(c)          # what A's key would be inside a bound one larger
        kb = cl.umi_compact(b) | int(c)
        assert ka == kb
    assert len(same) == 40 and len(set(cl.filter_slot(same | np.uint64(col)).tolist())) == 1
    assert descs[1].jmin == bound + 2


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("n_cols", [(1 << 17) + 1, 1 << 18, 1 << 19])
def test_filter_bound(gpu_ctx, monkeypatch, mode, n_cols):
    B, bound, *_ = filter_batch(n_cols)
    exp = check(gpu_ctx, monkeypatch, B.reads(n_cols), B.gid, B.beg, B.end, n_cols, Conf(), MODES[mode], min_nnz=100)
    row, val = exp[0], exp[2]
    assert val[row == bound + 2].sum() == 40 and val[row == bound].sum() == 256


# ------------------------------------------------------------------------------- 7. filter clearing across tiles
N_CLEAR_TILES = 4096


def clearing_batch():
    """One run of N_CLEAR_TILES full tiles; tile t has its own two features [100 t, +40) and [100 t + 30, +30)
    (jmin = 2 t) and one counted read over both, with the same UMI and cell in every tile: the same filter keys
    (local features 0 and 1).  The tile's 1023 other reads are dropped by the flag or MAPQ filter."""
    T = N_CLEAR_TILES
    base = np.repeat(100 * np.arange(T, dtype=np.int64), 1024)
    off = np.tile(np.arange(1024, dtype=np.int64) * 50 // 1024, T)
    pos = base + off
    hit = np.tile(np.arange(1024) == 512, T)
    flag = np.where(hit, 0, np.where(np.arange(T * 1024) % 2, 4, 0))
    mapq = np.where(hit | (flag != 0), 60, 0)
    gid = np.zeros(2 * T, np.int32)
    beg = np.stack([100 * np.arange(T), 100 * np.arange(T) + 30], axis=1).reshape(-1)
    end = beg + np.tile([40, 30], T)
    u = umis(1)
    reads = build(pos, cell_keys(N_CELLS)[7], u[0], [(0, 0, 0, len(pos))], end=pos + 10, flag=flag, mapq=mapq)
    return reads, gid, beg.astype(np.int32), end.astype(np.int32)


@pytest.fixture(scope="module")
def clearing():
    return clearing_batch()


def test_filter_clearing_layout(clearing):
    reads, gid, beg, end = clearing
    ix = cl.Index(gid, beg, end, 1)
    descs = cl.tile_descs(reads, ix)
    assert len(descs) == N_CLEAR_TILES > 148 * 4 * 4
    assert [d.jmin for d in descs] == list(range(0, 2 * N_CLEAR_TILES, 2))
    assert all(d.n_rec == 1024 and d.live for d in descs)
    pe = reads.pos_end
    for d in descs[::97]:                             # the counted read overlaps local features 0 and 1 only
        i = d.rec_beg + 512
        hits = [j for j in range(len(ix.sf_row)) if ix.sf_beg[j] < pe[i, 1] and ix.sf_end[j] > pe[i, 0]]
        assert [j - d.jmin for j in hits] == [0, 1]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["seg", "sets"])
def test_filter_clearing(gpu_ctx, monkeypatch, clearing, mode):
    reads, gid, beg, end = clearing
    exp = check(gpu_ctx, monkeypatch, reads, gid, beg, end, N_CELLS, Conf(), MODES[mode])
    assert len(exp[2]) == 2 * N_CLEAR_TILES and (exp[1] == 7).all() and (exp[2] == 1).all()


# ----------------------------------------------------------------------------------------------- 8. tile pipeline
LIVE_SIZES = (1, 31, 32, 33, 255, 256, 257, 1024, 1500, 700)
DEAD_RUNS = (1, 2, 3, 4, 5, 0, 2, 5)


def pipeline_batch():
    """Live runs of LIVE_SIZES records on contigs 0 and 1 (features over [0, 200 000) and [400 000, 600 000)),
    alternating with 0 to 5 dead one-tile runs: on contig 2, which has no features, or on contig 0 past its last
    feature.  (A tile between two features is live: its window takes the segment after its last read.)  BAM = run
    index % 16 (the column in sample mode)."""
    rng = np.random.RandomState(18)
    B = Batch()
    for g in (0, 1):
        B.feat(g, 0, 200000)
        B.feat(g, 400000, 600000)
        for _ in range(40):
            b = int(rng.choice([rng.randint(0, 200000), rng.randint(400000, 600000)]))
            B.feat(g, b, b + int(rng.randint(300, 20000)))
    u = umis(3000)
    n_run = 0
    for i in range(1100):
        n = LIVE_SIZES[i % len(LIVE_SIZES)]
        lo = int(rng.choice([rng.randint(0, 150000), rng.randint(400000, 550000)]))
        pos = np.sort(rng.randint(lo, lo + 40000, n))
        B.run(i % 2, pos, pos + rng.randint(30, 120, n), col=rng.randint(0, N_CELLS, n),
              umi=u[rng.randint(0, len(u), n)], bam=n_run % 16, mapq=np.where(rng.rand(n) < 0.05, 0, 60))
        n_run += 1
        for q in range(DEAD_RUNS[(i // len(LIVE_SIZES) + i) % len(DEAD_RUNS)]):
            m = int(rng.randint(1, 40))
            g, lo = (2, 0) if q % 2 else (0, 700000)
            pos = np.sort(rng.randint(lo, lo + 5000, m))
            B.run(g, pos, pos + 60, col=rng.randint(0, N_CELLS, m), umi=u[rng.randint(0, len(u), m)], bam=n_run % 16)
            n_run += 1
    return B


@pytest.fixture(scope="module")
def pipeline():
    B = pipeline_batch()
    return B, B.reads(N_CELLS)


def test_tile_pipeline_layout(pipeline):
    B, reads = pipeline
    _, descs = B.layout(reads)
    assert len(descs) > 3000
    live = [d.live for d in descs]
    gaps, run = set(), 0
    for x in live:
        if x:
            gaps.add(run)
            run = 0
        else:
            run += 1
    assert {0, 1, 2, 3, 4, 5} <= gaps
    assert {1, 31, 32, 33, 255, 256, 257, 1024} <= {d.n_rec for d in descs if d.live}
    assert sum(a.gid != b.gid for a, b in zip(descs, descs[1:])) > 1000
    assert sum(1 for d in descs if not d.live and d.gid == 0) > 500           # past the last feature of contig 0


@pytest.mark.gpu
@pytest.mark.parametrize("barcodes", [True, False])
@pytest.mark.parametrize("tiles", [None, "2"])
def test_tile_pipeline(gpu_ctx, monkeypatch, pipeline, barcodes, tiles):
    B, reads = pipeline
    env = {"XG_EPOCH_TILES": tiles} if tiles else {}
    n_cols = N_CELLS if barcodes else 16
    check(gpu_ctx, monkeypatch, reads, B.gid, B.beg, B.end, n_cols, Conf(barcodes=barcodes), env, min_nnz=1000)


# ------------------------------------------------------------------------------------------ 9. read-level edges
def edge_batch():
    """One tile on contig 0: reads that end where a feature begins (with and without a CIGAR; a later read inside the
    feature gives it candidates, and the tile's last read keeps its boundary inside the window); a spliced read whose N covers a whole feature; reads
    with pos == s0 and end == e0; reads one base longer than their feature (CIGARs, aligned length 101 and 100)."""
    B = Batch()
    for b, e in ((150, 250), (1200, 1300), (3000, 3100), (4000, 4100), (5000, 5100)):
        B.feat(0, b, e)
    pos = [100, 100, 200, 1000, 3000, 3000, 4000, 5000, 6000]
    ops = [None, [(S, 2), (M, 50)], [(M, 30)], [(M, 50), (N, 500), (M, 50)], None, [(M, 40), (D, 5), (M, 55)],
           [(M, 101)], [(M, 50), (D, 1), (M, 50)], [(M, 30)]]
    end = [150, 0, 0, 0, 3100, 0, 0, 0, 0]
    B.run(0, pos, end, ops, col=np.arange(9), umi=umis(9))
    return B


def test_read_edges_layout():
    B = edge_batch()
    reads = B.reads(9)
    ix, descs = B.layout(reads)
    d, pe = descs[0], reads.pos_end
    assert len(descs) == 1 and d.live
    assert pe[0, 1] == pe[1, 1] == 150 and cl.first_bnd_above(ix, d, 100) < d.by     # 150 lies inside the window
    assert (pe[3, 0], pe[3, 1]) == (1000, 1600)                   # aligned [1000, 1050) and [1550, 1600)
    assert (pe[4, 0], pe[4, 1]) == (pe[5, 0], pe[5, 1]) == (3000, 3100)
    assert (pe[6, 0], pe[6, 1]) == (4000, 4101) and (pe[7, 0], pe[7, 1]) == (5000, 5101)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("incl", [0, 100, 101])
def test_read_edges(gpu_ctx, monkeypatch, mode, incl):
    B = edge_batch()
    exp = check(gpu_ctx, monkeypatch, B.reads(9), B.gid, B.beg, B.end, 9, Conf(min_include=incl), MODES[mode],
                min_nnz=0)
    got = dict(zip(zip(exp[0].tolist(), exp[1].tolist()), exp[2].tolist()))
    if incl == 0:         # every candidate counts, the spliced read over the feature in its gap too; reads 0, 1 never
        assert got == {(0, 2): 1, (1, 3): 1, (2, 4): 1, (2, 5): 1, (3, 6): 1, (4, 7): 1}
    else:                 # the reads one base longer than their feature keep 100 and 99 of 101 and 100 aligned bases
        assert got == ({(2, 4): 1, (3, 6): 1} if incl == 100 else {})
