"""The baf kernels at their capacity switches and on every CIGAR operator, each case against oracle.baf through
baf_pileup + baf_count and through baf_fc (SNP filter on the device), for both no_dup_hap values; and basefc on
the CIGAR operators the synthetic inputs never carry.  Every case asserts that it reached the branch it names.

  k_baf_finalize  column ranges of 14 * 1024 cells: 14 336 (one range, full), 14 337 (a second range of one
                  column), 40 000 (three ranges); listed cells with reads on both sides of each range edge
  k_baf_scan      SNPs under a tile's window: <= 8 (linear count), 9 .. 256 (staged in shared memory), > 256
                  (binary search in global memory), none (tile skipped)
  pair buffer     starts at max(2^16, n_reads / 4) (read, SNP) pairs; more pairs grow it and rerun the scan
  first read wins one (cell, UMI) over one SNP in thousands of reads: the first read in record order claims the
                  UMI even with a D / N over the SNP; a read that fails a filter claims nothing"""

import numpy as np
import pytest

from recsets import CIGAR_PANEL, CODE, D, EQ, H, I, M, N, P, S, X, build, cell_keys, cigar_panel, query_len, \
    umi_keys
from xcltk_b200 import engine

pytestmark = pytest.mark.gpu

LETTERS = "ACGTN"
HIST_COLS = 14 * 1024            # cells per column range of k_baf_finalize (baf.cu)
SCAN_SNP_CAP = 256               # SNP positions of a tile staged in shared memory by k_baf_scan


class Conf(object):
    min_mapq, min_len, min_include = 0, 1, 0
    incl_flag, excl_flag, no_orphan = 0, 0, False
    barcodes = True

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return self.barcodes

    def use_umi(self):
        return True


def regions(lists):
    reg_ptr = np.concatenate([[0], np.cumsum([len(r) for r in lists])]).astype(np.int64)
    reg_snp = np.concatenate([np.asarray(r, np.int64) for r in lists] + [np.zeros(0, np.int64)]).astype(np.int32)
    return reg_ptr, reg_snp


def check_baf(ctx, reads, ck, n_cols, snp_pos, ref, alt, reg, conf=None, min_count=1, min_maf=0.0):
    """All SNPs on contig 0.  Returns ({no_dup: the oracle's (AD, DP, OTH)}, timing() of the pileup)."""
    from oracle import oracle
    conf = conf or Conf()
    ref, alt = np.asarray(ref, np.uint8), np.asarray(alt, np.uint8)
    snp_pos = np.asarray(snp_pos, np.int32)
    n = len(snp_pos)
    snp_gid = np.zeros(n, np.int32)
    ii = np.arange(n)
    ref_idx = (ii % 2).astype(np.uint8)
    hap = np.full((n, 8), 2, np.uint8)
    hap[ii, ref] = ref_idx
    hap[ii, alt] = 1 - ref_idx                     # the ALT entry wins when ref == alt, as in SNP.gt
    reg_ptr, reg_snp = regions(reg)
    params = engine.make_params(conf, reads.max_aln_len, with_include=False)
    out, t = {}, None
    d = ctx.upload(reads)
    try:
        for no_dup in (True, False):
            exp = oracle.baf(reads, snp_gid, snp_pos, "".join(LETTERS[x] for x in ref), "".join(LETTERS[x] for x in alt),
                             ref_idx, 1 - ref_idx, reg_ptr, reg_snp, ck, n_cols, oracle.params(conf), min_count, min_maf,
                             no_dup, 4)
            totals, st = ctx.baf_pileup(d, snp_gid, snp_pos, ck, n_cols, params)
            t = ctx.timing()
            tot = totals.sum(axis=1)
            minor = np.minimum(totals[ii, ref], totals[ii, alt])
            keep = ((tot >= min_count) & ~(minor < tot * min_maf)).astype(np.uint8)
            got = ctx.baf_count(st, reg_ptr, reg_snp, hap, keep, no_dup)
            st.close()
            fc = ctx.baf_fc(d, snp_gid, snp_pos, ck, n_cols, params, ref, alt, min_count, min_maf, reg_ptr, reg_snp, hap,
                            no_dup)
            for name, g, f, e in zip(("AD", "DP", "OTH"), got, fc, exp):
                for k in range(3):
                    assert np.array_equal(np.asarray(g[k]), e[k]), (name, no_dup, "baf_count")
                    assert np.array_equal(np.asarray(f[k]), e[k]), (name, no_dup, "baf_fc")
            out[no_dup] = exp
    finally:
        d.close()
    return out, t


def entries(m, row=None):
    """{(row, col): val} of one (row, col, val) triple, optionally of one row only."""
    return {(r, c): v for r, c, v in zip(m[0].tolist(), m[1].tolist(), m[2].tolist()) if row is None or r == row}


def random_codes(rng, n):
    return rng.choice([1, 2, 4, 8], size=n).astype(np.uint8)


# ------------------------------------------------------------------------------------------ k_baf_finalize ranges
@pytest.mark.parametrize("n_cols", [HIST_COLS, HIST_COLS + 1, 40000])
def test_baf_finalize_column_ranges(gpu_ctx, n_cols):
    rng = np.random.RandomState(n_cols)
    n_pass = -(-n_cols // HIST_COLS)
    edges = sorted({c for c in (0, HIST_COLS - 1, HIST_COLS, 2 * HIST_COLS - 1, 2 * HIST_COLS, n_cols - 1) if c < n_cols})
    others = rng.choice(n_cols, size=min(3000, n_cols), replace=False)
    n_reads, L = 30000, 60
    cell = np.concatenate([np.repeat(edges, 25), others[rng.randint(0, len(others), n_reads - 25 * len(edges))]])
    rng.shuffle(cell)
    pos = np.sort(rng.randint(900, 3100, size=n_reads))
    ck = cell_keys(n_cols)
    umi = umi_keys(4)[rng.randint(0, 4, size=n_reads)]          # few UMIs per cell: molecules with several reads
    seq = rng.choice([1, 2, 4, 8, 15], p=[.24, .24, .24, .24, .04], size=(n_reads, L)).astype(np.uint8)
    reads = build(pos, ck[cell], umi, [(0, 0, 0, n_reads)], end=pos + L, seq=seq)
    snp_pos = 1000 + 7 * np.arange(300)
    ref = rng.randint(0, 4, size=300)
    alt = (ref + rng.randint(1, 4, size=300)) % 4
    reg = [np.arange(300)]                                      # a region with entries in every column range
    for k in range(0, 290, 5):                                  # overlapping regions (shared SNPs) ...
        reg.append(np.arange(k, k + 10))
        if k % 20 == 0:
            reg.append([])                                      # ... with empty regions between them
    out, _ = check_baf(gpu_ctx, reads, ck, n_cols, snp_pos, ref, alt, reg)
    ad, dp, oth = out[False]                                    # (no_dup_hap drops molecules seen on both haplotypes)
    c0 = dp[1][dp[0] == 0]
    for p in range(n_pass):                                     # region 0 has entries in every column range
        assert np.any((c0 >= p * HIST_COLS) & (c0 < (p + 1) * HIST_COLS)), p
    assert set(edges) <= set(np.concatenate([dp[1], oth[1]]).tolist())     # ... and both sides of each range edge


# ------------------------------------------------------------------------------------------ k_baf_scan staging
def dense_stretch():
    """One contig: a SNP at every position of [10000, 11000), one every 50 bp elsewhere.  Eight tiles of 1024 reads
    whose windows [first_pos, max_end) hold 8 (sparse), 8, 9, 256, 257, 470, about 200 (sparse) and no SNP."""
    snp_pos = np.concatenate([np.arange(0, 10000, 50), np.arange(10000, 11000), np.arange(11000, 40000, 50)])
    T = 1024
    tiles = [(2000, 2300, 100), (10000, 10000, 8), (10008, 10008, 9), (10017, 10173, 100), (10273, 10430, 100),
             (10430, 10800, 100), (20000, 30000, 100), (45000, 45100, 100)]
    pos = np.concatenate([np.linspace(a, b, T).astype(np.int64) for a, b, _ in tiles])
    end = pos + np.repeat([l for _, _, l in tiles], T)
    rng = np.random.RandomState(77)
    n = len(pos)
    # the 470-SNP tile carries every CIGAR operator (reference length 100, query length 102)
    cig = [(S, 3), (M, 40), (I, 2), (EQ, 20), (D, 5), (X, 35), (S, 2)]
    ops = [cig if 5 * T <= k < 6 * T and k % 3 else None for k in range(n)]
    seq = [random_codes(rng, query_len(o) if o else int(e - p)) for o, p, e in zip(ops, pos, end)]
    ck = cell_keys(50)
    umi = umi_keys(200)[rng.randint(0, 200, size=n)]
    reads = build(pos, ck[rng.randint(0, 50, size=n)], umi, [(0, 0, 0, n)], end=end, ops=ops, seq=seq)
    return reads, ck, snp_pos


def tile_snp_counts(ctx, reads, snp_pos):
    d = ctx.upload(reads)
    try:
        _, tiles = d.index()
    finally:
        d.close()
    s = np.sort(snp_pos)
    return [int(np.searchsorted(s, t[4]) - np.searchsorted(s, t[3])) for t in tiles]


def test_baf_scan_snps_per_tile(gpu_ctx):
    reads, ck, snp_pos = dense_stretch()
    counts = tile_snp_counts(gpu_ctx, reads, snp_pos)
    assert counts[:6] == [8, 8, 9, SCAN_SNP_CAP, SCAN_SNP_CAP + 1, 470] and 150 < counts[6] < SCAN_SNP_CAP
    assert counts[7] == 0
    rng = np.random.RandomState(5)
    ref = rng.randint(0, 4, size=len(snp_pos))
    alt = (ref + rng.randint(1, 4, size=len(snp_pos))) % 4
    lo = np.searchsorted(snp_pos, 10000)
    reg = [np.arange(len(snp_pos)), np.arange(lo, lo + 1000), np.arange(lo + 250, lo + 300), np.arange(0, lo)]
    for c in (Conf(), Conf(min_len=50)):
        out, _ = check_baf(gpu_ctx, reads, ck, 50, snp_pos, ref, alt, reg, conf=c, min_count=2, min_maf=0.1)
        assert len(out[True][1][2]) > 100


def test_baf_pair_buffer_grows_and_the_scan_reruns(gpu_ctx):
    """3 000 reads of 100 bases over the dense stretch: ~300 000 (read, SNP) pairs for a first buffer of 65 536."""
    rng = np.random.RandomState(8)
    n, L = 3000, 100
    pos = np.sort(rng.randint(10000, 10900, size=n))
    snp_pos = np.concatenate([np.arange(5000, 10000, 40), np.arange(10000, 11000)])
    ck = cell_keys(30)
    reads = build(pos, ck[rng.randint(0, 30, size=n)], umi_keys(40)[rng.randint(0, 40, size=n)], [(0, 0, 0, n)],
                  end=pos + L, seq=random_codes(rng, n * L).reshape(n, L))
    ref = rng.randint(0, 4, size=len(snp_pos))
    alt = (ref + 1) % 4
    lo = np.searchsorted(snp_pos, 10000)
    reg = [np.arange(lo, len(snp_pos))] + [np.arange(k, k + 40) for k in range(lo, len(snp_pos) - 40, 30)]
    out, t = check_baf(gpu_ctx, reads, ck, 30, snp_pos, ref, alt, reg)
    assert t[6] > max(65536, n // 4)                 # more pairs than the first buffer held: it grew, the scan reran
    assert len(out[True][1][2]) > 100


# ------------------------------------------------------------------------------------------ first read wins
SNP0 = 5000
CONTENDED = 3000           # reads of the one contended (cell 0, UMI 0) molecule over SNP0 at 4960 .. 5020


def contention_batch(case):
    """(reads, cell keys, n_cols, conf): the contended molecule's first read is the case's, its second has G."""
    rng = np.random.RandomState(len(case))
    n_other = 600
    n = CONTENDED + n_other
    pos = np.full(n, 4960, np.int64)
    q = SNP0 - 4960                                             # query index of SNP0 in a simple read
    ops = [None] * n
    first = {"deletion": [(M, 30), (D, 20), (M, 30)], "refskip": [(M, 30), (N, 20), (M, 30)],
             "min_len": [(M, 45), (D, 15)]}.get(case)
    conf = Conf(min_mapq=20, excl_flag=1024, min_len=50)
    flag, mapq = np.zeros(n, np.uint32), np.full(n, 60, np.uint32)
    if first is not None:
        ops[0] = first
    if case == "mapq":
        mapq[0] = 3
    if case == "flag":
        flag[0] = 1024
    seq = [random_codes(rng, query_len(o) if o else 60) for o in ops]
    b1 = {"N": CODE["N"], "eq": CODE["="], "iupac": CODE["R"]}.get(case, CODE["G"])
    if q < len(seq[0]):                                         # M 45 D 15 / simple: SNP0 is query base q
        seq[0][q] = b1
    seq[1][q] = CODE["G"]
    ck = cell_keys(10)
    if case == "two_bams":                                      # sample mode: column = BAM; one UMI in both runs
        conf.barcodes = False
        h = n // 2
        seq[0][q], seq[h][q] = CODE["A"], CODE["G"]
        reads = build(pos, 0, umi_keys(1)[0], [(0, 0, 0, h), (1, 0, h, n)], end=pos + 60, ops=ops, seq=seq,
                      flag=flag, mapq=mapq)
        return reads, None, 2, conf
    cell = np.concatenate([np.zeros(CONTENDED, np.int64), 1 + rng.randint(0, 9, size=n_other)])
    umi = np.concatenate([np.zeros(CONTENDED, np.int64), 1 + rng.randint(0, 50, size=n_other)])
    reads = build(pos, ck[cell], umi_keys(51)[umi], [(0, 0, 0, n)], end=pos + 60, ops=ops, seq=seq, flag=flag,
                  mapq=mapq)
    return reads, ck, 10, conf


@pytest.mark.parametrize("case", ["deletion", "refskip", "mapq", "flag", "min_len", "N", "eq", "iupac", "two_bams"])
def test_baf_first_read_wins_under_contention(gpu_ctx, case):
    reads, ck, n_cols, conf = contention_batch(case)
    snp_pos = [SNP0, 4970, 5015]
    ref, alt = [0, 0, 1], [2, 2, 3]                             # SNP0: REF A (haplotype 0), ALT G (haplotype 1)
    out, _ = check_baf(gpu_ctx, reads, ck, n_cols, snp_pos, ref, alt, [[0], [0, 1, 2]], conf=conf)
    for no_dup in (True, False):
        ad, dp, oth = (entries(m, row=0) for m in out[no_dup])
        if case == "two_bams":                                  # each BAM's first read: A in column 0, G in column 1
            assert ad == {(0, 1): 1} and dp == {(0, 0): 1, (0, 1): 1} and oth == {}
            continue
        c0 = [{k: v for k, v in m.items() if k[1] == 0} for m in (ad, dp, oth)]
        if case in ("deletion", "refskip"):                     # the first read claims the UMI and counts nowhere
            assert c0 == [{}, {}, {}]
        elif case in ("mapq", "flag", "min_len"):               # the first read claims nothing: the second (G) wins
            assert c0 == [{(0, 0): 1}, {(0, 0): 1}, {}]
        else:                                                   # N, '=' or IUPAC: neither allele
            assert c0 == [{}, {}, {(0, 0): 1}]
        assert len(dp) > 3                                      # the other cells' molecules are counted


# ------------------------------------------------------------------------------------------ CIGAR operators
PANEL_SNPS = [105, 106, 107, 108, 109, 110, 112, 150, 207, 211, 258]
WIDE = ("R6", 106, [(M, 1), (I, 1)] * 150 + [(EQ, 5)], "ACGTT" * 61)    # 301 ops: a count word before the stream


def test_baf_cigar_operators_at_the_snp(gpu_ctx):
    """The hand-built panel (leading S / H, = / X blocks, P, zero-length M, I right before / after a SNP, D and N
    over one) plus a read of 301 ops; REF N and each ALT in turn, one region per SNP and one over all."""
    reads, ck = cigar_panel(CIGAR_PANEL + [WIDE])
    n = len(PANEL_SNPS)
    reg = [[k] for k in range(n)] + [list(range(n))]
    seen = set()
    for a in range(4):
        out, _ = check_baf(gpu_ctx, reads, ck, len(ck), PANEL_SNPS, [4] * n, [a] * n, reg, min_count=0)
        seen |= set(out[True][0][1].tolist())
    assert seen == set(range(len(ck)))                          # every read is some SNP's ALT allele


def exotic(rng):
    """Random CIGARs with the operators aligners other than the synthetic generator emit."""
    a, b = int(rng.randint(0, 40)), int(rng.randint(1, 40))
    k = rng.randint(0, 8)
    if k == 0:
        return [(S, int(rng.randint(1, 10))), (M, a + 1), (I, 2), (M, b)]
    if k == 1:
        return [(H, 5), (S, 3), (EQ, a + 1), (X, 1), (EQ, b), (H, 7)]
    if k == 2:
        return [(M, a + 1), (P, 2), (I, 1), (M, 0), (X, b), (D, 3), (EQ, 4)]
    if k == 3:
        return [(M, 0), (EQ, a + 1), (N, int(rng.randint(10, 500))), (X, b), (S, 4)]
    if k == 4:
        return [(X, a + 1), (I, 1), (EQ, b), (P, 1), (D, 2), (M, 0), (M, 5)]
    if k == 5:
        return [(H, 10), (M, a + 1), (H, 2)]
    if k == 6:
        return [(M, 1), (I, 1)] * 140 + [(X, b)]
    return None


def exotic_batch(seed, n, contig_len, n_cells, n_umis, with_seq):
    rng = np.random.RandomState(seed)
    pos = np.sort(rng.randint(0, contig_len, size=n))
    ops = [exotic(rng) for _ in range(n)]
    end = np.array([p + (sum(l for op, l in o if op in (M, D, N, EQ, X)) if o else int(rng.randint(20, 120)))
                    for p, o in zip(pos, ops)])
    end = np.maximum(end, pos + 1)
    seq = [random_codes(rng, query_len(o) if o else int(e - p)) for o, p, e in zip(ops, pos, end)] if with_seq else None
    ck = cell_keys(n_cells)
    reads = build(pos, ck[rng.randint(0, n_cells, size=n)], umi_keys(n_umis)[rng.randint(0, n_umis, size=n)],
                  [(0, 0, 0, n)], end=end, ops=ops, seq=seq)
    return reads, ck


def test_baf_random_exotic_cigars(gpu_ctx):
    """SNPs every 3 bp under reads of random exotic CIGARs: I / D / N / S next to SNPs in every arrangement."""
    reads, ck = exotic_batch(11, 3000, 4000, 20, 30, True)
    rng = np.random.RandomState(12)
    snp_pos = np.arange(0, 4200, 3)
    ref = rng.randint(0, 4, size=len(snp_pos))
    alt = (ref + rng.randint(1, 4, size=len(snp_pos))) % 4
    reg = [np.arange(k, min(k + 25, len(snp_pos))) for k in range(0, len(snp_pos), 20)]
    for conf in (Conf(), Conf(min_len=30)):
        out, _ = check_baf(gpu_ctx, reads, ck, 20, snp_pos, ref, alt, reg, conf=conf)
        assert len(out[True][1][2]) > 100


# ------------------------------------------------------------------------------------------ basefc CIGAR semantics
@pytest.mark.parametrize("min_include", [0.3, 0.75, 1, 10, 40])
def test_basefc_exotic_cigars_match_oracle(gpu_ctx, min_include):
    """Features every 13 bp, 5 to 60 bp long, cut through = / X / I / D / N / P / zero-length blocks; min_include as
    a fraction and as an integer, so that the included length m decides."""
    from oracle import oracle
    reads, ck = exotic_batch(21, 4000, 20000, 25, 40, False)
    rng = np.random.RandomState(22)
    beg = np.arange(0, 20000, 13).astype(np.int32)
    end = (beg + rng.randint(5, 61, size=len(beg))).astype(np.int32)
    beg, end = np.append(beg, [0, 5000]).astype(np.int32), np.append(end, [20600, 5300]).astype(np.int32)
    gid = np.zeros(len(beg), np.int32)
    for min_len in (1, 30):
        conf = Conf(min_include=min_include, min_len=min_len)
        d = gpu_ctx.upload(reads)
        try:
            row, col, val, _ = gpu_ctx.basefc(d, gid, beg, end, ck, 25, engine.make_params(conf, reads.max_aln_len, True))
        finally:
            d.close()
        o = oracle.basefc(reads, gid, beg, end, ck, 25, oracle.params(conf), 4)
        assert np.array_equal(row, o[0]) and np.array_equal(col, o[1]) and np.array_equal(val, o[2])
        assert len(val) > 1000
