"""SNP discovery (xg_snp_discover) at the edges of its raw scan, target layouts, filter thresholds and sharded units.

Every case compares sites, alleles, totals and the matrices of the kept sites with the brute-force oracle
(orc_snp_discover, `check` of test_gpu_snp_discover), and the raw scan's counters -- timing()[5] covered windows,
[6] positions scanned, [13] (read, window) entries, [7] raw candidates -- with their exact mirror orc_disc_raw.  The
site oracle sees a raw scan that drops a read (a site at its threshold is lost); the mirror sees one that counts a
read twice or keeps a count from an earlier window (a candidate too many, an entry too many), which changes no
site.  Each case also asserts the route or edge it names."""

import gzip
import math
import os

import numpy as np
import pytest

import discover_oracle
from discover_oracle import orc_disc_raw, raw_counters
from recsets import CIGAR_PANEL, CODE, I, M, N, S, build, cell_keys, umi_keys
from test_gpu_baf_edges import WIDE, Conf, check_baf, exotic_batch
from test_gpu_snp_discover import check
from test_gpu_snp_pileup import oracle_snp, same
from xcltk_b200 import engine
from xcltk_b200.lib import XgError

pytestmark = pytest.mark.gpu

W = 2048                   # DISC_W of discover.cu: positions per raw-scan window
HIST_GRID = 148 * 5        # CTAs of k_disc_hist: more covered windows than this and CTAs take several in turn
KEY_NONE = 0xFFFFFFFFFFFFFFFF
XG_E_ARG = -1              # include/xcltk_b200.h


def thresholds(min_count, min_maf):
    """(t_sum, t_alt) of the raw pre-filter, computed as xg_snp_discover does (double product)."""
    t_sum = math.ceil(min_count) if min_count > 0 else 0
    t_alt = max(1, math.ceil(min_count * min_maf)) if min_count > 0 and min_maf > 0 else 1
    return t_sum, t_alt


def kept(c, min_count, min_maf):
    """The discovery filter on deduplicated counts c (A C G T N): ALT = second largest of A..T."""
    alt = sorted(c[:4])[2]
    s = sum(c)
    return alt >= 1 and not s < min_count and not alt < s * min_maf


def discover(ctx, reads, ck, n_cols, tg, conf=None, min_count=20, min_maf=0.1):
    """`check` (sites, totals, matrices, [14]) plus the raw counters against orc_disc_raw.  Returns (sites, timing)."""
    conf = conf or Conf()
    got, t = check(ctx, reads, ck, n_cols, tg, conf=conf, min_count=min_count, min_maf=min_maf)
    from oracle import oracle
    exp = orc_disc_raw(reads, *(np.asarray(x, np.int32) for x in tg), ck, oracle.params(conf), min_count, min_maf)
    assert raw_counters(t) == exp, (raw_counters(t), exp)
    assert t[14] == len(got["pos"])
    return got, t


class Rows(object):
    """Records collected one by one, then sorted by (run, pos) -- stably, so equal starts keep their order -- into
    one batch.  seq: letters of NT16, a code array, or None (no SEQ, then `end` is needed); ops None: one M block of
    len(seq) (or up to `end`).  cell: an index into the cell keys, umi: a molecule number (default: a new one per
    record); cell_key / umi_key give the raw key instead (unlisted, none, empty)."""

    def __init__(self):
        self.r = []

    def add(self, pos, seq, cell=0, umi=None, ops=None, flag=0, mapq=60, run=0, end=None, cell_key=None,
            umi_key=None):
        if isinstance(seq, str):
            seq = np.array([CODE[b] for b in seq], np.uint8)
        if umi_key is None:
            umi_key = int(umi_keys(1, salt=len(self.r) if umi is None else 1000000 + umi)[0])
        self.r.append(dict(pos=pos, seq=seq, cell=cell, cell_key=cell_key, umi_key=umi_key, ops=ops, flag=flag,
                           mapq=mapq, run=run, end=end))

    def site(self, p, counts, cell0=0, n_cells=50, L=20, back="C"):
        """One read per base of counts (A C G T N), each its own (cell, UMI): reads of L bases with the site at query
        index L // 2 and `back` elsewhere."""
        for b, k in zip("ACGTN", counts):
            for _ in range(k):
                s = back * (L // 2) + b + back * (L - L // 2 - 1)
                self.add(p - L // 2, s, cell=(cell0 + len(self.r)) % n_cells)

    def build(self, ck, runs=((0, 0),)):
        """runs: (bam_idx, gid) per run index used in add(run=...)."""
        rows = sorted(self.r, key=lambda x: (x["run"], x["pos"]))
        n = len(rows)
        pos = np.array([x["pos"] for x in rows], np.int64)
        ops = [x["ops"] for x in rows]
        end = np.array([x["end"] if x["end"] is not None else x["pos"] + len(x["seq"]) for x in rows], np.int64)
        cells = np.array([x["cell_key"] if x["cell_key"] is not None else int(ck[x["cell"]]) if ck is not None else 0
                          for x in rows], np.uint64)
        umis = np.array([x["umi_key"] for x in rows], np.uint64)
        out, at = [], 0
        for k, (bam, gid) in enumerate(runs):
            c = sum(1 for x in rows if x["run"] == k)
            out.append((bam, gid, at, at + c))
            at += c
        reads = build(pos, cells, umis, out, end=end, ops=ops if any(o is not None for o in ops) else None,
                      flag=np.array([x["flag"] for x in rows], np.uint32),
                      mapq=np.array([x["mapq"] for x in rows], np.uint32), seq=[x["seq"] for x in rows])
        for i, x in enumerate(rows):
            if x["flag"] & 4:                       # an unmapped record ends at pos + 1 whatever its CIGAR says
                reads.pos_end[i, 1] = x["pos"] + 1
            elif x["end"] is not None:
                reads.pos_end[i, 1] = x["end"]
        return reads


# ------------------------------------------------------------------------------------------ filter thresholds
THRESHOLDS = [(20, 0.1), (20, 0.25), (50, 0.3), (100, 0.07), (20.5, 0.1), (0, 0.0), (1000, 0.1)]


@pytest.mark.parametrize("mc,maf", THRESHOLDS, ids=["%s-%s" % x for x in THRESHOLDS])
def test_filter_thresholds_at_equality(gpu_ctx, mc, maf):
    """Sites at exactly sum = t_sum with ALT = t_alt, one below each, REF / ALT ties at the threshold and N bases
    that count in the sum only; every read its own passing UMI, so the raw counts are the deduplicated ones.
    (50, 0.3): the product is 15.0 in double (16 in single precision); (100, 0.07): 7.000000000000001, ALT 8."""
    t_sum, t_alt = thresholds(mc, maf)
    assert (mc, maf) != (50, 0.3) or t_alt == 15
    assert (mc, maf) != (100, 0.07) or t_alt == 8
    T, A = (max(t_sum, 2), t_alt) if t_sum <= 200 else (60, 6)      # min_count 1000: above every depth
    n_n = max(0, min(3, T - 2 * A - 1))
    designs = [                                         # (A, C, G, T, N)
        (T - A - n_n, 0, A, 0, n_n),                     # at both thresholds, with N in the sum
        (T - A, 0, A - 1, 0, 1),                         # ALT one below (the sum kept by an N)
        (T - A - 1, 0, A, 0, 0),                         # sum one below
        (A, 0, A, 0, T - 2 * A),                         # REF / ALT tie at the threshold: REF A, ALT G
        (T - 2 * A, A, A, 0, 0) if T >= 3 * A else (0, A, A, 0, T - 2 * A),     # ALT tie C / G: ALT is C
        (0, 0, 0, A, T - A),                             # one A..T bucket only: ALT 0
    ]
    rows = Rows()
    sites = []
    for k, c in enumerate(designs):
        if min(c) < 0:
            continue
        p = 1000 + 200 * k
        sites.append((p, c))
        rows.site(p, c)
    ck = cell_keys(50)
    reads = rows.build(ck)
    got, t = discover(gpu_ctx, reads, ck, 50, ([0], [0], [3000]), min_count=mc, min_maf=maf)
    want = [p for p, c in sites if kept(c, mc, maf)]
    assert got["pos"].tolist() == want
    cand = [p for p, c in sites if sum(c) >= t_sum and sorted(c[:4])[2] >= t_alt]
    assert t[7] == len(cand)                            # the background (C only) is never a candidate
    if mc <= 200:
        assert 1000 in want                              # the site at both thresholds is kept
    else:
        assert t[7] == 0 and not want
    for k, p in enumerate(got["pos"].tolist()):       # ties go to the lower index, for REF and for ALT
        c = dict(sites)[p][:4]
        r = c.index(max(c))
        a = max((x for x in range(4) if x != r), key=lambda x: (c[x], -x))
        assert (got["ref"][k], got["alt"][k]) == (r, a)
    assert mc > 200 or 1600 in want                     # REF / ALT tie


# ------------------------------------------------------------------------------------------ target layouts
def layout_batch():
    """Sites (18 A / 12 G, passing (20, 0.1)) at target edges, at windows edges relative to a target's beg and one
    base outside targets, on two contigs; reads of 40 bases at every start from site - 39 to site, so that reads
    straddle every edge and some end exactly at a window edge."""
    big = (1 << 20) + 5
    sites0 = [999, 1000, 1000 + W - 1, 1000 + W, 3070, 3071, 3072, 5000, big - 1, big, big + W, big + 4999, big + 5000]
    sites1 = [499, 500, 3000, 6999, 7000]
    rows = Rows()
    for run, sites in ((0, sites0), (1, sites1)):
        for p in sites:
            for k in range(30):
                s0 = p - 39 + (k * 39) // 29
                seq = ["T"] * 40
                seq[p - s0] = "A" if k % 5 < 3 else "G"
                rows.add(s0, "".join(seq), cell=k, run=run)
    ck = cell_keys(30)
    return rows.build(ck, runs=((0, 0), (0, 1))), ck, big


def test_target_layouts_caller_order_and_skipped_targets(gpu_ctx):
    """beg not a multiple of 2048 (1 000, 3 071, 2^20 + 5), a target of length 1, one ending mid-window, adjacent
    targets and gaps, contig 1 before contig 0, and skipped targets (gid -1, gid past the last contig, end <= beg)
    at the front, in the middle and at the end.  The sites follow caller order, then position; a site one base
    outside a target is never reported, the first and last base of a target are."""
    reads, ck, big = layout_batch()
    tg = ([-1, 1, 0, 0, 2, 0, 0, 0, 0, 0, 7],
          [0, 500, 3072, 4000, 0, 1000, 3071, big, 20000, 9000, 0],
          [100, 7000, 9000, 4000, 50, 3071, 3072, big + 5000, 10000, 9500, 10])
    got, t = discover(gpu_ctx, reads, ck, 30, tg)
    pos = got["pos"].tolist()
    order = list(zip(got["gid"].tolist(), pos))
    want = [(1, 500), (1, 3000), (1, 6999), (0, 3072), (0, 5000), (0, 1000), (0, 1000 + W - 1), (0, 1000 + W),
            (0, 3070), (0, 3071), (0, big), (0, big + W), (0, big + 4999)]
    assert order == want
    for x in ((0, 999), (0, big - 1), (0, big + 5000), (1, 499), (1, 7000)):
        assert x not in order
    # covered windows: [500, 7000) 3 of 4, [3072, 9000) 1 of 3, [1000, 3071) 2 (the second ends mid-window),
    # [3071, 3072) 1, [2^20 + 5, +5000) 3 of 3, [9000, 9500) none
    assert t[5] == 10


def test_target_per_window_edge_entries(gpu_ctx):
    """Many adjacent targets of 2 049 positions from 1 000, like the sharded units: reads end exactly at a window
    edge relative to a target's beg (3 048) and cross target edges; every (read, window) entry counted once, which
    [13] shows against the mirror.  The same targets shuffled, with skipped empties, give the same counters."""
    reads, ck, big = layout_batch()
    beg = 1000 + np.arange(6) * (W + 1)
    tg0 = (np.zeros(len(beg), np.int32), beg, beg + W + 1)
    got, t = discover(gpu_ctx, reads, ck, 30, tg0)
    assert {1000, 1000 + W, 3070, 3071, 3072, 5000} <= set(got["pos"].tolist())
    rng = np.random.RandomState(1)
    perm = rng.permutation(len(beg))
    tg1 = (np.concatenate([tg0[0][perm], [0, 0]]), np.concatenate([tg0[1][perm], [5, 7]]),
           np.concatenate([tg0[2][perm], [5, 3]]))
    got1, t1 = discover(gpu_ctx, reads, ck, 30, tg1)
    assert sorted(got1["pos"].tolist()) == sorted(got["pos"].tolist())
    assert raw_counters(t1) == raw_counters(t)


# ------------------------------------------------------------------------------------------ CIGARs in the raw scan
def test_cigar_panel_and_301_op_read_at_window_edges(gpu_ctx):
    """The CIGAR panel (S / H / = / X / D / N / P / I / zero-length M) and the 301-op read twice: at their own
    place and moved so that they cross the window edge 2047 / 2048.  Filler reads carry A everywhere, so a
    position is a candidate where a panel read's aligned base is not A: a misplaced query offset after I / S shows
    as a different candidate count."""
    rows = Rows()
    panel = CIGAR_PANEL + [WIDE]
    for shift in (0, 1938):                             # R0's I sits on the window edge 2 047 / 2 048
        for k, (_lab, p, ops, s) in enumerate(panel):
            q = len(s) if ops is None else None
            rows.add(p + shift, s, cell=k, ops=ops, end=(p + shift + q) if q else None)
        for j in range(12):                             # A-only filler over the panel
            rows.add(90 + shift + 15 * j, "A" * 120, cell=10 + j)
    ck = cell_keys(30)
    reads = rows.build(ck)
    for mc, maf in ((0, 0.0), (2, 0.1)):
        got, t = discover(gpu_ctx, reads, ck, 30, ([0], [0], [5000]), min_count=mc, min_maf=maf)
        assert t[7] > 20 and (mc > 0 or len(got["pos"]) > 20)
    assert t[5] == 2                                   # windows 0 and 1: the moved copy crosses 2 048


def test_random_exotic_cigars(gpu_ctx):
    """5 000 reads of random exotic CIGARs (I / D / N / S / H / P / = / X, 281-op reads) over 20 kb."""
    reads, ck = exotic_batch(31, 5000, 20000, 30, 300, True)
    for mc, maf in ((2, 0.1), (4, 0.3)):
        got, t = discover(gpu_ctx, reads, ck, 30, ([0, 0], [0, 9000], [8500, 21000]), min_count=mc, min_maf=maf)
        assert len(got["pos"]) > 100 and t[5] == 11


def test_long_blocks_gaps_and_reads_without_bases(gpu_ctx):
    """One aligned block of 5 000 bases over three windows; an N gap that skips whole windows (not covered: [5] and
    [6]); reads without an aligned base (all S, all I) under min_len 0 that claim their UMI with a None allele;
    unmapped-flag reads with excl_flag 0 (they end at pos + 1 but their blocks are walked by the raw scan); SEQ-less
    first reads of a UMI."""
    rows = Rows()
    rows.add(2148, "A" * 2500 + "G" + "A" * 2499, cell=0)            # 2 148 .. 7 148: windows 1, 2, 3
    rows.add(2148, "A" * 5000, cell=1)
    rows.add(20000, "A" * 50 + "C" * 50, cell=2, ops=[(M, 50), (N, 40000), (M, 50)])   # windows 9 and 29 only
    site = 100000
    rows.site(site, (14, 0, 6, 0, 0))
    rows.site(site + 500, (14, 0, 6, 0, 0))
    uid = 5000
    # claimers: all-S / all-I / no-SEQ first reads of three UMIs whose second read carries G at the site
    for k, (ops, seq) in enumerate([([(S, 30)], "A" * 30), ([(I, 30)], "A" * 30), (None, None)]):
        u = uid + k
        if seq is None:
            rows.add(site, None, cell=40 + k, umi=u, end=site + 20)
        else:
            rows.add(site, seq, cell=40 + k, umi=u, ops=ops)
        rows.add(site, "G" + "C" * 19, cell=40 + k, umi=u)
    # unmapped reads: each claims its UMI at its pos only, the raw scan counts all of its block
    for k in range(6):
        rows.add(site + 500 - 3, "CCCG" + "C" * 36, cell=45 + k, umi=uid + 10 + k, flag=4)
    ck = cell_keys(60)
    reads = rows.build(ck)
    conf = Conf(min_len=0)
    tg = ([0], [0], [200000])
    got, t = discover(gpu_ctx, reads, ck, 60, tg, conf=conf, min_count=2, min_maf=0.1)
    g = {p: list(c) for p, c in zip(got["pos"].tolist(), got["totals"])}
    assert g[2148 + 2500] == [1, 0, 1, 0, 0]
    assert g[site] == [14, 0, 6, 0, 0]                  # the claimers' later G reads do not count
    assert t[5] == len({1, 2, 3, 9, 29, site // W, (site + 500) // W}) == 7     # windows 10 .. 28 are not covered
    assert t[6] == 7 * W


# ------------------------------------------------------------------------------------------ read filters
def test_read_filters_at_their_edges(gpu_ctx):
    """Threshold sites (sum 20, ALT 2 under (20, 0.1)) whose passing reads sit at a filter's edge: mapq = min_mapq
    (and a float min_mapq), aligned length = min_len for simple and CIGAR reads, incl_flag / excl_flag bits, paired
    reads that are not orphans.  A raw filter stricter than the pileup's loses the site.  Failing reads (orphans,
    excluded flags, mapq below, short, unlisted cells, missing cell keys, none / empty UMIs) carry a third base at
    sites just below the threshold: a raw filter looser than the pileup's makes them candidates."""
    conf = Conf(min_mapq=20.5, min_len=30, incl_flag=2, excl_flag=1024, no_orphan=True)
    rows = Rows()
    ok = dict(flag=3, mapq=21)
    edge = [dict(mapq=21), dict(seq30=True), dict(cig30=True), dict(flag=2), dict(flag=3 | 16)]
    for k, e in enumerate(edge):
        p = 1000 + 300 * k
        for j in range(20):
            b = "G" if j >= 18 else "A"
            kw = dict(ok)
            if j in (0, 18):                          # the edge read: one REF, one ALT
                kw.update(e)
            if kw.pop("seq30", False):
                rows.add(p - 10, "C" * 10 + b + "C" * 19, cell=j, **kw)
            elif kw.pop("cig30", False):
                rows.add(p - 10, "TTTTT" + "C" * 10 + b + "C" * 19 + "TT", cell=j, ops=[(S, 5), (M, 10), (I, 0),
                                                                                          (M, 20), (S, 2)], **kw)
            else:
                rows.add(p - 10, "C" * 10 + b + "C" * 29, cell=j, **kw)
    bad = [dict(flag=1), dict(flag=3 | 1024), dict(flag=0), dict(mapq=20), dict(short=True), dict(cell_key=1 << 40),
           dict(cell_key=KEY_NONE), dict(umi_key=KEY_NONE), dict(umi_key=0)]
    for k, e in enumerate(bad):
        p = 3000 + 300 * k
        for j in range(19):
            b = "A" if j < 17 else "G"
            rows.add(p - 10, "C" * 10 + b + "C" * 29, cell=j, **ok)
        kw = dict(ok)
        kw.update(e)
        short = kw.pop("short", False)
        rows.add(p - 10, "C" * 10 + "T" + "C" * (18 if short else 29), cell=30, **kw)
    ck = cell_keys(31)
    reads = rows.build(ck)
    got, t = discover(gpu_ctx, reads, ck, 31, ([0], [0], [10000]), conf=conf)
    assert got["pos"].tolist() == [1000 + 300 * k for k in range(len(edge))]
    assert t[7] == len(edge)


def test_sample_mode_three_bams(gpu_ctx):
    """Sample-ID mode with three BAMs: one UMI key in every BAM is three molecules (column = BAM)."""
    rows = Rows()
    for run in range(3):
        for j in range(7):
            rows.add(990, "C" * 10 + ("G" if j == 0 and run < 2 else "A") + "C" * 9, umi=j, run=run)
    rows.site(1500, (8, 0, 0, 2, 0))
    reads = rows.build(None, runs=((0, 0), (1, 0), (2, 0)))
    conf = Conf(barcodes=False)
    got, t = discover(gpu_ctx, reads, None, 3, ([0], [0], [3000]), conf=conf, min_count=21, min_maf=0.09)
    assert got["pos"].tolist() == [1000] and got["totals"][0].tolist() == [19, 0, 2, 0, 0]


# ------------------------------------------------------------------------------------------ persistent CTAs
def test_persistent_ctas_many_windows(gpu_ctx):
    """1 600 covered windows (more than the 740 CTAs of k_disc_hist), dense windows of 300 reads (more than 8 x 32)
    next to sparse ones, under (2, 0.1): a count left from a CTA's previous window would be an extra candidate."""
    rng = np.random.RandomState(17)
    n_win = 1600
    dense = rng.rand(n_win) < 0.15
    starts = []
    for w in range(n_win):
        k = 300 if dense[w] else int(rng.randint(1, 4))
        starts.append(w * W + rng.randint(0, W - 60, size=k))
    pos = np.sort(np.concatenate(starts))
    n, L = len(pos), 60
    ref = rng.choice([1, 2, 4, 8], size=n_win * W + L).astype(np.uint8)
    seq = ref[pos[:, None] + np.arange(L)]
    het = rng.rand(n, L) < 0.05
    seq[het] = rng.choice([1, 2, 4, 8, 15], size=int(het.sum()))
    ck = cell_keys(100)
    reads = build(pos, ck[rng.randint(0, 100, size=n)], umi_keys(n), [(0, 0, 0, n)], end=pos + L, seq=seq)
    got, t = discover(gpu_ctx, reads, ck, 100, ([0], [0], [n_win * W]), min_count=2, min_maf=0.1)
    assert t[5] == n_win > 2 * HIST_GRID and len(got["pos"]) > 1000


# ------------------------------------------------------------------------------------------ calls on one context
def test_calls_on_one_context(gpu_ctx):
    """snp_pileup, discovery with every candidate its own pileup slice (the SNP table re-keyed each time), baf_fc,
    discovery again: each against the oracle."""
    rows = Rows()
    for k, c in enumerate([(15, 0, 5, 0, 0), (10, 10, 0, 0, 0), (19, 1, 0, 0, 0), (12, 0, 0, 8, 2)]):
        rows.site(1000 + 100 * k, c)
    ck = cell_keys(50)
    reads = rows.build(ck)
    snp_pos = np.array([1000, 1100, 1200, 1300], np.int32)
    ref, alt = np.array([0, 0, 0, 0], np.uint8), np.array([2, 1, 1, 3], np.uint8)
    conf = Conf()
    params = engine.make_params(conf, reads.max_aln_len, with_include=False)
    d = gpu_ctx.upload(reads)
    try:
        got = gpu_ctx.snp_pileup(d, np.zeros(4, np.int32), snp_pos, ck, 50, params, ref, alt, 0, 0.0)
        same(got, oracle_snp(reads, np.zeros(4, np.int32), snp_pos, ref, alt, ck, 50, conf, 0, 0.0), "snp_pileup")
    finally:
        d.close()
    try:
        gpu_ctx.set_option("discover_slice", 1)
        a, t = discover(gpu_ctx, reads, ck, 50, ([0], [0], [2000]), min_count=2, min_maf=0.1)
        assert t[11] == t[7] == 4 and a["pos"].tolist() == [1000, 1100, 1300]    # 1200: ALT 1 < 20 * 0.1
    finally:
        gpu_ctx.set_option("discover_slice", 0)
    check_baf(gpu_ctx, reads, ck, 50, snp_pos, ref, alt, [[0, 1], [2, 3]])
    b, t = discover(gpu_ctx, reads, ck, 50, ([0], [0], [2000]), min_count=2, min_maf=0.1)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert t[11] == 1


# ------------------------------------------------------------------------------------------ errors
def test_argument_errors_leave_the_context_usable(gpu_ctx):
    """Overlapping targets (one nested), reads without sequences, 2^24 columns, a barcode-key count that is not the
    number of columns, more BAMs than sample columns: XG_E_ARG, and the next call still matches the oracle."""
    rows = Rows()
    rows.site(1000, (15, 0, 5, 0, 0))
    ck = cell_keys(50)
    reads = rows.build(ck)
    bare = build(np.array([990, 995], np.int64), ck[:2], umi_keys(2), [(0, 0, 0, 2)], end=np.array([1010, 1015]))
    rows3 = Rows()
    for run in range(3):
        rows3.add(990, "C" * 20, umi=1, run=run)
    three = rows3.build(None, runs=((0, 0), (1, 0), (2, 0)))
    conf, sconf = Conf(), Conf(barcodes=False)
    p = engine.make_params(conf, 40, with_include=False)
    sp = engine.make_params(sconf, 40, with_include=False)
    calls = [(reads, ([0, 0], [0, 500], [1000, 1500]), ck, 50, p), (reads, ([0, 0], [0, 100], [3000, 200]), ck, 50, p),
             (bare, ([0], [0], [2000]), ck, 50, p), (reads, ([0], [0], [2000]), None, 1 << 24, sp),
             (reads, ([0], [0], [2000]), ck[:49], 50, p), (three, ([0], [0], [2000]), None, 2, sp)]
    for r, tg, keys, n_cols, par in calls:
        d = gpu_ctx.upload(r)
        try:
            with pytest.raises(XgError) as e:
                gpu_ctx.snp_discover(d, *tg, keys, n_cols, par, 20, 0.1)
            assert e.value.code == XG_E_ARG
        finally:
            d.close()
        got, _ = discover(gpu_ctx, reads, ck, 50, ([0], [0], [2000]))
        assert got["pos"].tolist() == [1000]


# ------------------------------------------------------------------------------------------ sharded discovery
def test_sharded_discovery_at_unit_edges(gpu_ctx, tmp_path, monkeypatch):
    """3M reads over two contigs of about 4 Mb with SNPs planted at every unit edge k * 2^20 - 1 and k * 2^20 plus
    random ones, written as a BAM: pileup_wrapper without candidates on one GPU and on 3 and 6 emulated shards
    gives the same bytes, the oracle's sites over whole contigs, no site twice and every deep enough planted edge
    SNP; --chrom in reverse BAM order gives the same sites with the VCF in that order."""
    from oracle import oracle
    from xcltk_b200 import lib
    from xcltk_b200.baf.pileup import DISCOVER_UNIT, pileup_wrapper
    lens = [4 * DISCOVER_UNIT + 3000, 4 * DISCOVER_UNIT - 7]
    names = ["chr21", "chr22"]
    rng = np.random.RandomState(23)
    sg, sp, edge = [], [], []
    for g, ln in enumerate(lens):
        edges = [e for k in range(1, 5) for e in (k * DISCOVER_UNIT - 1, k * DISCOVER_UNIT) if e < ln - 200]
        edge += [(names[g], e + 1) for e in edges]
        rand = rng.choice(np.arange(200, ln - 200), 150, replace=False)
        p = np.unique(np.concatenate([edges, rand]))
        sg += [g] * len(p)
        sp += p.tolist()
    sg, sp = np.array(sg, np.int32), np.array(sp, np.int32)
    n_snp = len(sp)
    sref = rng.randint(0, 4, n_snp).astype(np.uint8)
    salt = ((sref + 1 + rng.randint(0, 3, n_snp)) % 4).astype(np.uint8)
    snps = (sg, sp, sref, salt, rng.randint(0, 2, n_snp).astype(np.uint8))
    n_cells = 500
    d, bk = gpu_ctx.synth_reads(3000000, n_cells, [0, 1], [0, 0], lens, seed=31, want_seq=True, snps=snps,
                                ref_error=0.001)
    try:
        host = d.download()
    finally:
        d.close()
    bam = str(tmp_path / "lib.bam")
    lib.write_bam(bam, host, list(zip(names, lens)), None, "CB", "UB", level=1, n_threads=4)
    ks = lib.KeySpace()
    bc = str(tmp_path / "bc.tsv")
    open(bc, "w").write("".join(ks.decode(int(k)) + "\n" for k in bk))
    conf = Conf(min_mapq=20, min_len=30, excl_flag=772, no_orphan=True)
    exp = discover_oracle.orc_snp_discover(host, [0, 1], [0, 0], lens, bk, oracle.params(conf), 20, 0.1)
    host.close()
    runs = {}
    for label, gpus, chrom in (("one", None, "21,22"), ("three", "3", "21,22"), ("six", "6", "21,22"),
                               ("rev", "3", "22,21")):
        with monkeypatch.context() as mp:
            if gpus:
                mp.setenv("XCLTK_B200_GPUS", gpus)
                mp.setenv("XCLTK_B200_EMULATE_SHARDS", "1")
            out = str(tmp_path / label)
            assert pileup_wrapper(bam, bc, None, out, ncores=4, chrom=chrom) == 0
        runs[label] = {f: open(os.path.join(out, f), "rb").read() for f in sorted(os.listdir(out))}
    assert runs["one"] == runs["three"] == runs["six"]
    vcf = [x.split("\t") for x in gzip.decompress(runs["one"]["cellSNP.base.vcf.gz"]).decode().splitlines()[2:]]
    got = [(x[0], int(x[1]), x[3], x[4]) for x in vcf]
    assert len(set(got)) == len(got) > 100
    want = [(names[g], p + 1, "ACGT"[r], "ACGT"[a]) for g, p, r, a in zip(exp["gid"], exp["pos"], exp["ref"],
                                                                          exp["alt"])]
    assert got == want
    for x, tot, r, a in zip(vcf, exp["totals"], exp["ref"], exp["alt"]):
        assert x[7] == "AD=%d;DP=%d;OTH=%d" % (tot[a], tot[a] + tot[r], tot.sum() - tot[a] - tot[r])
    # the planted edge SNPs: both sides of every unit edge (8 on the first contig, 6 on the second, whose last unit
    # is short); those with enough depth are found
    found = set((x[0], int(x[1])) for x in vcf)
    assert len(edge) == 14 and sum(e in found for e in edge) >= 10
    rev = [x.split("\t") for x in gzip.decompress(runs["rev"]["cellSNP.base.vcf.gz"]).decode().splitlines()[2:]]
    revs = [(x[0], int(x[1]), x[3], x[4]) for x in rev]
    assert sorted(revs) == sorted(got)
    assert revs == [s for s in got if s[0] == "chr22"] + [s for s in got if s[0] == "chr21"]
