"""SNP-level counting (xg_snp_pileup / Context.snp_pileup / pileup_wrapper) against the CPU oracle.

The oracle is oracle.baf with one region per SNP and GT 0|1 (reg_ptr = arange(n + 1), reg_snp = arange(n),
ref_idx 0, alt_idx 1): AD = UMIs with the ALT base, DP = UMIs with REF or ALT, OTH = the others.  Every hand-built
case runs on an uploaded batch and on the same records mapped from pinned host memory (xg_map_reads), and is also
compared with baf_fc on one region per SNP.  Cases that name a branch of k_snp_finalize assert it through
timing()[14] (SNPs reduced by one warp) and [15] (by a whole CTA)."""

import gzip
import logging
import os

import numpy as np
import pytest
import scipy.io
import scipy.sparse

from recsets import D, M, build, cell_keys, umi_keys
from test_gpu_baf_edges import Conf, contention_batch, entries, exotic_batch, random_codes
from xcltk_b200 import engine

pytestmark = pytest.mark.gpu
logging.disable(logging.CRITICAL)

LETTERS = "ACGTN"
WARP_MAX = 128                 # SNP_WARP_MAX of baf.cu: winners a warp reduces
HIST_COLS = 4096               # SNP_HIST_COLS of baf.cu: cells per column range of the CTA path
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def one_region_per_snp(n):
    return np.arange(n + 1, dtype=np.int64), np.arange(n, dtype=np.int32)


def hap_01(ref, alt):
    """hap_of of GT 0|1: REF -> haplotype 0, ALT -> 1 (written second: ALT wins when REF == ALT, as SNP.gt)."""
    n = len(ref)
    hap = np.full((n, 8), 2, np.uint8)
    hap[np.arange(n), ref] = 0
    hap[np.arange(n), alt] = 1
    return hap


def oracle_snp(host, snp_gid, snp_pos, ref, alt, ck, n_cols, conf, min_count, min_maf):
    from oracle import oracle
    n = len(snp_pos)
    reg_ptr, reg_snp = one_region_per_snp(n)
    return oracle.baf(host, snp_gid, snp_pos, "".join(LETTERS[x] for x in ref), "".join(LETTERS[x] for x in alt),
                      np.zeros(n, np.int8), np.ones(n, np.int8), reg_ptr, reg_snp, ck, n_cols, oracle.params(conf),
                      min_count, min_maf, True, 4)


def same(got, exp, what):
    for name, g, e in zip(("AD", "DP", "OTH"), got, exp):
        for k in range(3):
            assert np.array_equal(np.asarray(g[k]), np.asarray(e[k])), (what, name, k)


def check_snp(ctx, reads, ck, n_cols, snp_pos, ref, alt, conf=None, min_count=0, min_maf=0.0, snp_gid=None,
              zero_copy=True):
    """Returns ((AD, DP, OTH), timing(), keep, totals) of snp_pileup on the uploaded batch, after asserting that the
    oracle, baf_fc with one region per SNP and the zero-copy batch give the same."""
    conf = conf or Conf()
    ref, alt = np.asarray(ref, np.uint8), np.asarray(alt, np.uint8)
    snp_pos = np.asarray(snp_pos, np.int32)
    n = len(snp_pos)
    snp_gid = np.zeros(n, np.int32) if snp_gid is None else np.asarray(snp_gid, np.int32)
    params = engine.make_params(conf, reads.max_aln_len, with_include=False)
    exp = oracle_snp(reads, snp_gid, snp_pos, ref, alt, ck, n_cols, conf, min_count, min_maf)
    d = ctx.upload(reads)
    try:
        ad, dp, oth, totals, keep = ctx.snp_pileup(d, snp_gid, snp_pos, ck, n_cols, params, ref, alt, min_count, min_maf,
                                                   want_totals=True, want_keep=True)
        t = ctx.timing()
        got = (ad, dp, oth)
        same(got, exp, "snp_pileup")
        reg_ptr, reg_snp = one_region_per_snp(n)
        fc = ctx.baf_fc(d, snp_gid, snp_pos, ck, n_cols, params, ref, alt, min_count, min_maf, reg_ptr, reg_snp,
                        hap_01(ref, alt), True, want_totals=True, want_keep=True)
        same(fc[:3], exp, "baf_fc")
        assert np.array_equal(fc[3], totals) and np.array_equal(fc[4], keep)
        for m in got:                                            # a SNP removed by the filter has empty rows
            assert not np.any(keep[np.asarray(m[0], np.int64)] == 0)
        if zero_copy:
            host = d.download()
            mapped = ctx.map_reads(host)
            try:
                zc = ctx.snp_pileup(mapped, snp_gid, snp_pos, ck, n_cols, params, ref, alt, min_count, min_maf)
                same(zc, exp, "zero-copy")
            finally:
                mapped.close()
                host.close()
    finally:
        d.close()
    return got, t, keep, totals


# ------------------------------------------------------------------------------------------ first read wins
@pytest.mark.parametrize("case", ["deletion", "refskip", "mapq", "flag", "min_len", "N", "eq", "iupac", "two_bams"])
def test_first_read_wins(gpu_ctx, case):
    """One (cell, UMI) in 3 000 reads over SNP 0: its first read has a D / N over the SNP (allele None: claims the
    UMI, counts nowhere), fails a filter (claims nothing), carries N, '=' or an IUPAC code (OTH); or the molecule
    is in two BAMs (sample-ID mode, one column each)."""
    reads, ck, n_cols, conf = contention_batch(case)
    got, _, _, _ = check_snp(gpu_ctx, reads, ck, n_cols, [5000, 4970, 5015], [0, 0, 1], [2, 2, 3], conf=conf)
    ad, dp, oth = (entries(m, row=0) for m in got)
    if case == "two_bams":                                      # each BAM's first read: A in column 0, G in column 1
        assert ad == {(0, 1): 1} and dp == {(0, 0): 1, (0, 1): 1} and oth == {}
        return
    c0 = [{k: v for k, v in m.items() if k[1] == 0} for m in (ad, dp, oth)]
    if case in ("deletion", "refskip"):
        assert c0 == [{}, {}, {}]
    elif case in ("mapq", "flag", "min_len"):                   # the second read (G = ALT) wins
        assert c0 == [{(0, 0): 1}, {(0, 0): 1}, {}]
    else:
        assert c0 == [{}, {}, {(0, 0): 1}]
    assert len(dp) > 3


# ------------------------------------------------------------------------------------------ alleles and SNP tables
def test_alleles_and_snp_table_edges(gpu_ctx):
    """Reads with every base class (A C G T, N, '=', IUPAC) under SNPs with REF == ALT, REF N, ALT N, duplicate
    positions, SNPs on an unknown contig (gid -1, or a contig with no reads) and at 0-based pos < 0; the exotic
    CIGARs put I / D / N / S next to the SNPs."""
    rng = np.random.RandomState(3)
    n, L = 3000, 60                                             # ~60 reads per SNP: all on the warp path
    pos = np.sort(rng.randint(0, 3000, size=n))
    codes = rng.choice([1, 2, 4, 8, 15, 0, 5, 10], p=[.2, .2, .2, .2, .08, .04, .04, .04], size=(n, L)).astype(np.uint8)
    ck = cell_keys(40)
    reads = build(pos, ck[rng.randint(0, 40, size=n)], umi_keys(60)[rng.randint(0, 60, size=n)], [(0, 0, 0, n)],
                  end=pos + L, seq=codes)
    k = 400
    snp_pos = np.sort(rng.randint(0, 3050, size=k)).astype(np.int32)
    snp_pos[10:20] = snp_pos[10]                                # duplicate positions
    ref = rng.randint(0, 5, size=k)
    alt = rng.randint(0, 5, size=k)
    ref[20:40] = alt[20:40]                                     # REF == ALT (ALT wins)
    ref[40:60], alt[60:80] = 4, 4                               # REF N, ALT N
    gid = np.zeros(k, np.int32)
    gid[80:85], gid[85:90] = -1, 3                              # unknown contigs
    snp_pos[90:95] = -1
    got, t, keep, totals = check_snp(gpu_ctx, reads, ck, 40, snp_pos, ref, alt, snp_gid=gid)
    ad, dp, oth = got
    assert keep.all()                                           # the default filter (0, 0) keeps every SNP
    assert not np.isin(np.arange(80, 95), np.concatenate([dp[0], oth[0]])).any()
    rows = lambda m, a, b: np.asarray(m[0])[(np.asarray(m[0]) >= a) & (np.asarray(m[0]) < b)]
    assert len(rows(ad, 20, 40)) and np.array_equal(np.unique(rows(ad, 20, 40)), np.unique(rows(dp, 20, 40)))
    assert len(rows(dp, 40, 80)) and len(rows(oth, 0, 400)) > 100
    assert t[7] == totals.sum() and t[14] > 300 and t[15] == 0
    reads, ck = exotic_batch(11, 3000, 4000, 20, 30, True)
    snp_pos = np.arange(0, 4200, 3)
    ref = rng.randint(0, 4, size=len(snp_pos))
    check_snp(gpu_ctx, reads, ck, 20, snp_pos, ref, (ref + rng.randint(1, 4, size=len(snp_pos))) % 4)


# ------------------------------------------------------------------------------------------ k_snp_finalize paths
def covering(rng, snp, n_win, n_none, cells, ck, umi_base):
    """n_win reads with an allele at `snp`, then n_none reads with a D over it; distinct UMIs, the cells taken from
    `cells` in turn (every listed cell is covered when n_win >= len(cells))."""
    n = n_win + n_none
    pos = np.full(n, snp - 20, np.int64)
    ops = [None] * n_win + [[(M, 20), (D, 5), (M, 20)]] * n_none
    seq = [random_codes(rng, 40 if o else 45) for o in ops]
    return pos, ck[np.resize(cells, n)], umi_keys(n, salt=umi_base), ops, seq


def path_batch(n_cols, groups, seed):
    """groups: [(snp, winners, None-winners, cells)] -> one batch over contig 0, SNP positions."""
    rng = np.random.RandomState(seed)
    ck = cell_keys(n_cols)
    parts = [covering(rng, s, w, z, cells, ck, 1 + g) for g, (s, w, z, cells) in enumerate(groups)]
    pos = np.concatenate([p[0] for p in parts])
    reads = build(pos, np.concatenate([p[1] for p in parts]), np.concatenate([p[2] for p in parts]),
                  [(0, 0, 0, len(pos))], ops=sum([p[3] for p in parts], []), seq=sum([p[4] for p in parts], []),
                  end=pos + 45)
    return reads, ck, [g[0] for g in groups]


def test_finalize_warp_and_cta_paths_at_the_threshold(gpu_ctx):
    """SNPs with WARP_MAX and WARP_MAX + 1 winners (a few cells, so columns repeat with mixed classes), one covered
    by None alleles only, one by nothing."""
    few = np.arange(7)
    groups = [(1000, WARP_MAX, 30, few), (2000, WARP_MAX + 1, 0, few), (3000, 0, 200, few), (4000, 1, 0, few)]
    reads, ck, snp_pos = path_batch(50, groups, 1)
    snp_pos.append(5000)                                       # no read
    rng = np.random.RandomState(2)
    ref = rng.randint(0, 4, size=len(snp_pos))
    got, t, _, totals = check_snp(gpu_ctx, reads, ck, 50, snp_pos, ref, (ref + 1) % 4)
    assert (t[14], t[15]) == (2, 1)                            # SNPs 0 and 3 by a warp, SNP 1 by the CTA
    assert t[7] == 2 * WARP_MAX + 2 and totals[2].sum() == 0
    rows = [set(np.asarray(m[0]).tolist()) for m in got]
    assert {0, 1} <= rows[1] | rows[2] and not (2 in rows[0] | rows[1] | rows[2] or 4 in rows[0] | rows[1] | rows[2])


@pytest.mark.parametrize("n_cols", [HIST_COLS, HIST_COLS + 1, 40000])
def test_finalize_cta_path_column_ranges(gpu_ctx, n_cols):
    """A SNP covered by thousands of cells, with cells on both sides of every column-range edge."""
    edges = sorted({c for k in range(1, 10) for c in (k * HIST_COLS - 1, k * HIST_COLS) if c < n_cols} |
                   {0, n_cols - 1})
    rng = np.random.RandomState(n_cols)
    cells = np.concatenate([np.repeat(edges, 3), rng.randint(0, n_cols, size=6000)])
    reads, ck, snp_pos = path_batch(n_cols, [(1000, len(cells), 100, cells), (2000, 40, 5, cells[:50])], 4)
    got, t, _, _ = check_snp(gpu_ctx, reads, ck, n_cols, snp_pos, [0, 1], [2, 3])
    assert (t[14], t[15]) == (1, 1)
    cols = set(np.concatenate([np.asarray(m[1])[np.asarray(m[0]) == 0] for m in got]).tolist())
    assert set(edges) <= cols and len(cols) > 2000


def test_nothing_covered_and_empty_batch(gpu_ctx):
    from xcltk_b200 import lib
    rng = np.random.RandomState(5)
    pos = np.sort(rng.randint(0, 1000, size=500))
    ck = cell_keys(10)
    reads = build(pos, ck[rng.randint(0, 10, size=500)], umi_keys(500), [(0, 0, 0, 500)], end=pos + 50,
                  seq=random_codes(rng, 500 * 50).reshape(500, 50))
    got, t, _, _ = check_snp(gpu_ctx, reads, ck, 10, [5000, 6000], [0, 1], [1, 2])
    assert all(len(m[2]) == 0 for m in got) and t[7] == 0 and t[14] == t[15] == 0
    z = np.zeros(0, np.uint32)
    empty = lib.ArrayReads(np.zeros((0, 2), np.int32), z, np.zeros(1, np.uint32), np.zeros((0, 2), np.uint64),
                           np.zeros(1, np.uint32), [], z, np.zeros(1, np.uint32), max_aln_len=1, max_span=1)
    got, t, _, _ = check_snp(gpu_ctx, empty, ck, 10, [5000, 6000], [0, 1], [1, 2], zero_copy=False)
    assert all(len(m[2]) == 0 and m[3] == (2, 10) for m in got) and t[6] == 0
    got, _, _, _ = check_snp(gpu_ctx, empty, ck, 10, [], [], [], zero_copy=False)
    assert all(m[3] == (0, 10) for m in got)


# ------------------------------------------------------------------------------------------ filter
@pytest.mark.parametrize("min_count,min_maf", [(3, 0.1), (2, 0.3), (1, 1.0 / 3), (0, 0.7), (10 ** 6, 0.0)])
def test_filter(gpu_ctx, min_count, min_maf):
    """Thresholds that float cannot represent exactly (0.1, 0.3, 1/3); and one that removes every SNP."""
    rng = np.random.RandomState(9)
    n, L = 20000, 40
    pos = np.sort(rng.randint(0, 5000, size=n))
    ck = cell_keys(30)
    reads = build(pos, ck[rng.randint(0, 30, size=n)], umi_keys(20)[rng.randint(0, 20, size=n)], [(0, 0, 0, n)],
                  end=pos + L, seq=rng.choice([1, 2], size=(n, L)).astype(np.uint8))       # only A and C
    snp_pos = np.arange(0, 5100, 4)
    ref, alt = np.zeros(len(snp_pos), np.uint8), np.ones(len(snp_pos), np.uint8)
    got, _, keep, totals = check_snp(gpu_ctx, reads, ck, 30, snp_pos, ref, alt, min_count=min_count, min_maf=min_maf)
    cnt = totals.sum(axis=1)
    assert np.array_equal(keep, ((cnt >= min_count) & ~(np.minimum(totals[:, 0], totals[:, 1]) < cnt * min_maf)))
    if min_count == 10 ** 6:
        assert not keep.any() and all(len(m[2]) == 0 for m in got)
    else:
        assert 0 < keep.sum() < len(keep) or min_count == 0


# ------------------------------------------------------------------------------------------ bench-shaped batch
def test_snp_pileup_equals_baf_fc_on_a_synthetic_library(gpu_ctx):
    from xcltk_b200 import workload
    b = workload.make_baf_workload(gpu_ctx, 3000000, 2000, 60000, seed=17, chroms={"19", "20", "21", "22"})
    try:
        n = len(b.snp_pos)
        reg_ptr, reg_snp = one_region_per_snp(n)
        for mc, mm in ((0, 0.0), (2, 0.1)):
            sp = gpu_ctx.snp_pileup(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 2000, b.params, b.snp_ref, b.snp_alt,
                                    mc, mm, want_keep=True)
            t = gpu_ctx.timing()
            fc = gpu_ctx.baf_fc(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 2000, b.params, b.snp_ref, b.snp_alt, mc,
                                mm, reg_ptr, reg_snp, hap_01(b.snp_ref, b.snp_alt), True, want_keep=True)
            same(sp[:3], fc[:3], (mc, mm))
            assert np.array_equal(sp[3], fc[3])
            assert len(sp[1][2]) > 20000 and t[14] > 1000
    finally:
        b.dreads.close()


# ------------------------------------------------------------------------------------------ end to end
def golden_inputs(name):
    g = os.path.join(GOLD, name)
    if name == "c1_chr22_10x":
        return dict(sam=os.path.join(g, "a.bam"), barcodes=os.path.join(g, "barcodes.tsv"),
                    snps=os.path.join(g, "snps.tsv"), features=os.path.join(g, "features.tsv"),
                    kw=dict(cell_tag="CB", umi_tag="UB"))
    return dict(sam=os.path.join(g, "BCH869.output.bam"), barcodes=os.path.join(g, "barcodes.tsv"),
                snps=os.path.join(g, "snps.tsv"), features=os.path.join(g, "features.tsv.gz"),
                kw=dict(cell_tag="RG", umi_tag=None))


def oracle_dir(r, out):
    """The oracle's per-SNP matrices of the golden inputs, written with scipy as a cellSNP directory."""
    from oracle import oracle
    from xcltk_b200 import lib
    from xcltk_b200.baf import pileup
    from xcltk_b200.utils.sam import build_tid_maps
    sites = pileup.load_sites(r["snps"]).snps
    with open(r["barcodes"]) as fp:
        samples = sorted(x.strip() for x in fp)
    chroms = list(dict.fromkeys(s.chrom for s in sites))
    gid_of, tid_maps = build_tid_maps([lib.bam_references(r["sam"])], chroms)
    ks = lib.KeySpace()
    umi = r["kw"]["umi_tag"]
    host = lib.decode_bams([r["sam"]], tid_maps, r["kw"]["cell_tag"], umi, True, ks, 4)
    conf = Conf(min_mapq=20, min_len=30, incl_flag=0, excl_flag=772 if umi else 1796, no_orphan=True)
    conf.use_umi = lambda: umi is not None
    gid = np.array([gid_of.get(s.chrom, -1) for s in sites], np.int32)
    pos0 = np.array([s.pos - 1 for s in sites], np.int32)
    ref = np.array([LETTERS.index(s.ref) for s in sites], np.uint8)
    alt = np.array([LETTERS.index(s.alt) for s in sites], np.uint8)
    exp = oracle_snp(host, gid, pos0, ref, alt, np.array([ks.encode(b) for b in samples], np.uint64), len(samples), conf,
                     0, 0.0)
    host.close()
    os.makedirs(out)
    with open(os.path.join(out, "cellSNP.samples.tsv"), "w") as fp:
        fp.write("".join(s + "\n" for s in samples))
    with gzip.open(os.path.join(out, "cellSNP.base.vcf.gz"), "wt") as fp:
        fp.write("#CHROM\tPOS\tID\tREF\tALT\n" + "".join("%s\t%d\t.\t%s\t%s\n" % (s.chrom_text, s.pos, s.ref, s.alt)
                                                          for s in sites))
    dense = []
    for tag, (row, col, val) in zip(("AD", "DP", "OTH"), exp):
        m = scipy.sparse.coo_matrix((val, (row, col)), shape=(len(sites), len(samples)))
        scipy.io.mmwrite(os.path.join(out, "cellSNP.tag.%s.mtx" % tag), m)
        dense.append(m.toarray())
    return dense


@pytest.mark.parametrize("case", ["c1_chr22_10x", "bch869_smartseq"])
def test_pileup_wrapper_end_to_end(gpu_ctx, case, tmp_path, monkeypatch):
    """pileup_wrapper through the device decoder, the host decoder (zero-copy batch) and two emulated GPU shards:
    the matrices equal the oracle's, the three directories are byte-identical; then afc_wrapper's local phasing
    reads the directory and writes what it writes from the oracle's directory."""
    from xcltk_b200.baf.fc.main import afc_wrapper
    from xcltk_b200.baf.pileup import pileup_wrapper
    r = golden_inputs(case)
    exp = oracle_dir(r, str(tmp_path / "oracle"))
    assert exp[1].sum() > 100
    runs = {}
    for mode in ("device", "host", "sharded"):
        with monkeypatch.context() as mp:
            if mode == "host":
                mp.setenv("XCLTK_B200_DEVICE_DECODE", "0")
            if mode == "sharded":
                mp.setenv("XCLTK_B200_GPUS", "2")
                mp.setenv("XCLTK_B200_EMULATE_SHARDS", "1")
            out = str(tmp_path / mode)
            assert pileup_wrapper(r["sam"], r["barcodes"], r["snps"], out, ncores=4, **r["kw"]) == 0
        runs[mode] = {f: open(os.path.join(out, f), "rb").read() for f in sorted(os.listdir(out))}
        for tag, e in zip(("AD", "DP", "OTH"), exp):
            got = scipy.io.mmread(os.path.join(out, "cellSNP.tag.%s.mtx" % tag))
            assert np.array_equal(np.asarray(scipy.sparse.coo_matrix(got).toarray()), e), (mode, tag)
    assert sorted(runs["device"]) == ["cellSNP.base.vcf.gz", "cellSNP.samples.tsv", "cellSNP.tag.AD.mtx",
                                      "cellSNP.tag.DP.mtx", "cellSNP.tag.OTH.mtx"]
    assert runs["device"] == runs["host"] == runs["sharded"]
    res = {}
    for src in ("device", "oracle"):
        out = str(tmp_path / ("afc_" + src))
        assert afc_wrapper(r["sam"], r["barcodes"], r["features"], r["snps"], out, cellsnp_dir=str(tmp_path / src),
                           output_all_reg=True, ncores=4, **r["kw"]) == 0
        res[src] = {f: open(os.path.join(out, f), "rb").read()
                    for f in ("xcltk.region.tsv", "xcltk.AD.mtx", "xcltk.DP.mtx", "xcltk.OTH.mtx")}
    assert res["device"] == res["oracle"]
    assert res["device"]["xcltk.DP.mtx"].count(b"\n") > 10
