"""SNP discovery (xg_snp_discover / Context.snp_discover / pileup_wrapper without candidate SNPs) against the CPU
oracle orc_snp_discover, a brute force over every covered target position with plp_snp's first-read-wins pileup
and no pre-filter.  Every case compares sites, alleles, totals and the matrices of the kept sites, and asserts the
stage counters it targets: timing()[6] positions scanned, [7] raw candidates, [11] pileup slices, [14] kept sites."""

import gzip
import os

import numpy as np
import pytest

import discover_oracle
from recsets import CODE, D, M, N, build, cell_keys, umi_keys
from test_gpu_baf_edges import Conf
from test_gpu_snp_pileup import GOLD, golden_inputs, oracle_snp, same
from xcltk_b200 import engine

pytestmark = pytest.mark.gpu

W = 2048                   # DISC_W of discover.cu: positions per raw-scan window


def codes(s):
    return np.array([CODE[b] for b in s], dtype=np.uint8)


def check(ctx, reads, ck, n_cols, tg, conf=None, min_count=20, min_maf=0.1):
    """tg: (gid, beg, end) arrays.  Returns (sites, timing())."""
    from oracle import oracle
    conf = conf or Conf()
    g, b, e = (np.asarray(x, np.int32) for x in tg)
    params = engine.make_params(conf, reads.max_aln_len, with_include=False)
    exp = discover_oracle.orc_snp_discover(reads, g, b, e, ck, oracle.params(conf), min_count, min_maf)
    d = ctx.upload(reads)
    try:
        got = ctx.snp_discover(d, g, b, e, ck, n_cols, params, min_count, min_maf)
        t = ctx.timing()
        for k in ("gid", "pos", "ref", "alt", "totals"):
            assert np.array_equal(got[k], exp[k]), (k, got[k][:10], exp[k][:10])
        assert t[14] == len(exp["pos"])
        if len(got["pos"]):
            mats = ctx.snp_pileup(d, got["gid"], got["pos"], ck, n_cols, params, got["ref"], got["alt"], min_count,
                                  min_maf)
            same(mats, oracle_snp(reads, got["gid"], got["pos"], got["ref"], got["alt"], ck, n_cols, conf,
                                  min_count, min_maf), "matrices of the discovered sites")
    finally:
        d.close()
    return got, t


def test_first_read_wins_with_none_and_n(gpu_ctx):
    """At p = 1000 the first read of each (cell, UMI) has a deletion, an N skip or an N base there: it claims the
    UMI and counts nowhere (or in N), so later reads of that UMI with the ALT base do not count."""
    ck = cell_keys(40)
    rows = []                          # (pos, ops, seq, cell, umi)
    L = 60
    for c in range(40):                # 40 UMIs with REF A at 1000 (query index 10 of reads at 990)
        rows.append((990, [(M, L)], "C" * 10 + "A" + "C" * (L - 11), c, c))
    for c in range(12):                # 12 UMIs with ALT G
        rows.append((990, [(M, L)], "C" * 10 + "G" + "C" * (L - 11), c, 100 + c))
    for c, kind in enumerate(["del", "skip", "N"] * 6):     # 18 UMIs whose first read has None / N at 1000
        u = 200 + c
        if kind == "del":
            rows.append((995, [(M, 5), (D, 2), (M, 40)], "C" * 45, c, u))
        elif kind == "skip":
            rows.append((995, [(M, 5), (N, 30), (M, 40)], "C" * 45, c, u))
        else:
            rows.append((995, [(M, L)], "CCCCCN" + "C" * (L - 6), c, u))
        rows.append((996, [(M, L)], "CCCC" + "G" + "C" * (L - 5), c, u))   # later read, same UMI, ALT G
    rows.sort(key=lambda r: r[0])
    pos = [r[0] for r in rows]
    reads = build(pos, ck[[r[3] for r in rows]], umi_keys(300)[[r[4] for r in rows]], [(0, 0, 0, len(rows))],
                  ops=[r[1] for r in rows], seq=[codes(r[2]) for r in rows])
    got, t = check(gpu_ctx, reads, ck, 40, ([0], [0], [5000]), min_count=20, min_maf=0.1)
    i = list(got["pos"]).index(1000)
    assert list(got["totals"][i]) == [40, 0, 12, 0, 6]
    assert (got["ref"][i], got["alt"][i]) == (0, 2)
    assert t[7] >= 1 and 0 < t[6] <= 2 * W


def test_window_boundaries_long_gap_and_contig_edges(gpu_ctx):
    """Reads cross window edges (2047 / 2048), one read skips >= 500 kb with N, sites at position 0 and at the last
    base of the target; a second contig holds a target without reads."""
    rng = np.random.RandomState(3)
    ck = cell_keys(30)
    clen = 700000
    sites = [0, 2047, 2048, 4095, 650000, clen - 1]
    rows = []
    for p in sites:
        for k in range(30):
            base = "A" if k < 18 else "T"
            s0 = max(0, min(p - rng.randint(0, 50), clen - 60))
            q = p - s0
            seq = "".join(rng.choice(list("CG"), 60))
            seq = seq[:q] + base + seq[q + 1:]
            rows.append((s0, [(M, 60)], seq, k, len(rows)))
    # one spliced read per cell: 30 M at 2030, N of 600 000, 30 M at 602 060 -- aligned on both sides
    for k in range(30):
        rows.append((2030, [(M, 30), (N, 600000), (M, 30)], "G" * 60, k, 5000 + k))
    rows.sort(key=lambda r: r[0])
    reads = build([r[0] for r in rows], ck[[r[3] for r in rows]], umi_keys(6000)[[r[4] for r in rows]],
                  [(0, 0, 0, len(rows))], ops=[r[1] for r in rows], seq=[codes(r[2]) for r in rows])
    got, t = check(gpu_ctx, reads, ck, 30, ([0, 1], [0, 0], [clen, 5000]))
    assert set(sites) <= set(got["pos"].tolist())
    assert (got["pos"] == clen - 1).any() and (got["pos"] == 0).any()
    # the N gap is not scanned: positions of windows with reads only, far fewer than the contig
    assert t[6] < clen / 4


def test_depth_70000(gpu_ctx):
    """70 000 UMIs at one position: no counter wraps, the site is kept with the oracle's totals."""
    n = 70000
    ck = cell_keys(500)
    pos = np.full(n, 100, np.int64)
    seq = np.tile(codes("C" * 20 + "A" + "C" * 29), (n, 1))
    seq[::3, 20] = CODE["G"]
    reads = build(pos, ck[np.arange(n) % 500], umi_keys(n), [(0, 0, 0, n)], end=pos + 50, seq=seq)
    got, t = check(gpu_ctx, reads, ck, 500, ([0], [0], [1000]))
    i = list(got["pos"]).index(120)
    assert got["totals"][i].sum() == n and got["totals"][i][2] == (n + 2) // 3


def test_prefilter_passes_then_umi_collapse_fails(gpu_ctx):
    """Raw counts pass at 300 and 400 but the deduplicated ones do not: at 300 the ALT reads are 30 copies of one
    UMI (MAF fails), at 400 all reads are copies of 5 UMIs (count fails).  500 passes both."""
    ck = cell_keys(10)
    rows = []
    for p, n_ref, n_alt, alt_umis, ref_umis in ((300, 60, 30, 1, 60), (400, 40, 20, 2, 3), (500, 60, 30, 30, 60)):
        for k in range(n_ref):
            rows.append((p - 5, "CCCCCA" + "C" * 44, 0 if p == 400 else k % 10, 1000 * p + k % ref_umis))
        for k in range(n_alt):
            rows.append((p - 5, "CCCCCT" + "C" * 44, k % 10 if p == 500 else 0, 1000 * p + 500 + k % alt_umis))
    rows.sort(key=lambda r: r[0])
    uk = {u: i for i, u in enumerate(sorted(set(r[3] for r in rows)))}
    keys = umi_keys(len(uk))
    reads = build([r[0] for r in rows], ck[[r[2] for r in rows]], keys[[uk[r[3]] for r in rows]],
                  [(0, 0, 0, len(rows))], end=np.array([r[0] for r in rows]) + 50,
                  seq=[codes(r[1]) for r in rows])
    got, t = check(gpu_ctx, reads, ck, 10, ([0], [0], [2000]))
    assert got["pos"].tolist() == [500]
    assert t[7] == 3 and t[14] == 1          # raw candidates 300 / 400 / 500, one kept


def test_sample_mode_and_slices(gpu_ctx):
    """Sample-ID mode (column = BAM, two BAMs) and the exact stage in slices of 3 candidates."""
    rng = np.random.RandomState(5)
    n = 4000
    pos = np.sort(rng.randint(0, 3000, n))
    seq = np.tile(codes("A" * 50), (n, 1))
    ref = rng.randint(0, 4, 3100)
    for j in range(50):
        seq[:, j] = np.array([CODE["ACGT"[x]] for x in ref[pos + j]])
    het = rng.rand(n, 50) < 0.3
    seq[het & ((pos[:, None] + np.arange(50)) % 97 == 0)] = CODE["T"]
    bam = (rng.rand(n) < 0.5).astype(np.int64)
    order = np.lexsort((pos, bam))
    h = int((bam == 0).sum())
    reads = build(pos[order], 0, umi_keys(n)[rng.randint(0, n, n)][order], [(0, 0, 0, h), (1, 0, h, n)],
                  end=pos[order] + 50, seq=seq[order])
    conf = Conf(barcodes=False)
    got, t = check(gpu_ctx, reads, None, 2, ([0], [0], [3100]), conf=conf, min_count=10, min_maf=0.05)
    assert len(got["pos"]) > 5 and t[11] == 1
    d = gpu_ctx.upload(reads)
    try:
        params = engine.make_params(conf, reads.max_aln_len, with_include=False)
        gpu_ctx.set_option("discover_slice", 3)
        sl = gpu_ctx.snp_discover(d, [0], [0], [3100], None, 2, params, 10, 0.05)
        assert gpu_ctx.timing()[11] == -(-gpu_ctx.timing()[7] // 3) > 1
    finally:
        gpu_ctx.set_option("discover_slice", 0)
        d.close()
    for k in got:
        assert np.array_equal(got[k], sl[k]), k


def test_empty_batch_and_target_without_reads(gpu_ctx):
    from xcltk_b200 import lib
    ck = cell_keys(4)
    z = np.zeros(0, np.uint32)
    empty = lib.ArrayReads(np.zeros((0, 2), np.int32), z, np.zeros(1, np.uint32), np.zeros((0, 2), np.uint64),
                           np.zeros(1, np.uint32), [], z, np.zeros(1, np.uint32), max_aln_len=1, max_span=1)
    got, t = check(gpu_ctx, empty, ck, 4, ([0], [0], [100000]))
    assert len(got["pos"]) == 0 and t[7] == 0
    pos = np.arange(0, 200, 2, dtype=np.int64)
    reads = build(pos, ck[pos % 4], umi_keys(100), [(0, 0, 0, 100)], end=pos + 40,
                  seq=np.tile(codes("ACGT" * 10), (100, 1)))
    got, t = check(gpu_ctx, reads, ck, 4, ([1], [0], [100000]))      # contig 1 has no reads
    assert len(got["pos"]) == 0 and t[6] == 0


def test_synthetic_3m_pseudo_reference(gpu_ctx):
    """3M device-synthesised reads over a pseudo-reference with 0.1 % errors and 300 planted SNPs: every planted
    SNP with enough depth is found, the site set equals the oracle's and the raw counters equal orc_disc_raw's."""
    from oracle import oracle
    rng = np.random.RandomState(9)
    span = (np.array([0], np.int32), np.array([0], np.int32), np.array([2000000], np.int32))
    n_snp = 300
    sp = np.sort(rng.choice(np.arange(100, 1999000), n_snp, replace=False)).astype(np.int32)
    sref = rng.randint(0, 4, n_snp).astype(np.uint8)
    salt = ((sref + 1 + rng.randint(0, 3, n_snp)) % 4).astype(np.uint8)
    snps = (np.zeros(n_snp, np.int32), sp, sref, salt, rng.randint(0, 2, n_snp).astype(np.uint8))
    d, bk = gpu_ctx.synth_reads(3000000, 2000, *span, seed=21, want_seq=True, snps=snps, ref_error=0.001)
    try:
        host = d.download()
        conf = Conf(min_mapq=20, min_len=30, excl_flag=772, no_orphan=True)
        params = engine.make_params(conf, host.max_aln_len, with_include=False)
        got = gpu_ctx.snp_discover(d, [0], [0], [2000000], bk, 2000, params, 20, 0.1)
        t = gpu_ctx.timing()
    finally:
        d.close()
    exp = discover_oracle.orc_snp_discover(host, [0], [0], [2000000], bk, oracle.params(conf), 20, 0.1)
    for k in ("gid", "pos", "ref", "alt", "totals"):
        assert np.array_equal(got[k], exp[k]), k
    # the raw scan's covered windows, positions scanned, entries and candidates equal their mirror's
    raw = discover_oracle.orc_disc_raw(host, [0], [0], [2000000], bk, oracle.params(conf), 20, 0.1)
    assert discover_oracle.raw_counters(t) == raw and raw[0] == -(-2000000 // W)
    found = set(got["pos"].tolist())
    assert t[7] < t[6] / 100 and t[14] <= t[7]        # the pre-filter pruned the background
    deep = [p for p in sp.tolist() if p in found]
    assert len(deep) > 0.8 * n_snp
    host.close()


@pytest.mark.parametrize("case", ["c1_chr22_10x", "bch869_smartseq"])
def test_pileup_wrapper_discovers_end_to_end(gpu_ctx, case, tmp_path, monkeypatch):
    """pileup_wrapper without candidate SNPs through the device decoder, the host decoder and two emulated shards
    gives identical bytes; fed back as -P its own cellSNP.base.vcf.gz gives identical matrices."""
    from xcltk_b200.baf.pileup import pileup_wrapper
    r = golden_inputs(case)
    chrom = "22" if case == "c1_chr22_10x" else ",".join(str(i) for i in range(1, 23))
    runs = {}
    for mode in ("device", "host", "sharded"):
        with monkeypatch.context() as mp:
            if mode == "host":
                mp.setenv("XCLTK_B200_DEVICE_DECODE", "0")
            if mode == "sharded":
                mp.setenv("XCLTK_B200_GPUS", "2")
                mp.setenv("XCLTK_B200_EMULATE_SHARDS", "1")
            out = str(tmp_path / mode)
            assert pileup_wrapper(r["sam"], r["barcodes"], None, out, ncores=4, chrom=chrom, min_count=4,
                                  min_maf=0.1, **r["kw"]) == 0
        runs[mode] = {f: open(os.path.join(out, f), "rb").read() for f in sorted(os.listdir(out))}
    assert runs["device"] == runs["host"] == runs["sharded"]
    vcf = gzip.decompress(runs["device"]["cellSNP.base.vcf.gz"]).decode().splitlines()
    assert len(vcf) > 3
    if case == "c1_chr22_10x":
        assert all(x.startswith("chr22\t") for x in vcf[2:])      # the BAM header's spelling
    again = str(tmp_path / "again")
    assert pileup_wrapper(r["sam"], r["barcodes"], os.path.join(str(tmp_path / "device"), "cellSNP.base.vcf.gz"),
                          again, ncores=4, **r["kw"]) == 0
    for tag in ("AD", "DP", "OTH"):
        f = "cellSNP.tag.%s.mtx" % tag
        assert open(os.path.join(again, f), "rb").read() == runs["device"][f], tag
