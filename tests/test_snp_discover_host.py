"""SNP discovery on the CPU: the oracle orc_snp_discover on hand-built records (allele inference, filter edges,
first-read-wins), its totals against the baf oracle on the golden library, and the host side of `xcltk pileup`
without candidate SNPs (options, --chrom resolution, defaults, the VCF's contig names)."""

import gzip
import os

import numpy as np
import pytest

import discover_oracle
from recsets import CODE, D, M, build, cell_keys, umi_keys
from xcltk_b200.baf import pileup
from xcltk_b200.baf.fc.config import Config

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Conf(object):
    min_mapq, min_len, min_include = 0, 1, 0
    incl_flag, excl_flag, no_orphan = 0, 0, False

    def use_barcodes(self):
        return True

    def use_umi(self):
        return True


def column(bases, first=None):
    """Reads over position 10, one (cell, UMI) per base of `bases` (letters of NT16); `first`: per UMI an earlier
    read given as (ops, letter at 10) that claims it."""
    rows = []
    for u, b in enumerate(bases):
        if first and u in first:
            ops, letter = first[u]
            rows.append((ops, letter, u))
        rows.append(([(M, 20)], b, u))
    seqs, opsl = [], []
    for ops, letter, _u in rows:
        q = sum(l for op, l in ops if op == M)
        s = ["C"] * q
        if ops == [(M, 20)]:
            s[10] = letter
        seqs.append(np.array([CODE[x] for x in s], np.uint8))
        opsl.append(ops)
    n = len(rows)
    ck = cell_keys(1)
    return build(np.zeros(n, np.int64), ck[0], umi_keys(len(bases))[[r[2] for r in rows]], [(0, 0, 0, n)],
                 ops=opsl, seq=seqs), ck


def discover(reads, ck, min_count, min_maf):
    from oracle import oracle
    return discover_oracle.orc_snp_discover(reads, [0], [0], [100], ck, oracle.params(Conf()), min_count, min_maf)


def at10(res):
    k = np.nonzero(res["pos"] == 10)[0]
    return None if len(k) == 0 else (int(res["ref"][k[0]]), int(res["alt"][k[0]]), res["totals"][k[0]].tolist())


@pytest.mark.parametrize("bases,ref,alt", [("AACC", 0, 1), ("CCAA", 0, 1), ("GGTT", 2, 3), ("TTTG", 3, 2),
                                           ("CGGT", 2, 1), ("ATTTNNNNNN", 3, 0)])
def test_allele_inference_tie_order(bases, ref, alt):
    reads, ck = column(bases)
    got = at10(discover(reads, ck, 0, 0.0))
    assert got is not None and got[:2] == (ref, alt)
    assert got[2] == [bases.count(b) for b in "ACGTN"]


def test_alt_at_least_one_and_n_counts_in_the_sum_only():
    reads, ck = column("AAAANNNN")
    assert at10(discover(reads, ck, 0, 0.0)) is None          # ALT (C) = 0: never a site
    reads, ck = column("AAAGNNNNNN")
    assert at10(discover(reads, ck, 10, 0.1)) == (0, 2, [3, 0, 1, 0, 6])     # sum 10 with the N
    assert at10(discover(reads, ck, 11, 0.0)) is None
    assert at10(discover(reads, ck, 10, 0.1000001)) is None   # ALT 1 < 10 * 0.1000001


def test_filter_at_equality():
    reads, ck = column("AAAAAAAAGG")                           # sum 10, ALT 2
    assert at10(discover(reads, ck, 10, 0.2)) is not None     # 2 >= 10 * 0.2
    assert at10(discover(reads, ck, 10, 0.21)) is None


def test_none_winners_are_skipped():
    """The first read of UMIs 0..2 has a deletion at 10 (None): those UMIs count nowhere, whatever their later
    reads carry."""
    first = {u: ([(M, 10), (D, 1), (M, 9)], None) for u in range(3)}
    reads, ck = column("GGGAAAAC", first=first)
    assert at10(discover(reads, ck, 0, 0.0)) == (0, 1, [4, 1, 0, 0, 0])


def test_oracle_totals_equal_the_baf_oracle_on_golden():
    """At the discovered sites of the golden 10x library the deduplicated totals are the baf oracle's: with one
    region per site, GT 0|1 and no filter, AD sums to ALT and DP to REF + ALT."""
    from oracle import oracle
    from test_gpu_snp_pileup import oracle_snp
    from xcltk_b200 import lib
    from xcltk_b200.utils.sam import build_tid_maps
    g = os.path.join(GOLD, "c1_chr22_10x")
    bam = os.path.join(g, "a.bam")
    _gid_of, tid_maps = build_tid_maps([lib.bam_references(bam)], ["22"])
    ks = lib.KeySpace()
    host = lib.decode_bams([bam], tid_maps, "CB", "UB", True, ks, 2)
    with open(os.path.join(g, "barcodes.tsv")) as fp:
        bcs = sorted(x.strip() for x in fp)
    ck = np.array([ks.encode(b) for b in bcs], np.uint64)
    conf = Conf()
    conf.min_mapq, conf.min_len, conf.excl_flag, conf.no_orphan = 20, 30, 772, True
    res = discover_oracle.orc_snp_discover(host, [0], [0], [50818468], ck, oracle.params(conf), 4, 0.1)
    n = len(res["pos"])
    assert n > 10
    ad, dp, _oth = oracle_snp(host, res["gid"], res["pos"], res["ref"], res["alt"], ck, len(bcs), conf, 0, 0.0)
    t, ii = res["totals"], np.arange(n)
    assert np.array_equal(np.bincount(ad[0], weights=ad[2], minlength=n), t[ii, res["alt"]])
    assert np.array_equal(np.bincount(dp[0], weights=dp[2], minlength=n), t[ii, res["alt"]] + t[ii, res["ref"]])
    host.close()


def test_chrom_option_and_mode_defaults():
    conf = Config()
    conf.min_count = conf.min_maf = conf.chrom = None
    assert pileup.parse_args(["xcltk", "pileup", "-s", "a.bam", "--chrom", "1,X", "-O", "o"], conf) is None
    assert conf.chrom == "1,X" and conf.snp_fn is None
    pileup.filter_defaults(conf)
    assert (conf.min_count, conf.min_maf) == (20, 0.1)
    conf = Config()
    conf.min_count = conf.min_maf = None
    conf.snp_fn = "x.vcf"
    pileup.filter_defaults(conf)
    assert (conf.min_count, conf.min_maf) == (0, 0.0)
    conf = Config()
    conf.min_count, conf.min_maf = 3, None
    pileup.filter_defaults(conf)
    assert (conf.min_count, conf.min_maf) == (3, 0.1)
    import io
    buf = io.StringIO()
    pileup.usage(buf)
    assert "--chrom" in buf.getvalue() and "[0 with -P, 20 without]" in buf.getvalue()


def test_chrom_resolution_with_and_without_chr():
    c1 = os.path.join(GOLD, "c1_chr22_10x", "a.bam")              # header: chr22
    bch = os.path.join(GOLD, "bch869_smartseq", "BCH869.output.bam")   # header: 1, 2, ..., 22, X, ...
    assert pileup.discover_targets([c1], "22") == [("22", "chr22", 50818468)]
    assert pileup.discover_targets([c1], "chr22,21") == [("chr22", "chr22", 50818468)]
    t = pileup.discover_targets([bch], pileup.DEFAULT_CHROMS)
    assert [x[0] for x in t] == [str(i) for i in range(1, 23)]
    assert t[21][1:] == ("22", 51304566)
    assert pileup.discover_targets([bch], "chr22")[0][1] == "22"


def test_vcf_uses_the_header_contig_names(tmp_path):
    sites = [pileup.Site("22", "chr22", 17, "A", "G"), pileup.Site("22", "chr22", 40, "T", "C")]
    z = np.zeros(0, np.int32)
    ad = (np.array([0, 1], np.int32), np.array([0, 0], np.int32), np.array([2, 1], np.int32), (2, 1))
    dp = (np.array([0, 1], np.int32), np.array([0, 0], np.int32), np.array([3, 4], np.int32), (2, 1))
    pileup.write_cellsnp_dir(str(tmp_path), ["c"], sites, ad, dp, (z, z, z, (2, 1)), np.ones(2, np.uint8))
    lines = gzip.open(str(tmp_path / "cellSNP.base.vcf.gz"), "rt").read().splitlines()
    assert lines[2:] == ["chr22\t17\t.\tA\tG\t.\tPASS\tAD=2;DP=3;OTH=0", "chr22\t40\t.\tT\tC\t.\tPASS\tAD=1;DP=4;OTH=0"]


def test_no_candidates_and_no_contigs_is_an_error(tmp_path):
    bam = os.path.join(GOLD, "c1_chr22_10x", "a.bam")
    bc = os.path.join(GOLD, "c1_chr22_10x", "barcodes.tsv")
    assert pileup.pileup_wrapper(bam, bc, None, str(tmp_path / "o"), chrom="Z9") == -1     # not in the BAM


def test_ctypes_mirrors_match_the_header(tmp_path):
    """The ctypes structs of the discovery entry point and of the extended synth parameters have the header's
    field offsets and sizes."""
    import ctypes as C
    import subprocess
    from xcltk_b200 import lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    mirrors = {"xg_sites": lib.Sites, "xg_discover_filter": lib.DiscoverFilter, "xg_synth_params": lib.SynthParams}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "xcltk_b200.h"', "int main(void) {"]
    for cname, py in mirrors.items():
        lines.append('printf("%%s %%zu\\n", "%s", sizeof(%s));' % (cname, cname))
        for f, _t in py._fields_:
            lines.append('printf("%%s.%%s %%zu\\n", "%s", "%s", offsetof(%s, %s));' % (cname, f, cname, f))
    lines.append("return 0; }")
    src, exe = tmp_path / "abi.c", str(tmp_path / "abi")
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), "-o", exe, str(src)], check=True)
    got = dict(x.split() for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split("\n")
               if x)
    for cname, py in mirrors.items():
        assert int(got[cname]) == C.sizeof(py), cname
        for f, _t in py._fields_:
            assert int(got["%s.%s" % (cname, f)]) == getattr(py, f).offset, (cname, f)


# ---- the raw-scan mirror (orc_disc_raw) against a plain per-read loop -------------------------------------------
W = 2048                   # DISC_W of discover.cu


def py_disc_raw(reads, tg, ck, conf, min_count, min_maf):
    """The raw scan's counters restated read by read with sets and dicts: (covered windows, positions scanned,
    (read, window) entries, raw candidates)."""
    import math
    a = reads._arrays
    pe, fmq, keys = a["pos_end"].reshape(-1, 2), a["fmq"], a["keys"].reshape(-1, 2)
    cig_off, cigar, seq_off, seq = a["cig_off"], a["cigar"], a["seq_off"], a["seq"].view(np.uint8)
    none, empty = 0xFFFFFFFFFFFFFFFF, 0
    n_gid = max(r[1] for r in reads.runs) + 1
    live, n_win = [], 0                                  # (gid, beg, end, first window) in caller order
    for g, b, e in zip(*tg):
        if 0 <= g < n_gid and b >= 0 and e > b:
            live.append((g, b, e, n_win))
            n_win += -(-(e - b) // W)
    listed = set(int(k) for k in ck) if conf.use_barcodes() else None
    entries, hist = {}, {}
    for _bam, gid, rb, re_ in reads.runs:
        mine = [t for t in live if t[0] == gid]
        for i in range(rb, re_):
            pos, end = int(pe[i, 0]), int(pe[i, 1])
            if not any(b < end and pos < e for _g, b, e, _w in mine):
                continue
            flag, mapq = int(fmq[i]) & 0xFFFF, (int(fmq[i]) >> 16) & 0xFF
            if mapq < conf.min_mapq or (conf.excl_flag and flag & conf.excl_flag):
                continue
            if (conf.incl_flag and not flag & conf.incl_flag) or (conf.no_orphan and flag & 1 and not flag & 2):
                continue
            cell, umi = int(keys[i, 0]), int(keys[i, 1])
            if seq_off[i] == 0xFFFFFFFF or umi in (none, empty) or (listed is not None and cell not in listed):
                continue
            n_ops = int(fmq[i]) >> 24
            if n_ops == 0:
                ops = [(0, end - pos)]
            else:
                o = int(cig_off[i])
                k = int(cigar[o - 1]) if n_ops == 255 else n_ops
                ops = [(int(w) & 15, int(w) >> 4) for w in cigar[o:o + k]]
            if sum(l for op, l in ops if op in (0, 7, 8)) < conf.min_len:
                continue
            wins, rp, qp = set(), pos, 0
            for op, l in ops:
                if op in (0, 7, 8):
                    for j in range(l):
                        p, q = rp + j, qp + j
                        for _g, b, e, w0 in mine:
                            if b <= p < e:
                                w = w0 + (p - b) // W
                                wins.add(w)
                                byte = int(seq[4 * int(seq_off[i]) + (q >> 1)])
                                nib = byte & 15 if q & 1 else byte >> 4
                                c = hist.setdefault((w, p), [0] * 5)
                                c[{1: 0, 2: 1, 4: 2, 8: 3}.get(nib, 4)] += 1
                    rp += l
                    qp += l
                elif op in (2, 3):
                    rp += l
                elif op in (1, 4):
                    qp += l
            for w in wins:
                entries[w] = entries.get(w, 0) + 1
    t_sum = math.ceil(min_count) if min_count > 0 else 0
    t_alt = max(1, math.ceil(min_count * min_maf)) if min_count > 0 and min_maf > 0 else 1
    scanned = 0
    for _g, b, e, w0 in live:
        for w in range(w0, w0 + -(-(e - b) // W)):
            if w in entries:
                s = b + (w - w0) * W
                scanned += min(e, s + W) - s
    cand = sum(1 for c in hist.values() if sum(c) >= t_sum and sorted(c[:4])[2] >= t_alt)
    return len(entries), scanned, sum(entries.values()), cand


def mixed_batch(seed, n, contig_len):
    """Random exotic CIGARs on two contigs with every filter's failing values mixed in: flags (unmapped, orphan,
    duplicate), low mapq, short reads, unlisted / missing cells, none / empty UMIs, records without SEQ.  Unmapped
    reads end at pos + 1 but keep their CIGAR."""
    from test_gpu_baf_edges import exotic, random_codes
    from recsets import query_len
    rng = np.random.RandomState(seed)
    ops = [exotic(rng) for _ in range(n)]
    gid = (rng.rand(n) < 0.4).astype(np.int64)
    pos = rng.randint(0, contig_len, size=n)
    order = np.lexsort((pos, gid))
    gid, pos, ops = gid[order], pos[order], [ops[k] for k in order]
    ln = rng.randint(1, 120, size=n)
    seq = [None if rng.rand() < 0.03 else random_codes(rng, query_len(o) if o else int(l)) for o, l in zip(ops, ln)]
    ck = cell_keys(12)
    cell = np.concatenate([ck, cell_keys(3, salt=100), [0xFFFFFFFFFFFFFFFF]])[rng.randint(0, 16, size=n)]
    umi = umi_keys(200)[rng.randint(0, 200, size=n)]
    umi[rng.rand(n) < 0.03] = 0xFFFFFFFFFFFFFFFF
    umi[rng.rand(n) < 0.03] = 0
    flag = rng.choice([0, 0, 0, 4, 1, 3, 1024, 16], size=n).astype(np.uint32)
    mapq = rng.choice([60, 20, 19, 0], size=n).astype(np.uint32)
    h = int((gid == 0).sum())
    reads = build(pos, cell.astype(np.uint64), umi, [(0, 0, 0, h), (0, 1, h, n)], end=pos + ln, ops=ops, seq=seq,
                  flag=flag, mapq=mapq)
    un = np.nonzero(flag & 4)[0]
    reads.pos_end[un, 1] = reads.pos_end[un, 0] + 1
    return reads, ck


MIRROR_TARGETS = [
    ([0], [0], [9000]),
    ([1, -1, 0, 0, 5, 0, 1], [4000, 0, 3071, 1000, 0, 7000, 0], [9000, 50, 7000, 3071, 100, 6000, 4000]),
    ([0, 0, 1, 0], [2047, 2049, 1, 8191], [2048, 4097, 2, 8200]),
]


@pytest.mark.parametrize("tg", range(len(MIRROR_TARGETS)))
def test_raw_scan_mirror_against_a_per_read_loop(tg):
    """orc_disc_raw (C) equals a per-read Python restatement on the CIGAR panel with the 301-op read, and on a
    mixed batch of exotic CIGARs and failing filters; targets starting mid-window, of length 1, adjacent, on two
    contigs out of order, and skipped (gid -1, gid past the last contig, end <= beg)."""
    from oracle import oracle
    from recsets import CIGAR_PANEL, cigar_panel
    from test_gpu_baf_edges import WIDE
    tgt = tuple(np.array(x, np.int32) for x in MIRROR_TARGETS[tg])
    conf = Conf()
    panel, pck = cigar_panel(CIGAR_PANEL + [WIDE])
    mixed, mck = mixed_batch(4, 700, 9000)
    seen = []
    for reads, ck, mc, maf in ((panel, pck, 0, 0.0), (panel, pck, 2, 0.5), (mixed, mck, 0, 0.0),
                               (mixed, mck, 3, 0.1), (mixed, mck, 2.5, 0.4)):
        for c in (conf, type("C", (Conf,), {"min_mapq": 20, "min_len": 30, "excl_flag": 1024, "no_orphan": True,
                                             "incl_flag": 0})()):
            got = discover_oracle.orc_disc_raw(reads, *tgt, ck, oracle.params(c), mc, maf)
            assert got == py_disc_raw(reads, tgt, ck, c, mc, maf), (mc, maf)
            seen.append(got)
    assert all(s[2] >= s[0] > 0 and s[3] > 0 for s in seen[4:])


def test_raw_scan_mirror_rejects_what_the_device_rejects():
    from oracle import oracle
    reads, ck = column("AACC")
    with pytest.raises(ValueError):          # [0, 50) and [40, 60) overlap
        discover_oracle.orc_disc_raw(reads, [0, 0], [0, 40], [50, 60], ck, oracle.params(Conf()), 0, 0.0)
    bare = build(np.zeros(2, np.int64), ck[0], umi_keys(2), [(0, 0, 0, 2)], end=np.full(2, 20))
    with pytest.raises(ValueError):
        discover_oracle.orc_disc_raw(bare, [0], [0], [50], ck, oracle.params(Conf()), 0, 0.0)
