"""`xcltk pileup`: SNP-level allele counting at candidate SNPs on B200, written as a cellsnp-lite style directory.

The step in front of the local-phasing pre-step of `xcltk baf` (`afc_wrapper(cellsnp_dir=...)`), which the reference
leaves to the external cellsnp-lite binary.  Here the counts are defined by the reference's own per-SNP pileup
(plp_snp, xcltk/baf/fc/core.py:198-247, with first-read-wins per (SNP, cell, UMI) and the min_count / min_maf filter)
with every SNP counted as a region of one SNP with GT 0|1 (fc_fet1, core.py:143-194): per SNP and cell, over the
winning UMIs whose allele is not None, AD = UMIs carrying the ALT base, DP = UMIs carrying REF or ALT, OTH = the
others.  Reads -> HBM -> xg_snp_pileup -> cellSNP.samples.tsv, cellSNP.tag.{AD,DP,OTH}.mtx, cellSNP.base.vcf.gz.

Without a candidate list the sites are discovered from the reads (cellsnp-lite's second mode): every position of the
target contigs (--chrom) is piled up the same way, REF / ALT are the two most frequent of A / C / G / T, and the
sites that pass the filter are counted as above (xg_snp_discover, then xg_snp_pileup).
"""

import collections
import getopt
import gzip
import os
import sys
from logging import error, info

import numpy as np

from .. import engine, lib
from ..config import APP, VERSION
from ..utils.sam import build_tid_maps
from ..utils.xlog import init_logging
from .fc import main as afc
from .fc.config import Config
from .fc.utils import load_snp_from_tsv, load_snp_from_vcf

COMMAND = "pileup"
MIN_COUNT = 0            # the default filter (0, 0) keeps every SNP
MIN_MAF = 0.0
DISCOVER_MIN_COUNT = 20  # without candidate SNPs: cellsnp-lite's mode-2 defaults
DISCOVER_MIN_MAF = 0.1
DEFAULT_CHROMS = ",".join(str(i) for i in range(1, 23))
DISCOVER_UNIT = 1 << 20  # genomic windows handed to the GPUs with several devices
BASES = "ACGT"

Site = collections.namedtuple("Site", "chrom chrom_text pos ref alt")   # pos 1-based, as the SNP objects


def pileup_wrapper(sam_fn, barcode_fn, snp_fn, out_dir, sam_list_fn=None, sample_ids=None, sample_id_fn=None,
                   debug_level=0, ncores=1, cell_tag="CB", umi_tag="UB", min_count=None, min_maf=None,
                   min_mapq=20, min_len=30, incl_flag=0, excl_flag=None, no_orphan=True, chrom=None):
    """Python API.  snp_fn: candidate SNPs, a VCF (CHROM POS ID REF ALT; no genotype needed) or the 6-column SNP TSV
    of afc_wrapper (header line skipped, first four columns used).  Without snp_fn the sites are discovered on the
    contigs `chrom` (comma separated names, e.g. xcltk pileup's default "1,2,...,22"); with neither it is an error.
    min_count / min_maf default to 0 / 0 with candidates and to 20 / 0.1 when discovering.  Returns 0, or -1 on
    error."""
    conf = Config()
    conf.sam_fn, conf.sam_list_fn = sam_fn, sam_list_fn
    conf.barcode_fn, conf.snp_fn = barcode_fn, snp_fn
    conf.sample_id_str, conf.sample_id_fn = sample_ids, sample_id_fn
    conf.out_dir, conf.debug = out_dir, debug_level
    conf.cell_tag, conf.umi_tag = cell_tag, umi_tag
    conf.nproc = ncores
    conf.min_count, conf.min_maf = min_count, min_maf
    conf.min_mapq, conf.min_len = min_mapq, min_len
    conf.incl_flag = incl_flag
    conf.excl_flag = -1 if excl_flag is None else excl_flag
    conf.no_orphan = no_orphan
    conf.chrom = chrom
    return afc.afc_run(conf, core=pileup_core)


def load_sites(fn):
    """Candidate SNPs of a VCF or SNP TSV as an SNPSet (REF / ALT upper-cased; sites whose REF or ALT is not one of
    A C G T N are skipped with a warning; duplicates kept; `chrom_text` = CHROM as given)."""
    if fn.endswith((".vcf", ".vcf.gz", ".vcf.bgz")):
        return load_snp_from_vcf(fn, verbose=True, sites=True)
    return load_snp_from_tsv(fn, verbose=True, sites=True)


def _pileup_shard(conf, batch, snps):
    gid, pos0, cell_keys, params = afc.snp_arrays(conf, batch, snps)
    ref_i, alt_i = afc.allele_indices(snps)
    ad, dp, oth, keep = batch.ctx.snp_pileup(batch.dreads, gid, pos0, cell_keys, len(conf.samples), params, ref_i,
                                             alt_i, conf.min_count, conf.min_maf, want_keep=True)
    return (ad, dp, oth), [batch.ctx.timing()], keep


def count_snps(conf, snps, batch=None):
    """(AD, DP, OTH) as (row, col, val, shape) with rows = `snps`, and keep (uint8 per SNP: passed the filter)."""
    chroms = list(dict.fromkeys([s.chrom for s in snps]))
    out, parts = afc.count_units(conf, chroms, [s.chrom for s in snps], [s.pos - 1 for s in snps],
                                 [s.pos for s in snps], lambda b, idx: _pileup_shard(conf, b, [snps[i] for i in idx]),
                                 batch)
    # a SNP no GPU piled up (its genomic chunk holds no read) has zero totals: the filter on those
    keep = np.full(len(snps), 0 if 0 < conf.min_count else 1, dtype=np.uint8)
    for idx, k in parts:
        keep[np.asarray(idx)] = k
    return out, keep


def write_cellsnp_dir(out_dir, samples, snps, ad, dp, oth, keep, n_threads=1):
    """cellSNP.samples.tsv, cellSNP.tag.{AD,DP,OTH}.mtx (rows = the kept SNPs in input order, 1-based) and
    cellSNP.base.vcf.gz (one line per kept SNP, INFO = the three sums; gzip mtime 0: the bytes depend on the
    counts only)."""
    n = len(snps)
    emitted = np.asarray(keep, dtype=bool)
    with open(os.path.join(out_dir, "cellSNP.samples.tsv"), "w") as fp:
        fp.write("".join(smp + "\n" for smp in samples))
    sums = []
    for tag, (row, col, val, _shape) in (("AD", ad), ("DP", dp), ("OTH", oth)):
        row, val = np.asarray(row), np.asarray(val)
        engine.write_mtx(os.path.join(out_dir, "cellSNP.tag.%s.mtx" % tag), n, row, col, val, emitted, len(samples),
                         n_threads)
        sums.append(np.bincount(row, weights=val, minlength=n).astype(np.int64) if len(row) else np.zeros(n, np.int64))
    lines = ["##fileformat=VCFv4.2\n", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"]
    for i in np.nonzero(emitted)[0]:
        s = snps[i]
        lines.append("%s\t%d\t.\t%s\t%s\t.\tPASS\tAD=%d;DP=%d;OTH=%d\n" % (
            getattr(s, "chrom_text", s.chrom), s.pos, s.ref, s.alt, sums[0][i], sums[1][i], sums[2][i]))
    with open(os.path.join(out_dir, "cellSNP.base.vcf.gz"), "wb") as raw:
        with gzip.GzipFile(filename="", mode="wb", fileobj=raw, mtime=0) as fp:
            fp.write("".join(lines).encode())


def filter_defaults(conf):
    """min_count / min_maf left unset: (0, 0) with candidate SNPs, (20, 0.1) when discovering."""
    disc = not conf.snp_fn
    if conf.min_count is None:
        conf.min_count = DISCOVER_MIN_COUNT if disc else MIN_COUNT
    if conf.min_maf is None:
        conf.min_maf = DISCOVER_MIN_MAF if disc else MIN_MAF


def discover_targets(sam_fn_list, chrom):
    """Target contigs of discovery: [(name as given, name as the BAM header spells it, length)] for every name of the
    comma separated `chrom` found in a BAM (resolved with the 'chr' toggle of utils/sam.build_tid_maps); the header
    of the first BAM that has the contig gives its spelling and length."""
    chroms = list(dict.fromkeys(c.strip() for c in chrom.split(",") if c.strip()))
    bam_refs = [lib.bam_references(fn) for fn in sam_fn_list]
    _gid_of, tid_maps = build_tid_maps(bam_refs, chroms)
    out = []
    for g, c in enumerate(chroms):
        for refs, m in zip(bam_refs, tid_maps):
            if g in m:
                name, length = refs[m.index(g)]
                out.append((c, name, int(length)))
                break
    return out


def _discover_shard(conf, batch, unit_gid_name, unit_beg, unit_end, idx):
    """Discovery on the units `idx` of one batch, then the SNP x cell counts of the kept sites."""
    gid = np.array([batch.gid_of.get(unit_gid_name[i], -1) for i in idx], dtype=np.int32)
    beg = np.asarray(unit_beg, dtype=np.int64)[idx].astype(np.int32)
    end = np.asarray(unit_end, dtype=np.int64)[idx].astype(np.int32)
    cell_keys = None
    if conf.use_barcodes():
        cell_keys = np.array([batch.keyspace.encode(b) for b in conf.barcodes], dtype=np.uint64)
    params = engine.make_params(conf, batch.stats["max_aln_len"], with_include=False)
    ctx = batch.ctx
    sites = ctx.snp_discover(batch.dreads, gid, beg, end, cell_keys, len(conf.samples), params, conf.min_count,
                             conf.min_maf)
    t_disc = ctx.timing()
    mats = ctx.snp_pileup(batch.dreads, sites["gid"], sites["pos"], cell_keys, len(conf.samples), params, sites["ref"],
                          sites["alt"], conf.min_count, conf.min_maf)
    return sites, mats, [t_disc, ctx.timing()]


def discover_sites(conf, targets, batch=None):
    """Sites of `targets` (discover_targets) in target order, then by position, and their (AD, DP, OTH) as
    (row, col, val, shape) over those sites.  With several GPUs every GPU discovers inside its own windows of
    DISCOVER_UNIT bp only, so a read in two GPUs' halos never reports a site twice."""
    names = [t[0] for t in targets]
    unit_name, unit_beg, unit_end = [], [], []
    for name, _text, length in targets:
        for b in range(0, length, DISCOVER_UNIT):
            unit_name.append(name)
            unit_beg.append(b)
            unit_end.append(min(length, b + DISCOVER_UNIT))
    res, _sharded = afc.shard_units(conf, names, unit_name, unit_beg, unit_end,
                                    lambda b, idx: _discover_shard(conf, b, unit_name, unit_beg, unit_end, idx),
                                    batch)
    parts = [p for _idx, p in res if p is not None]
    conf.last_timing = parts[0][2] if parts else [[0.0] * 16, [0.0] * 16]
    gid = np.concatenate([p[0]["gid"] for p in parts] + [np.zeros(0, np.int32)])
    pos = np.concatenate([p[0]["pos"] for p in parts] + [np.zeros(0, np.int32)])
    ref = np.concatenate([p[0]["ref"] for p in parts] + [np.zeros(0, np.uint8)])
    alt = np.concatenate([p[0]["alt"] for p in parts] + [np.zeros(0, np.uint8)])
    # gid = index of the target in `names`: target order is gid order
    order = np.lexsort((pos, gid))
    new_row = np.empty(len(order), dtype=np.int64)
    new_row[order] = np.arange(len(order))
    shape = (len(order), len(conf.samples))
    mats, base = [[], [], []], 0
    for p in parts:
        for w in range(3):
            r, c, v = (np.asarray(x) for x in p[1][w][:3])
            mats[w].append((new_row[r.astype(np.int64) + base], c, v))
        base += len(p[0]["gid"])
    out = []
    for w in range(3):
        r = np.concatenate([m[0] for m in mats[w]] + [np.zeros(0, np.int64)])
        c = np.concatenate([np.asarray(m[1], dtype=np.int64) for m in mats[w]] + [np.zeros(0, np.int64)])
        v = np.concatenate([np.asarray(m[2], dtype=np.int64) for m in mats[w]] + [np.zeros(0, np.int64)])
        o = np.lexsort((c, r))
        out.append((r[o].astype(np.int32), c[o].astype(np.int32), v[o].astype(np.int32), shape))
    text = {t[0]: t[1] for t in targets}
    sites = [Site(names[g], text[names[g]], int(p) + 1, BASES[a], BASES[b])
             for g, p, a, b in zip(gid[order], pos[order], ref[order], alt[order])]
    return sites, tuple(out)


def discover_core(conf):
    targets = discover_targets(conf.sam_fn_list, conf.chrom)
    info("mode: SNP discovery (no candidate SNPs given) on %d contigs; min_count=%s, min_maf=%s; pile up in %d "
         "single cells." % (len(targets), conf.min_count, conf.min_maf, len(conf.samples)))
    if not targets:
        error("none of the contigs '%s' is in the BAM files." % conf.chrom)
        raise ValueError("errcode -2")
    info("program configuration:")
    conf.show(fp=sys.stderr, prefix="\t")
    sites, (ad, dp, oth) = discover_sites(conf, targets)
    info("#SNPs: discovered=%d." % len(sites))
    write_cellsnp_dir(conf.out_dir, conf.samples, sites, ad, dp, oth, np.ones(len(sites), np.uint8),
                      engine.n_decode_threads(conf.nproc))


def pileup_core(conf):
    if afc.prepare_samples(conf) < 0 or afc.prepare_tags(conf) < 0:
        raise ValueError("errcode -2")
    filter_defaults(conf)
    if not conf.snp_fn:
        if not getattr(conf, "chrom", None):
            error("SNP file needed! (or the contigs to discover sites on)")
            raise ValueError("errcode -2")
        return discover_core(conf)
    if not os.path.isfile(conf.snp_fn):
        error("snp file '%s' does not exist." % conf.snp_fn)
        raise ValueError("errcode -2")
    info("mode: pile up at candidate SNPs.")
    conf.snp_set = load_sites(conf.snp_fn)
    if not conf.snp_set or conf.snp_set.get_n() <= 0:
        error("failed to load snp file.")
        raise ValueError("errcode -2")
    info("%d SNPs loaded; pile up in %d single cells." % (conf.snp_set.get_n(), len(conf.samples)))
    info("program configuration:")
    conf.show(fp=sys.stderr, prefix="\t")
    snps = conf.snp_set.snps
    (ad, dp, oth), keep = count_snps(conf, snps)
    info("#SNPs: total=%d; passed the filter=%d." % (len(snps), int(np.count_nonzero(keep))))
    write_cellsnp_dir(conf.out_dir, conf.samples, snps, ad, dp, oth, keep, engine.n_decode_threads(conf.nproc))


def usage(fp=sys.stdout, d=None):
    d = d or Config().defaults
    rows = [
        "",
        "Version: %s" % VERSION,
        "Usage:   %s %s <options>" % (APP, COMMAND),
        "",
        "Options:",
        "  -s, --sam FILE         Comma separated indexed sam/bam/cram file.",
        "  -S, --samList FILE     A list file containing bam files, each per line.",
        "  -b, --barcode FILE     A plain file listing all effective cell barcode.",
        "  -i, --sampleList FILE  A list file containing sample IDs, each per line.",
        "  -I, --sampleIDs STR    Comma separated sample IDs.",
        "  -P, --snpvcf FILE      Candidate SNPs: a VCF (CHROM POS ID REF ALT; no genotype needed) or a TSV",
        "                         with a header line and the columns chrom, pos, ref, alt.  Without -P the",
        "                         sites are discovered from the reads on the --chrom contigs.",
        "  -O, --outdir DIR       Output directory: cellSNP.samples.tsv, cellSNP.tag.{AD,DP,OTH}.mtx,",
        "                         cellSNP.base.vcf.gz.",
        "  -h, --help             Print this message and exit.",
        "",
        "Optional arguments:",
        "  -p, --ncores INT       Number of processes [%d]" % d.NPROC,
        "      --cellTAG STR      Tag for cell barcodes, set to None when using sample IDs [%s]" % d.CELL_TAG,
        "      --UMItag STR       Tag for UMI, set to None when reads only [%s]" % d.UMI_TAG,
        "  -D, --debug INT        Used by developer for debugging [%d]" % d.DEBUG,
        "      --chrom STR        Contigs to discover sites on, comma separated; without -P only [1,...,22]",
        "",
        "SNP filtering:",
        "  --minCOUNT INT         Minimum aggregated count of a SNP [%d with -P, %d without]" % (
            MIN_COUNT, DISCOVER_MIN_COUNT),
        "  --minMAF FLOAT         Minimum minor allele fraction of a SNP [%s with -P, %s without]" % (
            MIN_MAF, DISCOVER_MIN_MAF),
        "",
        "Read filtering:",
        "  --inclFLAG INT          Required flags: skip reads with all mask bits unset [%d]" % d.INCL_FLAG,
        "  --exclFLAG INT          Filter flags: skip reads with any mask bits set [%d" % d.EXCL_FLAG_UMI,
        "                          (when use UMI) or %d (otherwise)]" % d.EXCL_FLAG_XUMI,
        "  --minLEN INT            Minimum mapped length for read filtering [%d]" % d.MIN_LEN,
        "  --minMAPQ INT           Minimum MAPQ for read filtering [%d]" % d.MIN_MAPQ,
        "  --countORPHAN           If use, do not skip anomalous read pairs.",
        "",
        "B200 notes: input must be coordinate-sorted BAM (a .bai is used when present; SAM/CRAM are not decoded);",
        "  -p sets the host BGZF/BAM decode threads; counting runs on the GPU (no CPU fallback).",
        "  A UMI is counted once per SNP and cell, with the allele of its first read in file order.",
        "  Without -P, REF and ALT of a site are its two most frequent bases among A, C, G, T (ties in that",
        "  order); a site is kept if ALT >= 1 and it passes --minCOUNT / --minMAF.",
        "",
    ]
    fp.write("\n".join(rows) + "\n")


_LONG = ["sam=", "samList=", "barcode=", "sampleList=", "sampleIDs=", "snpvcf=", "outdir=", "help", "ncores=",
         "cellTAG=", "UMItag=", "debug=", "minCOUNT=", "minMAF=", "inclFLAG=", "exclFLAG=", "minLEN=", "minMAPQ=",
         "countORPHAN", "chrom="]


def parse_args(argv, conf):
    """Options of argv[2:] into conf; None if ok, else the invalid option.  Long options are case-insensitive."""
    opts, _args = getopt.getopt(argv[2:], "-s:-S:-b:-i:-I:-P:-O:-h-p:-D:", _LONG)
    setters = {
        "-s": ("sam_fn", str), "--sam": ("sam_fn", str),
        "-S": ("sam_list_fn", str), "--samlist": ("sam_list_fn", str),
        "-b": ("barcode_fn", str), "--barcode": ("barcode_fn", str),
        "-i": ("sample_id_fn", str), "--samplelist": ("sample_id_fn", str),
        "-I": ("sample_id_str", str), "--sampleids": ("sample_id_str", str),
        "-P": ("snp_fn", str), "--snpvcf": ("snp_fn", str),
        "-O": ("out_dir", str), "--outdir": ("out_dir", str),
        "-p": ("nproc", int), "--ncores": ("nproc", int),
        "--celltag": ("cell_tag", str), "--umitag": ("umi_tag", str),
        "-D": ("debug", int), "--debug": ("debug", int),
        "--mincount": ("min_count", int), "--minmaf": ("min_maf", float),
        "--inclflag": ("incl_flag", int), "--exclflag": ("excl_flag", int),
        "--minlen": ("min_len", int), "--minmapq": ("min_mapq", float),
        "--chrom": ("chrom", str),
    }
    for op, val in opts:
        if len(op) > 2:
            op = op.lower()
        if op in ("-h", "--help"):
            return op
        elif op == "--countorphan":
            conf.no_orphan = False
        elif op in setters:
            attr, conv = setters[op]
            setattr(conf, attr, conv(val))
        else:
            return op
    return None


def pileup_main(argv):
    """Command-line interface; returns 0 on success, -1 otherwise."""
    conf = Config()
    conf.min_count = conf.min_maf = conf.chrom = None      # defaults depend on the mode (filter_defaults)
    if len(argv) <= 2:
        usage(sys.stdout, conf.defaults)
        sys.exit(0)
    conf.argv = argv.copy()
    init_logging(stream=sys.stderr)
    bad = parse_args(argv, conf)
    if bad in ("-h", "--help"):
        usage(sys.stdout, conf.defaults)
        sys.exit(0)
    if bad is not None:
        error("invalid option: '%s'." % bad)
        return -1
    if not conf.snp_fn and not conf.chrom:
        conf.chrom = DEFAULT_CHROMS
    return afc.afc_run(conf, core=pileup_core)
