"""Input loaders of the baf feature counter (behaviour of xcltk/baf/fc/utils.py:12-193)."""

import sys

from ...utils.zfile import zopen
from .gfeature import SNP, SNPSet, BlockRegion


def load_region_from_txt(fn, sep="\t", verbose=False):
    """Header-less TSV chrom/start/end(1-based inclusive)/name -> [BlockRegion] or None."""
    func = "load_region_from_txt"
    if verbose:
        sys.stderr.write("[I::%s] start to load regions from file '%s' ...\n" % (func, fn))
    regs = []
    with zopen(fn, "rt") as fp:
        for nl, line in enumerate(fp, 1):
            parts = line.rstrip().split(sep)
            if len(parts) < 4:
                if verbose:
                    sys.stderr.write("[E::%s] too few columns of line %d.\n" % (func, nl))
                return None
            regs.append(BlockRegion(parts[0], int(parts[1]), int(parts[2]) + 1, parts[3]))
    return regs


def _warn(verbose, func, msg, nl):
    if verbose:
        sys.stderr.write("[W::%s] %s line %d.\n" % (func, msg, nl))


def _valid_base(b):
    return len(b) == 1 and b in "ACGTN"


def _add_snp(snp_set, chrom, pos, ref, alt, a1, a2, verbose, func, nl):
    """Shared tail of both loaders: only 0|1 / 1|0 genotypes are phased het SNPs.  a1 = a2 = None: a candidate site
    without genotype, kept as 0|1 with its CHROM text as given (`chrom_text`)."""
    if a1 is None and a2 is None:
        snp = SNP(chrom=chrom, pos=int(pos), ref=ref, alt=alt, ref_idx=0, alt_idx=1)
        snp.chrom_text = chrom
        snp_set.add(snp)
    elif (a1 == "0" and a2 == "1") or (a1 == "1" and a2 == "0"):
        snp_set.add(SNP(chrom=chrom, pos=int(pos), ref=ref, alt=alt, ref_idx=int(a1), alt_idx=int(a2)))
    else:
        _warn(verbose, func, "invalid GT of", nl)


def load_snp_from_tsv(fn, verbose=False, sites=False):
    """TSV with a header line: chrom pos ref alt ref_hap alt_hap (utils.py:51-110).  sites: candidate sites, only
    the first four columns are used."""
    func = "load_snp_from_tsv"
    if verbose:
        sys.stderr.write("[I::%s] start to load SNPs from tsv '%s' ...\n" % (func, fn))
    snp_set = SNPSet()
    with zopen(fn, "rt") as fp:
        for nl, line in enumerate(fp, 1):
            if nl == 1:
                continue
            parts = line.rstrip().split("\t")
            if len(parts) < (4 if sites else 6):
                _warn(verbose, func, "too few columns of", nl)
                continue
            ref, alt = parts[2].upper(), parts[3].upper()
            if not _valid_base(ref):
                _warn(verbose, func, "invalid REF base of", nl)
                continue
            if not _valid_base(alt):
                _warn(verbose, func, "invalid ALT base of", nl)
                continue
            a1, a2 = (None, None) if sites else (parts[4], parts[5])
            _add_snp(snp_set, parts[0], parts[1], ref, alt, a1, a2, verbose, func, nl)
    return snp_set


def load_snp_from_vcf(fn, verbose=False, sites=False):
    """Phased VCF, GT of the first sample (utils.py:114-193).  sites: candidate sites, CHROM POS ID REF ALT only (no
    GT, no FORMAT)."""
    func = "load_snp_from_vcf"
    if verbose:
        sys.stderr.write("[I::%s] start to load SNPs from vcf '%s' ...\n" % (func, fn))
    snp_set = SNPSet()
    with zopen(fn, "rt") as fp:
        for nl, line in enumerate(fp, 1):
            if line[0] in ("#", "\n"):
                continue
            parts = line.rstrip().split("\t")
            if len(parts) < (5 if sites else 10):
                _warn(verbose, func, "too few columns of", nl)
                continue
            ref, alt = parts[3].upper(), parts[4].upper()
            if not _valid_base(ref):
                _warn(verbose, func, "invalid REF base of", nl)
                continue
            if not _valid_base(alt):
                _warn(verbose, func, "invalid ALT base of", nl)
                continue
            if sites:
                _add_snp(snp_set, parts[0], parts[1], ref, alt, None, None, verbose, func, nl)
                continue
            fields = parts[8].split(":")
            if "GT" not in fields:
                _warn(verbose, func, "GT not in", nl)
                continue
            values = parts[9].split(":")
            if len(values) != len(fields):
                _warn(verbose, func, "len(fields) != len(values) in", nl)
                continue
            gt = values[fields.index("GT")]
            sep = "|" if "|" in gt else ("/" if "/" in gt else "")
            if not sep:
                _warn(verbose, func, "invalid delimiter of", nl)
                continue
            a1, a2 = gt.split(sep)[:2]
            _add_snp(snp_set, parts[0], parts[1], ref, alt, a1, a2, verbose, func, nl)
    return snp_set
