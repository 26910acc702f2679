"""The CPU oracle on CIGAR operators that the synthetic and golden inputs never carry: leading S and H, `=` / `X`
blocks, P, zero-length ops, an I right before / after a position, D and N over it.  The expected values are written
by hand from the reference's own definitions, not from any kernel:
  basefc: m = len([p for p in read.positions if s <= p <= e]), n = len(read.positions)   (rdr/fc/core.py:32-62)
  baf:    allele = get_query_bases(read)[read.positions.index(snp.pos - 1)]                (baf/fc/mcount.py:39-60)
read.positions are the reference positions of M / = / X bases; get_query_bases lists the query bases of those
same operators in order.  The GPU tests compare the kernels with the oracle, so this pins what they compare with."""

import numpy as np
import pytest

from recsets import CIGAR_PANEL, cigar_panel

LABELS = [c[0] for c in CIGAR_PANEL]
COL = {lab: k for k, lab in enumerate(LABELS)}

# features, 0-based [beg, end)
FEATS = {"F0": (100, 120), "F1": (103, 110), "F2": (110, 115), "F3": (200, 210), "F4": (108, 113)}
# read.positions of each read, by hand from its CIGAR
POSITIONS = {
    "R0": list(range(100, 120)),                                       # 5S 10M 3I 10M
    "R1": list(range(100, 108)) + list(range(112, 120)),               # 4H 3S 6= 2X 4D 8M 2H
    "R2": list(range(100, 120)),                                       # 10M 2P 3I 0M 10M
    "R3": list(range(102, 107)) + list(range(207, 212)),               # 0M 5= 100N 5X 5S
    "R5": list(range(104, 114)),                                       # no CIGAR: one M block
    "R4": list(range(105, 112)) + list(range(113, 118)),               # 3M 2I 4X 1D 5=
}
# m per (read, feature), by hand; a read that does not reach a feature is not fetched for it (m = 0 then too)
M_INCL = {
    "R0": {"F0": 20, "F1": 7, "F2": 5, "F3": 0, "F4": 5},
    "R1": {"F0": 16, "F1": 5, "F2": 3, "F3": 0, "F4": 1},
    "R2": {"F0": 20, "F1": 7, "F2": 5, "F3": 0, "F4": 5},
    "R3": {"F0": 5, "F1": 4, "F2": 0, "F3": 3, "F4": 0},
    "R5": {"F0": 10, "F1": 6, "F2": 4, "F3": 0, "F4": 5},
    "R4": {"F0": 12, "F1": 5, "F2": 4, "F3": 0, "F4": 4},
}
SNPS = [105, 106, 107, 108, 109, 110, 112, 150, 207, 211]
# allele per (read, SNP) for every read whose [pos, end) holds the SNP: a letter, "N", "other" (= or IUPAC),
# or None (the SNP falls in a D / N: the read claims its UMI but counts nowhere)
ALLELE = {
    "R0": {105: "A", 106: "A", 107: "A", 108: "A", 109: "T", 110: "G", 112: "A"},
    "R1": {105: "C", 106: "G", 107: "T", 108: None, 109: None, 110: None, 112: "C"},
    "R2": {105: "A", 106: "A", 107: "A", 108: "A", 109: "G", 110: "C", 112: "A"},
    "R3": {105: "T", 106: "A", 107: None, 108: None, 109: None, 110: None, 112: None, 150: None, 207: "C",
           211: "G"},
    "R5": {105: "C", 106: "N", 107: "other", 108: "other", 109: "G", 110: "T", 112: "C"},
    "R4": {105: "A", 106: "C", 107: "G", 108: "C", 109: "A", 110: "G", 112: None},
}


class Conf(object):
    min_mapq, min_len, min_include = 0, 1, 1
    incl_flag, excl_flag, no_orphan = 0, 0, False

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return True

    def use_umi(self):
        return True


def test_hand_tables_agree_with_each_other():
    """M_INCL is the count of POSITIONS inside each feature (the tables above are one definition)."""
    for lab, ps in POSITIONS.items():
        for f, (b, e) in FEATS.items():
            assert M_INCL[lab][f] == sum(1 for p in ps if b <= p < e), (lab, f)


def _basefc(reads, ck, conf):
    from oracle import oracle
    names = sorted(FEATS)
    gid = np.zeros(len(names), np.int32)
    beg = np.array([FEATS[f][0] for f in names], np.int32)
    end = np.array([FEATS[f][1] for f in names], np.int32)
    row, col, val = oracle.basefc(reads, gid, beg, end, ck, len(ck), oracle.params(conf), 1)
    assert np.all(val == 1)                     # one UMI per cell
    return {(names[r], LABELS[c]) for r, c in zip(row.tolist(), col.tolist())}


@pytest.mark.parametrize("k", range(1, 22))
def test_oracle_basefc_included_length_integer_threshold(k):
    """min_include = k (an int): the pair counts iff m >= k -- over k this reads m back exactly."""
    reads, ck = cigar_panel()
    got = _basefc(reads, ck, Conf(min_include=k))
    exp = {(f, lab) for lab in LABELS for f in FEATS if M_INCL[lab][f] >= k}
    assert got == exp


@pytest.mark.parametrize("frac", [0.25, 0.3, 0.5, 0.7])
def test_oracle_basefc_included_fraction(frac):
    """0 < min_include < 1: the pair counts iff m / len(read.positions) >= min_include."""
    reads, ck = cigar_panel()
    got = _basefc(reads, ck, Conf(min_include=frac))
    exp = {(f, lab) for lab in LABELS for f in FEATS
           if M_INCL[lab][f] > 0 and M_INCL[lab][f] / float(len(POSITIONS[lab])) >= frac}
    assert got == exp


def test_oracle_min_len_counts_aligned_bases_only():
    """min_len compares len(read.positions): S, H, I and P bases do not count."""
    reads, ck = cigar_panel()
    for min_len in (10, 11, 13, 17, 21):
        got = _basefc(reads, ck, Conf(min_include=1, min_len=min_len))
        exp = {(f, lab) for lab in LABELS for f in FEATS if M_INCL[lab][f] >= 1 and len(POSITIONS[lab]) >= min_len}
        assert got == exp, min_len


def test_oracle_baf_allele_is_the_query_base_of_the_aligned_position():
    """One region per SNP, REF 'N' and ALT each of A/C/G/T in turn: the read's allele is the ALT for which it
    lands in AD; 'N' lands in DP only (REF); '=' and IUPAC codes land in OTH; a D / N over the SNP nowhere."""
    from oracle import oracle
    reads, ck = cigar_panel()
    n_snp = len(SNPS)
    gid = np.zeros(n_snp, np.int32)
    pos = np.array(SNPS, np.int32)
    reg_ptr = np.arange(n_snp + 1, dtype=np.int64)
    reg_snp = np.arange(n_snp, dtype=np.int32)
    got = {}
    for alt in "ACGT":
        ad, dp, oth = oracle.baf(reads, gid, pos, "N" * n_snp, alt * n_snp, np.zeros(n_snp), np.ones(n_snp), reg_ptr,
                                 reg_snp, ck, len(ck), oracle.params(Conf(min_include=0)), 0, 0.0, True, 1)
        ad_s = {(r, c) for r, c in zip(ad[0].tolist(), ad[1].tolist())}
        dp_s = {(r, c) for r, c in zip(dp[0].tolist(), dp[1].tolist())}
        oth_s = {(r, c) for r, c in zip(oth[0].tolist(), oth[1].tolist())}
        assert ad_s <= dp_s and not (dp_s & oth_s)
        assert np.all(ad[2] == 1) and np.all(dp[2] == 1) and np.all(oth[2] == 1)
        for key in ad_s:
            got.setdefault(key, set()).add(alt)
        for key in dp_s - ad_s:
            got.setdefault(key, set()).add("N")
        for key in oth_s:
            got.setdefault(key, set()).add("other")
    exp = {}
    for lab, al in ALLELE.items():
        for snp, a in al.items():
            if a is None:
                continue
            key = (SNPS.index(snp), COL[lab])
            # a letter is AD in its own pass and OTH (neither REF nor ALT) in the other three
            exp[key] = {a} if a in ("N", "other") else {a, "other"}
    assert got == exp
