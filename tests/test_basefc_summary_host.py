"""basefc's read-assignment summary on the CPU: the oracle (tests/summary_oracle.c) pinned on a hand-built batch whose
table is written out below record by record, the summary.tsv writer, the `--summary` option and fc_wrapper's
signature, and the `own` ranges of a library split by byte ranges."""

import inspect
import io

import numpy as np

import summary_oracle
from recsets import M, N, build, cell_keys, umi_keys
from xcltk_b200 import lib
from xcltk_b200.lib import XG_KEY_EMPTY, XG_KEY_NONE
from xcltk_b200.rdr.fc import main as rdr_main
from xcltk_b200.rdr.fc.config import Config


class Conf(object):
    min_mapq, min_len, min_include = 20, 10, 0.5
    incl_flag, excl_flag, no_orphan = 0, 772, True
    barcodes, umi = True, True

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return self.barcodes

    def use_umi(self):
        return self.umi


# features: F0 [100, 200), F1 = F2 = [300, 310) (duplicates), one on a contig without reads, one never fetched
FEATS = (np.array([0, 0, 0, 1, -1]), np.array([100, 300, 300, 0, 0]), np.array([200, 310, 310, 100, 0]))
A, B, U = cell_keys(3)
# (pos, end or CIGAR, cell, UMI, flag, mapq, row, fate): rows 0 = A, 1 = B, 2 = __no_cell; fate None = out of range
RECS = [
    (50, 100, A, 1, 0, 60, None, None),                      # ends at F0's beg
    (90, 120, A, 2, 0, 10, 0, "mapq"),
    (120, 140, A, 3, 4, 60, 0, "flag"),                      # UNMAP: excl_flag
    (120, 140, B, 4, 1, 60, 1, "flag"),                      # paired, not proper: orphan
    (130, 150, B, XG_KEY_NONE, 0, 60, 1, "no_umi"),
    (130, 150, B, XG_KEY_EMPTY, 0, 60, 1, "no_umi"),
    (140, 145, A, 7, 0, 60, 0, "short"),                     # 5 aligned bases < min_len
    (150, 170, B, 8, 0, 60, 1, "one_feature"),
    (180, [(M, 10), (N, 200), (M, 10)], A, 9, 0, 60, 0, "one_feature"),   # F0 10 / 20; F1, F2 through the N gap
    (190, 220, A, 10, 0, 60, 0, "not_included"),             # F0 10 / 30 < 0.5
    (290, [(M, 5), (N, 30), (M, 10)], A, 11, 0, 60, 0, "not_included"),  # F1, F2 overlapped by the N gap only
    (300, 310, U, 12, 0, 60, 2, "multi_feature"),            # unlisted barcode
    (302, 312, XG_KEY_NONE, 13, 0, 60, 2, "multi_feature"),  # no cell tag
    (305, 325, B, 14, 0, 60, 1, "not_included"),             # 5 / 20
    (500, 600, A, 15, 0, 60, None, None),                    # no feature there
]


def hand_batch():
    uk = umi_keys(20)
    pos = [r[0] for r in RECS]
    ops = [r[1] if isinstance(r[1], list) else None for r in RECS]
    end = [r[1] if isinstance(r[1], int) else 0 for r in RECS]
    umi = [r[3] if r[3] in (XG_KEY_NONE, XG_KEY_EMPTY) else int(uk[r[3]]) for r in RECS]
    return build(pos, [r[2] for r in RECS], np.array(umi, dtype=np.uint64), [(0, 0, 0, len(RECS))], end=end, ops=ops,
                 flag=[r[4] for r in RECS], mapq=[r[5] for r in RECS])


def expected(rows=3, row_of=None):
    t = np.zeros((rows, 7), dtype=np.int64)
    for r in RECS:
        if r[7] is not None:
            t[r[6] if row_of is None else row_of(r), summary_oracle.FATES.index(r[7])] += 1
    return t


def test_oracle_on_hand_built_batch():
    reads = hand_batch()
    got = summary_oracle.summary(reads, *FEATS, np.array([A, B], dtype=np.uint64), 2, summary_oracle.params(Conf()))
    assert got.tolist() == expected().tolist()
    assert got.tolist() == [[1, 1, 0, 1, 2, 1, 0], [0, 1, 2, 0, 1, 1, 0], [0, 0, 0, 0, 0, 0, 2]]


def test_oracle_sample_mode_without_umis():
    """Sample-ID mode: every record is the BAM's column and __no_cell stays 0; without a UMI tag the records with no
    or an empty UMI go on to the include test (both lie inside F0)."""
    conf = Conf(barcodes=False, umi=False)
    got = summary_oracle.summary(hand_batch(), *FEATS, None, 1, summary_oracle.params(conf))
    assert got.tolist() == [[1, 2, 0, 1, 3, 4, 2], [0] * 7]


def test_oracle_own_range_and_length_mode():
    """own keeps the records whose (gid, pos) lies in [lo, hi); min_include 20 is a length: F0 [150, 170) passes with
    20 bases, [180, 190) + [390, 400) does not (10)."""
    conf = Conf(min_include=20)
    keys = np.array([A, B], dtype=np.uint64)
    got = summary_oracle.summary(hand_batch(), *FEATS, keys, 2, summary_oracle.params(conf), own=(0, 150, 0, 181))
    assert got.tolist() == [[0, 0, 0, 0, 1, 0, 0], [0, 0, 0, 0, 0, 1, 0], [0] * 7]


def test_summary_tsv_format(tmp_path):
    p = str(tmp_path / "summary.tsv")
    rdr_main.write_summary(p, ["AAACCTG-1", "TTTGGTA-1"], [[1, 2, 3, 4, 5, 6, 7], [0] * 7, [0, 0, 0, 0, 0, 10, 0]])
    assert open(p, "rb").read() == (
        b"cell\ttotal\tmapq\tflag\tno_umi\tshort\tnot_included\tone_feature\tmulti_feature\n"
        b"AAACCTG-1\t28\t1\t2\t3\t4\t5\t6\t7\n"
        b"TTTGGTA-1\t0\t0\t0\t0\t0\t0\t0\t0\n"
        b"__no_cell\t10\t0\t0\t0\t0\t0\t10\t0\n")
    assert lib.SUMMARY_FATES == summary_oracle.FATES


def test_summary_option_is_parsed(monkeypatch):
    seen = []
    monkeypatch.setattr(rdr_main, "fc_run", lambda conf: seen.append(conf) or 0)
    assert rdr_main.fc_main(["xcltk", "basefc", "-s", "a.bam", "--summary"]) == 0
    assert rdr_main.fc_main(["xcltk", "basefc", "-s", "a.bam"]) == 0
    assert [c.summary for c in seen] == [True, False]
    fp = io.StringIO()
    rdr_main.usage(fp, Config().defaults)
    assert "      --summary          Also write summary.tsv" in fp.getvalue()


def test_fc_wrapper_signature_gains_summary_last():
    params = list(inspect.signature(rdr_main.fc_wrapper).parameters.values())
    assert [p.name for p in params] == [
        "sam_fn", "barcode_fn", "region_fn", "out_dir", "sam_list_fn", "sample_ids", "sample_id_fn", "debug_level",
        "ncores", "cell_tag", "umi_tag", "output_all_reg", "min_mapq", "min_len", "min_include", "incl_flag",
        "excl_flag", "no_orphan", "summary"]
    assert params[-1].default is False


def test_own_ranges_follow_the_gids_of_a_cut():
    neg = -(1 << 31)
    tid_map = [0, 1, -1, 2, 4, 3]                 # tid -> gid: tid 2 has no features, tids 4 / 5 swap their gids
    assert rdr_main.own_ranges((-1, -1), (1, 500), tid_map) == [(0, neg, 1, 500)]
    assert rdr_main.own_ranges((1, 500), (3, 7), tid_map) == [(1, 500, 2, 7)]
    assert rdr_main.own_ranges((3, 7), (1 << 40, 0), tid_map) == [(2, 7, 3, neg), (4, neg, 5, neg), (3, neg, 4, neg)]
    assert rdr_main.own_ranges((2, 10), (2, 99), tid_map) == []
