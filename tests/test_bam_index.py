"""The .bai reader (decode.cpp: xg_bam_index_open / xg_bam_index_ranges) against a brute force over the records:
for any interval, the byte ranges it gives hold the BGZF blocks of every record that overlaps the interval.  The
indexes come from a BAI writer built from SAMv1 section 5.2 (tests/bai.py); an index that cannot be trusted is
ignored with one warning and the BAM is read whole."""

import logging
import os
import random
import shutil

import numpy as np
import pytest

import bai

CONTIGS = [("chr1", 3000000), ("chr2", 1500000), ("chrE", 900000), ("chr3", 2200000), ("chrM", 16000)]


def _records(seed, n):
    """Sorted records over CONTIGS (chrE holds none): short reads, spliced reads with >= 500 kb N gaps (high bins),
    reads on 16 kb window edges, unmapped-flag reads with a position, and a tail of unplaced reads."""
    rng = random.Random(seed)
    recs = []
    for tid, (name, length) in enumerate(CONTIGS):
        if name == "chrE":
            continue
        pos = rng.randrange(0, 3000)
        k = 0
        while pos < length - 700000 or (length < 700000 and pos < length - 200):
            r = rng.random()
            if r < 0.02 and length > 1000000:
                cig = [(0, 40), (3, rng.randrange(500000, 650000)), (0, 51)]
            elif r < 0.05:
                cig = [(0, 30), (2, 5), (0, 20), (1, 4), (0, 37)]
            else:
                cig = [(0, 91)]
            flag = 4 if rng.random() < 0.01 else rng.choice([0, 16])
            seq = "".join(rng.choice("ACGT") for _ in range(sum(l for op, l in cig if op in (0, 1, 4, 7, 8))))
            recs.append(("q%d_%d" % (tid, k), flag, tid, pos, 60, cig, seq,
                         [("CB", "Z", "ACGTACGT-1"), ("UB", "Z", "AAAA")]))
            k += 1
            step = rng.choice([0, 1, 7, 30, 60, 300]) if rng.random() < 0.999 else rng.randrange(10000, 90000)
            if rng.random() < 0.03:                   # land on a 16 kb window edge
                step = ((pos >> 14) + 1 << 14) - pos - rng.choice([0, 1])
            pos += max(0, step)
            if k >= n // 4:
                break
    recs += [("u%d" % i, 4, -1, -1, 0, [], "ACGT", []) for i in range(5)]
    return recs


@pytest.fixture(scope="module")
def bams(tmp_path_factory):
    """{layout: path}: synth.write_bam's htslib layout, and the same reads through xg_write_bam"""
    from xcltk_b200 import lib, synth
    d = tmp_path_factory.mktemp("bai")
    p1 = str(d / "synth.bam")
    synth.write_bam(p1, CONTIGS, _records(5, 40000), level=1)
    ks = lib.KeySpace()
    h = lib.decode_bams([p1], [np.arange(len(CONTIGS), dtype=np.int32)], "CB", "UB", True, ks, 2)
    p2 = str(d / "xgw.bam")
    lib.write_bam(p2, h, CONTIGS, ks, level=1)
    h.close()
    return {"synth": p1, "xg_write_bam": p2}


MERGE_GAP = 256 << 10           # XG_BAM_INDEX_MERGE_GAP


def _covered(ranges, vb, ve):
    """the record [vb, ve) (virtual offsets) lies in one of the ranges (virtual offset of the first record, file
    offset after the last block)"""
    return any(lo <= vb and ((ve - 1) >> 16) < hi for lo, hi in ranges)


def _check_intervals(path, idx, recs, intervals, index):
    tid = np.array([t for t, _b, _e in intervals], dtype=np.int32)
    beg = np.array([b for _t, b, _e in intervals], dtype=np.int64)
    end = np.array([e for _t, _b, e in intervals], dtype=np.int64)
    size = os.path.getsize(path)
    block_starts = {c for c, _u in bai.bgzf_blocks(path)} | {size}
    record_starts = {r[4] for r in recs}
    narrower = 0
    for i in range(len(intervals)):                           # each interval on its own ...
        rng_ = idx.ranges(tid[i:i + 1], beg[i:i + 1], end[i:i + 1])
        assert rng_ == bai.query_ranges(path, index, intervals[i:i + 1], MERGE_GAP)
        for lo, hi in rng_:                                    # a range starts at a record and ends at a block start
            assert lo in record_starts and (lo >> 16) in block_starts and hi in block_starts and (lo >> 16) < hi
        assert all(a[1] + MERGE_GAP < (b[0] >> 16) for a, b in zip(rng_, rng_[1:]))   # ascending, merged
        for t, p, e, _f, vb, ve in recs:
            if t == tid[i] and p < end[i] and e > max(0, beg[i]) and end[i] > beg[i]:
                assert _covered(rng_, vb, ve), (intervals[i], p, e)
        unfiltered = bai.query_ranges(path, index, intervals[i:i + 1], MERGE_GAP, linear=False)
        narrower += sum(h - (l >> 16) for l, h in rng_) < sum(h - (l >> 16) for l, h in unfiltered)
    whole = idx.ranges(tid, beg, end)                          # ... and all of them at once
    assert whole == bai.query_ranges(path, index, intervals, MERGE_GAP)
    for t, p, e, _f, vb, ve in recs:
        hit = any(t == tid[i] and p < end[i] and e > max(0, beg[i]) and end[i] > beg[i] for i in range(len(intervals)))
        if hit:
            assert _covered(whole, vb, ve)
    return narrower


@pytest.mark.parametrize("layout", ["synth", "xg_write_bam"])
def test_ranges_hold_every_overlapping_record(bams, layout):
    from xcltk_b200 import lib
    path = bams[layout]
    n_ref, recs, index = bai.index_bam(path)
    idx = lib.BamIndex.open(path)
    assert idx is not None and idx.n_ref() == n_ref
    rng = random.Random(11)
    iv = []
    for _ in range(120):                                       # random intervals of every size
        t = rng.randrange(len(CONTIGS))
        b = rng.randrange(0, CONTIGS[t][1])
        iv.append((t, b, b + rng.choice([1, 2, 50, 1000, 16384, 300000, 2000000])))
    for k in (1, 2, 17, 60, 61):                               # 16 kb window edges
        e = k << 14
        iv += [(0, e - 1, e), (0, e, e + 1), (0, e - 1, e + 1), (3, e, e + 16384), (1, e - 100, e)]
    for t in range(len(CONTIGS)):                              # first and last records of a contig
        on = [r for r in recs if r[0] == t]
        if on:
            iv += [(t, on[0][1], on[0][1] + 1), (t, 0, 1), (t, on[-1][1], on[-1][1] + 1), (t, on[-1][2] - 1, on[-1][2])]
    iv += [(2, 0, 900000), (4, 0, 16000)]                      # the empty contig, and all of chrM
    iv += [(-1, 0, 100), (len(CONTIGS), 0, 100), (99, 0, 1 << 29), (0, 5000, 5000), (0, 9000, 10), (0, -50, 200)]
    narrower = _check_intervals(path, idx, recs, iv, index)
    assert narrower >= 20                                      # the linear index drops chunks for many of them
    assert idx.ranges([2], [0], [900000]) == []                # nothing on the empty contig
    assert idx.ranges([-1, 99, 0], [0, 0, 7], [10, 10, 7]) == []
    # the whole genome merges to one range, from the first record's block to the end of the last one
    allr = idx.ranges(list(range(len(CONTIGS))), [0] * len(CONTIGS), [c[1] for c in CONTIGS])
    placed = [r for r in recs if r[0] >= 0]
    assert allr == [(placed[0][4], os.path.getsize(path) - 28)]
    idx.close()


def test_long_spliced_reads_reach_their_far_windows(bams):
    """a read whose N gap spans >= 500 kb sits in a high-level bin: an interval inside its far exon still gets it"""
    from xcltk_b200 import lib
    path = bams["synth"]
    _n, recs, index = bai.index_bam(path)
    idx = lib.BamIndex.open(path)
    far = [r for r in recs if r[0] >= 0 and r[2] - r[1] > 500000]
    assert len(far) > 10
    iv = [(t, e - 10, e) for t, _p, e, _f, _vb, _ve in far[:40]]
    _check_intervals(path, idx, recs, iv, index)
    idx.close()


@pytest.mark.parametrize("layout", ["synth", "xg_write_bam"])
def test_writer_and_reader_agree_on_every_bin_and_linear_entry(bams, layout, tmp_path):
    from xcltk_b200 import lib
    path = str(tmp_path / "x.bam")
    shutil.copy(bams[layout], path)
    n_ref, _recs, index = bai.index_bam(path)
    idx = lib.BamIndex.open(path)
    assert idx.n_ref() == n_ref
    n_bins = 0
    for t in range(n_ref):
        bins, lin = idx.ref(t)
        exp_bins, exp_lin, _counts, _span = index[t]
        assert bins == {b: list(c) for b, c in exp_bins.items()}          # the pseudo-bin is left out
        assert [int(v) for v in lin] == exp_lin
        n_bins += len(bins)
    assert n_bins > 100
    assert any(b < 73 for t in range(n_ref) for b in idx.ref(t)[0])       # bins of the 1 Mb level and above
    idx.close()


def test_index_next_to_the_bam_without_its_suffix(bams, tmp_path):
    from xcltk_b200 import lib
    path = str(tmp_path / "y.bam")
    shutil.copy(bams["synth"], path)
    assert lib.BamIndex.open(path) is None                     # no index: the file is read whole
    with open(str(tmp_path / "y.bam.csi"), "wb") as fp:        # a .csi is not read
        fp.write(b"CSI\1")
    assert lib.BamIndex.open(path) is None
    bai.index_bam(path, str(tmp_path / "y.bai"))
    idx = lib.BamIndex.open(path)
    assert idx is not None and idx.n_ref() == len(CONTIGS)
    idx.close()


def _bad_index(case, path, tmp_path, other):
    n_ref, recs = bai.bam_records(path)
    if case == "n_ref":
        bai.write_bai(path + ".bai", n_ref, recs, extra_refs=1)
    elif case == "truncated":
        bai.write_bai(path + ".bai", n_ref, recs)
        with open(path + ".bai", "rb") as fp:
            data = fp.read()
        with open(path + ".bai", "wb") as fp:
            fp.write(data[:len(data) // 2])
    elif case == "past_eof":
        size = os.path.getsize(path)
        recs = [r[:4] + ((size + 10) << 16, (size + 20) << 16) if i == len(recs) // 2 else r for i, r in enumerate(recs)]
        bai.write_bai(path + ".bai", n_ref, recs)
    elif case == "older":
        bai.write_bai(path + ".bai", n_ref, recs)
        st = os.stat(path)
        os.utime(path + ".bai", (st.st_atime, st.st_mtime - 100))
    elif case == "other_bam":
        n2, recs2 = bai.bam_records(other)
        bai.write_bai(path + ".bai", n2, recs2)
        st = os.stat(path)
        os.utime(path + ".bai", (st.st_atime, st.st_mtime + 10))


@pytest.mark.parametrize("case", ["n_ref", "truncated", "past_eof", "older", "other_bam"])
def test_an_index_that_cannot_be_trusted_is_ignored_with_a_warning(bams, tmp_path, caplog, case):
    from xcltk_b200 import engine, lib
    from xcltk_b200.utils.sam import build_tid_maps
    path = str(tmp_path / "z.bam")
    shutil.copy(bams["synth"], path)
    _bad_index(case, path, tmp_path, bams["xg_write_bam"])
    names = [c[0] for c in CONTIGS]
    gid_of, tid_maps = build_tid_maps([lib.bam_references(path)], names)
    units = (["chr1", "chr3", "chr2"], [100000, 50000, 0], [400000, 900000, 1400000])
    with caplog.at_level(logging.WARNING, logger="xcltk_b200.engine"):
        got = engine.index_ranges([path], gid_of, tid_maps, units)
    assert got == [None]
    warned = [r for r in caplog.records if r.levelno == logging.WARNING]
    assert len(warned) == 1 and "whole" in warned[0].getMessage()


def test_a_good_index_gives_ranges_per_bam(bams, tmp_path, caplog):
    """one BAM indexed, one not: ranges for the first, the whole file for the second, no warning"""
    from xcltk_b200 import engine, lib
    from xcltk_b200.utils.sam import build_tid_maps
    a, b = str(tmp_path / "a.bam"), str(tmp_path / "b.bam")
    shutil.copy(bams["synth"], a)
    shutil.copy(bams["xg_write_bam"], b)
    bai.index_bam(a)
    names = ["1", "3"]                                         # resolved with the 'chr' toggle
    gid_of, tid_maps = build_tid_maps([lib.bam_references(a), lib.bam_references(b)], names)
    with caplog.at_level(logging.WARNING, logger="xcltk_b200.engine"):
        got = engine.index_ranges([a, b], gid_of, tid_maps, (["3", None, "7"], [10, 0, 0], [20000, 10, 10]))
    assert not [r for r in caplog.records if r.levelno == logging.WARNING]
    assert got[1] is None and len(got[0]) >= 1
    n_ref, recs = bai.bam_records(a)
    for t, p, e, _f, vb, ve in recs:
        if t == 3 and p < 20000 and e > 10:
            assert _covered(got[0], vb, ve)
    assert sum(hi - (lo >> 16) for lo, hi in got[0]) < os.path.getsize(a) / 4
