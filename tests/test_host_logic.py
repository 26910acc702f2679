"""Host-side logic that must reproduce the reference exactly: the integer forms of the float
comparisons, contig-name resolution, configuration errors, the SNP loaders and the join."""

import logging
import math
import os

import numpy as np
import pytest
from hypothesis import given, settings
from hypothesis import strategies as st

from util import GOLD

from xcltk_b200 import engine
from xcltk_b200.utils.sam import build_tid_maps, resolve_tid

logging.disable(logging.CRITICAL)


@settings(max_examples=200, deadline=None)
@given(st.floats(min_value=1e-6, max_value=0.999999), st.integers(min_value=1, max_value=400))
def test_include_table_is_the_reference_expression(f, n):
    """keep iff not (m / float(n) < min_include)  (rdr/fc/core.py:160-162)."""
    tab, _ = engine.include_threshold(f, 400)
    for m in range(0, n + 1):
        assert (m >= tab[n]) == (not (m / float(n) < f))


def test_include_length_mode_and_mapq():
    for v, exp in ((0, 0), (1, 1), (1.0, 1), (20, 20), (2.5, 3), (-3, -3)):
        tab, ln = engine.include_threshold(v, 100)
        assert tab is None and ln == exp
        for m in range(0, 30):
            assert (m >= ln) == (not (m < v))
    for x in (20, 20.0, 19.5, 0, 0.1, 255):
        for mapq in range(0, 256):
            assert (mapq < x) == (mapq < engine.min_mapq_int(x))
    assert engine.include_threshold(0.9, 91)[0][91] == 82          # 81/91 < 0.9 <= 82/91
    assert engine.include_threshold(0.9, 40)[0][40] == 36          # SURVEY D.1: 36/40 passes


def test_contig_resolution_follows_sam_fetch():
    idx = {"chr1": 0, "2": 1, "chrM": 2, "MT": 3}
    assert resolve_tid(idx, "1") == 0 and resolve_tid(idx, "2") == 1          # 'chr' toggled on / exact
    assert resolve_tid(idx, "chr2") == 1 and resolve_tid(idx, "M") == 2
    assert resolve_tid(idx, "3") == -1 and resolve_tid(idx, "MT") == 3
    gid_of, maps = build_tid_maps([[("chr1", 10), ("2", 10)], [("1", 10), ("chr2", 10), ("X", 5)]], ["2", "1", "Q"])
    assert gid_of == {"2": 0, "1": 1, "Q": 2}
    assert maps == [[1, 0], [1, 0, -1]]
    with pytest.raises(ValueError):
        build_tid_maps([[("chr1", 10)]], ["1", "chr1"])


def _conf(tmp_path, **kw):
    from xcltk_b200.rdr.fc.config import Config
    d = os.path.join(GOLD, "d1_basefc_mini")
    c = Config()
    c.sam_fn, c.barcode_fn = os.path.join(d, "a.bam"), os.path.join(d, "barcodes.tsv")
    c.region_fn, c.out_dir = os.path.join(d, "features.tsv"), str(tmp_path / "o")
    for k, v in kw.items():
        setattr(c, k, v)
    return c


@pytest.mark.parametrize("kw", [
    {"sam_list_fn": "x"}, {"sam_fn": None}, {"sam_fn": "/nonexistent.bam"}, {"sample_id_str": "a"},
    {"barcode_fn": "/nonexistent.tsv"}, {"out_dir": None}, {"region_fn": None}, {"region_fn": "/nonexistent"},
    {"cell_tag": "None"}, {"barcode_fn": None, "sample_id_str": "a,b"}, {"barcode_fn": None, "sample_id_str": "a"},
])
def test_basefc_configuration_errors_return_minus_one(tmp_path, kw):
    from xcltk_b200.rdr.fc.main import fc_run, prepare_config
    assert prepare_config(_conf(tmp_path, **kw)) == -1
    assert fc_run(_conf(tmp_path, **kw)) == -1                     # ValueError("errcode -2") -> -1


def test_basefc_prepare_config_derives_like_the_reference(tmp_path):
    from xcltk_b200.rdr.fc.main import prepare_config
    c = _conf(tmp_path, umi_tag="Auto")
    assert prepare_config(c) == 0
    assert c.samples == ["AAA", "BBB"] and c.umi_tag == "UB" and c.excl_flag == 772
    assert open(c.out_sample_fn).read() == "AAA\nBBB\n"
    assert [(r.chrom, r.start, r.end, r.get_id()) for r in c.reg_list][:2] == [("1", 175, 401, "g2"), ("1", 101, 201, "g1")]
    c = _conf(tmp_path, umi_tag="none")
    assert prepare_config(c) == 0 and c.umi_tag is None and c.excl_flag == 1796
    c = _conf(tmp_path, excl_flag=4)
    assert prepare_config(c) == 0 and c.excl_flag == 4              # CLI --exclFLAG is honoured


def test_basefc_cli_options(tmp_path, monkeypatch):
    """Option parsing of fc_main (long options case-insensitive, minINCLUDE int vs float)."""
    from xcltk_b200.rdr.fc import main as m
    seen = {}
    monkeypatch.setattr(m, "fc_run", lambda conf: seen.setdefault("conf", conf) and 0)
    monkeypatch.setattr(m, "init_logging", lambda **k: None)
    m.fc_main(["xcltk", "basefc", "-s", "a.bam", "-b", "b.tsv", "-R", "r.tsv", "-O", "o", "-p", "4", "--cellTAG", "RG",
               "--UMItag", "None", "--minMAPQ", "9.5", "--minINCLUDE", "20", "--countORPHAN", "--exclFLAG", "0"])
    c = seen["conf"]
    assert (c.sam_fn, c.nproc, c.cell_tag, c.umi_tag, c.min_mapq, c.min_include, c.no_orphan, c.excl_flag) == \
        ("a.bam", 4, "RG", "None", 9.5, 20, False, 0) and isinstance(c.min_include, int)
    seen.clear()
    m.fc_main(["xcltk", "basefc", "-s", "a.bam", "--minINCLUDE", "0.5", "--minLEN", "10", "--inclFLAG", "2"])
    assert seen["conf"].min_include == 0.5 and seen["conf"].min_len == 10 and seen["conf"].incl_flag == 2
    with pytest.raises(SystemExit):
        m.fc_main(["xcltk", "basefc"])


def test_snp_loaders_and_region_join():
    from xcltk_b200.baf.fc.utils import load_region_from_txt, load_snp_from_tsv, load_snp_from_vcf
    d = os.path.join(GOLD, "d2_baf_mini")
    tsv = load_snp_from_tsv(os.path.join(d, "snps.tsv"))
    assert [(s.chrom, s.pos, s.ref, s.alt, s.ref_idx, s.alt_idx) for s in tsv.snps] == \
        [("1", 120, "C", "T", 0, 1), ("1", 150, "G", "A", 1, 0), ("1", 550, "A", "C", 0, 1)]
    vcf = load_snp_from_vcf(os.path.join(d, "snps.vcf"))          # lower-case REF, '/' GT, multi-base ALT, 1|1, no GT
    assert [(s.chrom, s.pos, s.ref, s.alt, s.ref_idx) for s in vcf.snps] == \
        [("1", 120, "C", "T", 0), ("1", 150, "G", "A", 1), ("1", 550, "A", "C", 0)]
    regs = load_region_from_txt(os.path.join(d, "features.tsv"))
    got = [[s.pos for s in tsv.fetch(r.chrom, r.start, r.end)] for r in regs]
    assert got == [[120, 150], [550], [150]]
    assert tsv.fetch("chr1", 150, 151)[0].pos == 150 and tsv.fetch("2", 1, 1000) == [] and tsv.fetch("1", 151, 151) == []
    snp = tsv.snps[1]
    assert [snp.get_region_allele_index(b) for b in "GACTN"] == [1, 0, -1, -1, -1]


def test_baf_missing_cellsnp_dir_and_empty_region_list(tmp_path):
    from xcltk_b200.baf.fc.main import afc_wrapper
    d = os.path.join(GOLD, "d2_baf_mini")
    args = (os.path.join(d, "a.bam"), os.path.join(d, "barcodes.tsv"), os.path.join(d, "features.tsv"),
            os.path.join(d, "snps.tsv"), str(tmp_path / "o"))
    with pytest.raises(AssertionError):                           # assert_e(conf.cellsnp_dir), baf/fc/main.py:420
        afc_wrapper(*args, cellsnp_dir="/some/dir")
    far = str(tmp_path / "far.tsv")                               # no SNP in any region, output_all_reg=False:
    with open(far, "w") as fp:                                    # the reference divides by zero workers
        fp.write("9\t1\t100\tg\n")
    with pytest.raises(ZeroDivisionError):
        afc_wrapper(args[0], args[1], far, args[3], args[4])


def test_write_mtx_format(tmp_path):
    p = str(tmp_path / "m.mtx")
    emitted = np.array([True, True, False, True, True])           # input row 2 is not emitted
    engine.write_mtx(p, 5, np.array([0, 1, 1, 4]), np.array([0, 0, 1, 6]), np.array([1, 2, 1, 123456]), emitted, 7, 3)
    assert open(p).read() == ("%%MatrixMarket matrix coordinate integer general\n%%\n4\t7\t4\n"
                              "1\t1\t1\n2\t1\t2\n2\t2\t1\n4\t7\t123456\n")
    engine.write_mtx(p, 3, np.zeros(0, int), np.zeros(0, int), np.zeros(0, int), np.array([True, False, True]), 2)
    assert open(p).read() == "%%MatrixMarket matrix coordinate integer general\n%%\n2\t2\t0\n"
    rng = np.random.RandomState(1)                                # many slabs / threads == python formatting
    n, rows = 3000000, 5000
    row = np.sort(rng.randint(0, rows, size=n))
    col, val = rng.randint(0, 99999, size=n), rng.randint(1, 2 ** 31 - 1, size=n)
    engine.write_mtx(p, rows, row, col, val, np.ones(rows, dtype=bool), 99999, 5)
    body = open(p).read().split("\n", 3)[3]
    assert body == "".join("%d\t%d\t%d\n" % t for t in zip((row + 1).tolist(), (col + 1).tolist(), val.tolist()))


def test_write_mtx_rows_equals_csr_writer(tmp_path):
    """rows stored out of order and located by (row_beg, row_cnt) -- the layout basefc returns
    with XG_LAYOUT_ROWS -- give the text of the sorted CSR"""
    import numpy as np
    from xcltk_b200 import engine, lib
    rng = np.random.RandomState(4)
    n_rows, n_cols = 300, 50
    cnt = rng.randint(0, 12, size=n_rows).astype(np.int32)
    cnt[rng.rand(n_rows) < 0.3] = 0
    row = np.repeat(np.arange(n_rows, dtype=np.int32), cnt)
    col = np.concatenate([np.sort(rng.choice(n_cols, c, replace=False)) for c in cnt] + [np.zeros(0, int)]).astype(np.int32)
    val = rng.randint(1, 1000000, size=len(row)).astype(np.int32)
    emitted = cnt > 0
    emitted[::5] = True
    engine.write_mtx(str(tmp_path / "a.mtx"), n_rows, row, col, val, emitted, n_cols, 3)
    # scatter the rows in a random order, with gaps
    order = rng.permutation(n_rows)
    beg = np.zeros(n_rows, dtype=np.int64)
    pos = 0
    for r in order:
        beg[r] = pos
        pos += cnt[r]
    ptr = np.concatenate([[0], np.cumsum(cnt)])
    c2, v2 = np.zeros(pos, dtype=np.int32), np.zeros(pos, dtype=np.int32)
    for r in range(n_rows):
        c2[beg[r]:beg[r] + cnt[r]] = col[ptr[r]:ptr[r + 1]]
        v2[beg[r]:beg[r] + cnt[r]] = val[ptr[r]:ptr[r + 1]]
    seg = lib.RowSegments(beg, cnt, c2, v2, (n_rows, n_cols))
    out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
    lib.write_mtx_rows(str(tmp_path / "b.mtx"), seg, out_row, int(emitted.sum()), 2)
    assert open(str(tmp_path / "a.mtx"), "rb").read() == open(str(tmp_path / "b.mtx"), "rb").read()
    for a, b in zip(seg.to_sorted(), (row, col, val)):
        assert np.array_equal(a, b)


def test_snp_filter_is_the_references_scalar_expression():
    """vectorised plp_snp filter == `snp_cnt < min_count or min(ref, alt) < snp_cnt * min_maf`
    evaluated per SNP with Python ints / floats (baf/fc/core.py:238-246)"""
    import random
    import numpy as np
    from xcltk_b200.baf.fc.main import BASE_IDX, snp_filter

    class Obj(object):
        pass
    rng = random.Random(3)
    for trial in range(200):
        n = rng.randrange(0, 50)
        snps = []
        for _ in range(n):
            s = Obj()
            s.ref, s.alt = rng.choice("ACGTN"), rng.choice("ACGTN")
            snps.append(s)
        totals = np.array([[rng.choice([0, 0, 1, 2, 3, 7, 100, 2 ** 40]) for _ in range(5)] for _ in range(n)],
                          dtype=np.int64).reshape(n, 5)
        conf = Obj()
        conf.min_count = rng.choice([0, 1, 3, 20, 2.5, 1.0])
        conf.min_maf = rng.choice([0, 0.0, 0.1, 0.3, 0.5, 1, 0.05, 1 / 3.0])
        exp = []
        for i, s in enumerate(snps):
            t = [int(x) for x in totals[i]]
            cnt = sum(t)
            skip = cnt < conf.min_count or min(t[BASE_IDX[s.ref]], t[BASE_IDX[s.alt]]) < cnt * conf.min_maf
            exp.append(0 if skip else 1)
        assert list(snp_filter(conf, snps, totals)) == exp


def test_write_mtx_rows16_narrow_entries_and_side_list(tmp_path):
    """the packed layout (column | count << 16, counts >= 65535 in a side list) writes the text
    of the plain layout"""
    import numpy as np
    from xcltk_b200 import lib
    rng = np.random.RandomState(9)
    n_rows, n_cols = 120, 4000
    cnt = rng.randint(0, 30, size=n_rows).astype(np.int32)
    beg = np.concatenate([[0], np.cumsum(cnt)[:-1]]).astype(np.int64)
    nnz = int(cnt.sum())
    col = np.concatenate([np.sort(rng.choice(n_cols, c, replace=False)) for c in cnt] + [np.zeros(0, int)]).astype(np.int32)
    val = rng.randint(1, 300, size=nnz).astype(np.int32)
    big = rng.choice(nnz, 25, replace=False)
    val[big] = rng.randint(65535, 5000000, size=25)
    val[big[0]] = 65535                                   # exactly the escape value
    plain = lib.RowSegments(beg, cnt, col, val, (n_rows, n_cols))
    cv = (col.astype(np.uint32) | (np.minimum(val, 65535).astype(np.uint32) << np.uint32(16)))
    over_idx = np.nonzero(val >= 65535)[0].astype(np.int64)
    perm = rng.permutation(len(over_idx))                 # the side list is not ordered
    narrow = lib.RowSegments(beg, cnt, None, None, (n_rows, n_cols), cv16=cv, over=(over_idx[perm], val[over_idx][perm]))
    assert np.array_equal(narrow.col, col) and np.array_equal(narrow.val, val)
    emitted = cnt > 0
    out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
    lib.write_mtx_rows(str(tmp_path / "a.mtx"), plain, out_row, int(emitted.sum()), 2)
    lib.write_mtx_rows(str(tmp_path / "b.mtx"), narrow, out_row, int(emitted.sum()), 3)
    a, b = open(str(tmp_path / "a.mtx"), "rb").read(), open(str(tmp_path / "b.mtx"), "rb").read()
    assert a == b and b"\t65535\n" in a


def test_write_mtx_rows_tiny_delta_entries_and_side_list(tmp_path):
    """the 16-bit layout ((column - previous column - 1) << 4 | count; first of a row, gaps > 4095 and counts > 15 in
    a side list of (idx, val, col) in no particular order) decodes to, and writes the text of, the plain layout; the
    rows sit in the staging order of the device (not row order), with a gap of unused entries between two of them"""
    import numpy as np
    from xcltk_b200 import lib
    rng = np.random.RandomState(11)
    n_rows, n_cols = 300, 60000
    cnt = rng.randint(0, 40, size=n_rows).astype(np.int32)
    cnt[5] = 0
    cnt[17] = 1
    order = rng.permutation(n_rows)                       # completion order
    beg = np.zeros(n_rows, dtype=np.int64)
    at = 0
    for r in order:
        beg[r] = at
        at += int(cnt[r])
    nnz = at
    col = np.zeros(nnz, dtype=np.int32)
    val = rng.randint(1, 12, size=nnz).astype(np.int32)
    for r in range(n_rows):
        span = n_cols if r % 3 else 900                   # sparse rows: wide gaps; dense rows: small ones
        col[beg[r]:beg[r] + cnt[r]] = np.sort(rng.choice(span, cnt[r], replace=False))
    val[rng.choice(nnz, 40, replace=False)] = rng.randint(16, 3000000, size=40)
    val[3] = 15
    val[4] = 16                                           # the largest count that fits, the smallest that does not
    plain = lib.RowSegments(beg, cnt, col, val, (n_rows, n_cols))
    # encode as k_pack_rows_tiny does
    first = np.zeros(nnz, dtype=bool)
    first[beg[cnt > 0]] = True
    prev = np.concatenate([[0], col[:-1]])
    d = col.astype(np.int64) - prev - 1
    fits = ~first & (d >= 0) & (d <= 4094) & (val <= 15)
    w = np.where(fits, (d << 4) | val, 0).astype(np.uint16)
    idx = np.nonzero(~fits)[0].astype(np.int64)
    perm = rng.permutation(len(idx))
    tiny = lib.RowSegments(beg, cnt, None, None, (n_rows, n_cols), over=(idx[perm], val[idx][perm], col[idx][perm]), tiny=w)
    assert tiny.nnz == nnz and np.array_equal(tiny.col, col) and np.array_equal(tiny.val, val)
    assert (w[~first] != 0).sum() > nnz // 2              # most entries do travel as 16 bits
    for a, b in zip(tiny.to_sorted(), plain.to_sorted()):
        assert np.array_equal(a, b)
    emitted = cnt > 0
    emitted[5] = True                                     # an empty row that is emitted all the same
    out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
    lib.write_mtx_rows(str(tmp_path / "a.mtx"), plain, out_row, int(emitted.sum()), 2)
    for k, threads in enumerate((1, 5)):
        lib.write_mtx_rows(str(tmp_path / ("t%d.mtx" % k)), tiny, out_row, int(emitted.sum()), threads)
        assert open(str(tmp_path / "a.mtx"), "rb").read() == open(str(tmp_path / ("t%d.mtx" % k)), "rb").read()
    empty = lib.RowSegments(np.zeros(3, np.int64), np.zeros(3, np.int32), None, None, (3, 10),
                            over=(np.zeros(0, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int32)), tiny=np.zeros(0, np.uint16))
    assert empty.nnz == 0 and len(empty.col) == 0 and len(empty.val) == 0
    lib.write_mtx_rows(str(tmp_path / "e.mtx"), empty, np.array([1, 2, 3], np.int32), 3, 2)
    assert open(str(tmp_path / "e.mtx")).read().splitlines()[-1] == "3\t10\t0"


@settings(max_examples=40, deadline=None)
@given(st.integers(0, 2 ** 32 - 1), st.integers(1, 60), st.sampled_from([7, 300, 5000, 70000, 1 << 20]),
       st.sampled_from([3, 15, 16, 70000]))
def test_tiny_layout_round_trip_property(seed, n_rows, n_cols, max_val):
    """any matrix survives the 16-bit layout: encode as k_pack_rows_tiny does, decode with RowSegments, write with
    xg_write_mtx_rows_tiny -- equal to the plain layout entry for entry and byte for byte"""
    import tempfile
    from xcltk_b200 import lib
    rng = np.random.RandomState(seed)
    cnt = rng.randint(0, min(n_cols, 50) + 1, size=n_rows).astype(np.int32)
    order = rng.permutation(n_rows)
    beg = np.zeros(n_rows, dtype=np.int64)
    at = 0
    for r in order:
        beg[r] = at
        at += int(cnt[r])
    nnz = at
    col = np.zeros(nnz, dtype=np.int32)
    for r in range(n_rows):
        col[beg[r]:beg[r] + cnt[r]] = np.sort(rng.choice(n_cols, cnt[r], replace=False))
    val = rng.randint(1, max_val + 1, size=nnz).astype(np.int32)
    first = np.zeros(nnz, dtype=bool)
    first[beg[cnt > 0]] = True
    d = col.astype(np.int64) - np.concatenate([[0], col[:-1]]) - 1
    fits = ~first & (d >= 0) & (d <= 4094) & (val <= 15)
    w = np.where(fits, (d << 4) | val, 0).astype(np.uint16)
    idx = np.nonzero(~fits)[0].astype(np.int64)
    perm = rng.permutation(len(idx))
    tiny = lib.RowSegments(beg, cnt, None, None, (n_rows, n_cols), over=(idx[perm], val[idx][perm], col[idx][perm]), tiny=w)
    plain = lib.RowSegments(beg, cnt, col, val, (n_rows, n_cols))
    assert np.array_equal(tiny.col, col) and np.array_equal(tiny.val, val)
    emitted = cnt > 0
    out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
    with tempfile.TemporaryDirectory() as td:
        lib.write_mtx_rows(os.path.join(td, "a.mtx"), plain, out_row, int(emitted.sum()), 2)
        lib.write_mtx_rows(os.path.join(td, "b.mtx"), tiny, out_row, int(emitted.sum()), 3)
        assert open(os.path.join(td, "a.mtx"), "rb").read() == open(os.path.join(td, "b.mtx"), "rb").read()


def test_genomic_chunks_partition_the_library():
    """bench.py --scaling strong: the chunks' features are a disjoint cover of the feature list, and every chunk's
    read range reaches from HALO_BP before its first feature to the end of its last one (reads are sorted)."""
    import numpy as np
    from xcltk_b200 import lib, workload
    feats = workload.extend_features(workload.load_genes({"20", "21", "22"}), 3000, seed=5)
    gid_of = {"20": 0, "21": 1, "22": 2}
    gid, beg, end = workload.feature_arrays(feats + [("7", 10, 20, "other_contig"), ("21", 0, 50, "start0")], gid_of)
    sg, sb, se = workload.merged_spans(feats, gid_of)
    n_total, seed = 5000000, 11
    for world in (1, 2, 3, 8):
        seen = np.zeros(len(gid), dtype=np.int32)
        prev_i0 = -1
        for rank in range(world):
            idx, i0, n = workload.genomic_chunk(None, n_total, seed, sg, sb, se, gid, beg, end, (rank, world))
            seen[idx] += 1
            ok = idx[(gid[idx] >= 0) & (end[idx] > beg[idx])]
            if len(ok) == 0:
                continue
            assert i0 >= prev_i0 and 0 <= i0 and i0 + n <= n_total
            prev_i0 = i0
            first = ok[np.lexsort((beg[ok], gid[ok]))[0]]
            lo = lib.synth_read_index(n_total, sg, sb, se, int(gid[first]), max(0, int(beg[first]) - workload.HALO_BP), seed)
            assert i0 == lo
            for f in ok[:50]:        # the reads at a feature's end still belong to the chunk
                hi = lib.synth_read_index(n_total, sg, sb, se, int(gid[f]), int(end[f]), seed)
                assert i0 + n >= hi
        assert np.all(seen == 1)


def test_reference_import_paths_resolve_to_this_build():
    """Drop-in at the Python level: the reference's module paths and entry points (xcltk/rdr/fc/main.py:142,
    xcltk/baf/fc/main.py:32, xcltk/xcltk.py:40, setup.py:58-62) import from the `xcltk` name."""
    import importlib
    import inspect
    fc = importlib.import_module("xcltk.rdr.fc.main")
    afc = importlib.import_module("xcltk.baf.fc.main")
    cli = importlib.import_module("xcltk.xcltk")
    assert fc.__file__.endswith(os.path.join("xcltk_b200", "rdr", "fc", "main.py"))
    assert list(inspect.signature(fc.fc_wrapper).parameters)[:4] == ["sam_fn", "barcode_fn", "region_fn", "out_dir"]
    sig = inspect.signature(afc.afc_wrapper).parameters
    assert "cellsnp_dir" in sig and "ref_cell_fn" in sig and sig["output_all_reg"].default is False
    assert callable(cli.main)
    import xcltk
    assert xcltk.__version__ == "0.5.2"
