"""GPU parity on device-generated 10x-style batches: CUDA path (through the C-ABI) vs the CPU
oracle on the same records, bit-exact; plus size-independent properties at larger sizes."""

import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


class Conf(object):
    min_mapq, min_len, min_include = 20, 30, 0.9
    incl_flag, excl_flag, no_orphan = 0, 772, True

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return True

    def use_umi(self):
        return True


def gpu_params(conf, with_include=True):
    from xcltk_b200 import engine
    return engine.make_params(conf, 91, with_include)


@pytest.fixture(scope="module")
def fc_batch(gpu_ctx):
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 1500000, 2000, 33472, seed=21)
    w.host = w.dreads.download()
    return w


@pytest.mark.parametrize("kw", [
    {}, {"min_include": 0.5}, {"min_include": 30, "min_mapq": 0}, {"min_include": 0, "excl_flag": 0, "min_len": 1},
    {"min_include": 1.0, "incl_flag": 16}, {"min_include": 0.95, "min_mapq": 2.5, "no_orphan": False},
])
def test_basefc_matches_oracle(gpu_ctx, fc_batch, kw):
    from oracle import oracle
    conf, w = Conf(**kw), fc_batch
    row, col, val, shape = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, gpu_params(conf))
    o_row, o_col, o_val = oracle.basefc(w.host, w.gid, w.beg, w.end, w.cell_keys, 2000, oracle.params(conf), 4)
    assert shape == (len(w.gid), 2000) and len(val) > 1000
    assert np.array_equal(row, o_row) and np.array_equal(col, o_col) and np.array_equal(val, o_val)
    assert np.all(np.diff(row.astype(np.int64) * 2000 + col) > 0)          # sorted by (row, col), unique


@pytest.mark.parametrize("env", [
    {"XG_SEG_MODE": "0"},                               # a (cell, UMI) set per feature, no pair words
    {"XG_SEG_MAX": "0"},                                # pair-word mode, but every feature keeps a set
    {"XG_SEG_MAX": "1000"},                             # light features in segments, the rest in sets
    {"XG_SEG_MAX": "100000000", "XG_EPOCH_TILES": "97"},     # every feature a segment; heavy ones split by hash
    {"XG_HIST_COLS": "700"},                            # three column ranges per row
])
def test_basefc_counting_modes_match_oracle(gpu_ctx, fc_batch, monkeypatch, env):
    """Every way the counting kernel can route a (feature, cell, UMI) triple gives the oracle's matrix."""
    from oracle import oracle
    conf, w = Conf(), fc_batch
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    row, col, val, _ = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, gpu_params(conf))
    t = gpu_ctx.timing()
    o_row, o_col, o_val = oracle.basefc(w.host, w.gid, w.beg, w.end, w.cell_keys, 2000, oracle.params(conf), 4)
    assert np.array_equal(row, o_row) and np.array_equal(col, o_col) and np.array_equal(val, o_val)
    if env.get("XG_SEG_MODE") == "0" or env.get("XG_SEG_MAX") == "0":
        assert t[14] == 0 and t[15] > 0            # no segment features
    if env.get("XG_SEG_MAX") == "1000":
        assert t[14] > 0 and t[15] > 0             # both kinds


def test_basefc_heavy_segments_are_partitioned(gpu_ctx):
    """Few wide features: every segment holds far more pair words than the dedup table of a finalize CTA."""
    from oracle import oracle
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 3000000, 3000, 0, seed=13, chroms={"21", "22"}, bins_kb=2000)
    conf = Conf(min_include=0.5)
    row, col, val, _ = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 3000, gpu_params(conf))
    assert gpu_ctx.timing()[14] > 0 and gpu_ctx.timing()[15] == 0
    host = w.dreads.download()
    o = oracle.basefc(host, w.gid, w.beg, w.end, w.cell_keys, 3000, oracle.params(conf), 4)
    assert np.array_equal(row, o[0]) and np.array_equal(col, o[1]) and np.array_equal(val, o[2])


def test_basefc_umi_keys_that_do_not_fit_a_pair_word(gpu_ctx):
    """UMI keys with bits below bit 24 (strings longer than 13 symbols): the kernel notices, the call is
    redone with a set per feature, and the batch remembers."""
    from oracle import oracle
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 400000, 500, 33472, seed=17, chroms={"19", "20", "21", "22"})
    host = w.dreads.download()
    umi = host.keys[:, 1]
    real = (umi != np.uint64(0xFFFFFFFFFFFFFFFF)) & (umi != np.uint64(0))
    # a 14th and 15th symbol: bits 21..26 -- distinct UMIs stay distinct, equal ones stay equal
    umi[real] |= ((umi[real] >> np.uint64(40)) & np.uint64(0x3F)) << np.uint64(21) | np.uint64(1 << 21)
    d = gpu_ctx.upload(host)
    conf = Conf()
    for _ in range(2):                # second call: straight to the sets
        row, col, val, _ = gpu_ctx.basefc(d, w.gid, w.beg, w.end, w.cell_keys, 500, gpu_params(conf))
        assert gpu_ctx.timing()[14] == 0 and gpu_ctx.timing()[15] > 0
        o = oracle.basefc(host, w.gid, w.beg, w.end, w.cell_keys, 500, oracle.params(conf), 4)
        assert len(val) > 1000
        assert np.array_equal(row, o[0]) and np.array_equal(col, o[1]) and np.array_equal(val, o[2])
    d.close()
    host.close()


def test_basefc_epoch_size_invariance(gpu_ctx, fc_batch, monkeypatch):
    w, conf = fc_batch, Conf()
    ref = None
    for tiles in ("100000", "64", "7", "1"):
        monkeypatch.setenv("XG_EPOCH_TILES", tiles)
        out = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, gpu_params(conf))[:3]
        out = [np.array(x) for x in out]
        if ref is None:
            ref = out
        assert all(np.array_equal(a, b) for a, b in zip(ref, out)), tiles


def test_basefc_feature_rows_are_independent(gpu_ctx, fc_batch):
    """Duplicated / permuted features give duplicated / permuted rows (R9: features are counted
    independently, output rows follow input order)."""
    w, conf = fc_batch, Conf()
    rng = np.random.RandomState(3)
    perm = rng.permutation(len(w.gid))[:5000]
    idx = np.concatenate([perm, perm[:100]])                  # first 100 appear twice
    row, col, val, _ = gpu_ctx.basefc(w.dreads, w.gid[idx], w.beg[idx], w.end[idx], w.cell_keys, 2000,
                                      gpu_params(conf))
    r0, c0, v0, _ = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, gpu_params(conf))
    full = {}
    for r, c, v in zip(r0.tolist(), c0.tolist(), v0.tolist()):
        full.setdefault(r, []).append((c, v))
    got = {}
    for r, c, v in zip(row.tolist(), col.tolist(), val.tolist()):
        got.setdefault(r, []).append((c, v))
    for k, orig in enumerate(idx.tolist()):
        assert got.get(k, []) == full.get(orig, [])


def test_basefc_many_cells_multi_pass_histogram(gpu_ctx):
    """More cells than the shared-memory histogram holds (> 40 960): column-range passes."""
    from oracle import oracle
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 300000, 100000, 2000, seed=4, chroms={"20", "21", "22"})
    conf = Conf()
    row, col, val, _ = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 100000, gpu_params(conf))
    host = w.dreads.download()
    o = oracle.basefc(host, w.gid, w.beg, w.end, w.cell_keys, 100000, oracle.params(conf), 4)
    assert col.max() > 40960
    assert np.array_equal(row, o[0]) and np.array_equal(col, o[1]) and np.array_equal(val, o[2])


def test_basefc_bins_large_windows(gpu_ctx):
    """1 Mb bins (config 5 shape): few features, very large per-feature sets."""
    from oracle import oracle
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 2000000, 500, 0, seed=9, chroms={"21", "22"}, bins_kb=1000)
    conf = Conf(min_include=0.5)
    row, col, val, _ = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 500, gpu_params(conf))
    host = w.dreads.download()
    o = oracle.basefc(host, w.gid, w.beg, w.end, w.cell_keys, 500, oracle.params(conf), 4)
    assert np.array_equal(row, o[0]) and np.array_equal(col, o[1]) and np.array_equal(val, o[2])


@pytest.fixture(scope="module")
def baf_batch(gpu_ctx):
    from xcltk_b200 import workload
    b = workload.make_baf_workload(gpu_ctx, 1000000, 1000, 40000, seed=31, chroms={"19", "20", "21", "22"})
    b.host = b.dreads.download()
    return b


@pytest.mark.parametrize("min_count,min_maf,no_dup", [(1, 0, True), (1, 0, False), (3, 0.1, True), (2, 0.34, False)])
def test_baf_matches_oracle(gpu_ctx, baf_batch, min_count, min_maf, no_dup):
    from oracle import oracle
    b = baf_batch
    conf = Conf(min_include=0)
    totals, st = gpu_ctx.baf_pileup(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 1000, gpu_params(conf, False))
    tot = totals.sum(axis=1)
    idx = np.arange(len(tot))
    minor = np.minimum(totals[idx, b.snp_ref], totals[idx, b.snp_alt])
    keep = ((tot >= min_count) & ~(minor < tot * min_maf)).astype(np.uint8)
    ad, dp, oth = gpu_ctx.baf_count(st, b.reg_ptr, b.reg_snp, b.hap_of, keep, no_dup)
    st.close()
    letters = "ACGT"
    o = oracle.baf(b.host, b.snp_gid, b.snp_pos, "".join(letters[x] for x in b.snp_ref),
                   "".join(letters[x] for x in b.snp_alt), b.snp_ref_hap, 1 - b.snp_ref_hap, b.reg_ptr,
                   b.reg_snp, b.cell_keys, 1000, oracle.params(conf), min_count, min_maf, no_dup, 4)
    assert len(dp[2]) > 100
    for got, exp in zip((ad, dp, oth), o):
        assert all(np.array_equal(g, e) for g, e in zip(got[:3], exp))
    # the same through the one-call entry point, SNP filter evaluated on the device (xg_baf_fc)
    f_ad, f_dp, f_oth, f_tot, f_keep = gpu_ctx.baf_fc(
        b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 1000, gpu_params(conf, False), b.snp_ref, b.snp_alt, min_count,
        min_maf, b.reg_ptr, b.reg_snp, b.hap_of, no_dup, want_totals=True, want_keep=True)
    assert np.array_equal(f_tot, totals) and np.array_equal(f_keep, keep)
    for got, exp in zip((f_ad, f_dp, f_oth), o):
        assert all(np.array_equal(g, e) for g, e in zip(got[:3], exp))


@pytest.mark.parametrize("min_count,min_maf", [(0, 0.0), (2.5, 0.0), (1, 1.0 / 3.0), (4, 0.5), (1, 0.1 + 0.2), (10 ** 9, 0.0)])
def test_baf_device_snp_filter_is_pythons_arithmetic(gpu_ctx, baf_batch, min_count, min_maf):
    """plp_snp's filter (baf/fc/core.py:238-246) on the device == Python ints against a float, SNP by SNP: thresholds
    that are not representable (1/3, 0.1 + 0.2), a float min_count, ties (minor == cnt * maf), nothing / everything kept."""
    b = baf_batch
    p = gpu_params(Conf(min_include=0), False)
    out = gpu_ctx.baf_fc(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 1000, p, b.snp_ref, b.snp_alt, min_count, min_maf,
                         b.reg_ptr, b.reg_snp, b.hap_of, True, want_totals=True, want_keep=True)
    totals, keep = out[3], out[4]
    exp = np.zeros(len(keep), dtype=np.uint8)
    for i in range(len(keep)):
        t = [int(x) for x in totals[i]]
        cnt = sum(t)
        if cnt < min_count:
            continue
        if min(t[b.snp_ref[i]], t[b.snp_alt[i]]) < cnt * min_maf:
            continue
        exp[i] = 1
    assert np.array_equal(keep, exp)
    assert (min_count != 0) or keep.all()
    st_tot, st = gpu_ctx.baf_pileup(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 1000, p)
    ref = gpu_ctx.baf_count(st, b.reg_ptr, b.reg_snp, b.hap_of, exp, True)
    st.close()
    for x, y in zip(out[:3], ref):
        assert all(np.array_equal(u, v) for u, v in zip(x[:3], y[:3]))


def test_basefc_streamed_from_host_equals_resident(gpu_ctx, fc_batch, monkeypatch):
    """xg_basefc_host (records copied epoch by epoch under the kernels) == xg_basefc."""
    w, p = fc_batch, gpu_params(Conf())
    ref = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, p)[:3]]
    for tiles in ("8192", "100", "3"):
        monkeypatch.setenv("XG_EPOCH_TILES_HOST", tiles)
        out = [np.array(x) for x in gpu_ctx.basefc_host(w.host, w.gid, w.beg, w.end, w.cell_keys, 2000, p)[:3]]
        assert all(np.array_equal(a, b) for a, b in zip(ref, out)), tiles


def test_baf_zero_copy_batch_equals_uploaded(gpu_ctx, baf_batch):
    """xg_map_reads (records read from pinned host memory) gives the same pileup as the
    HBM-resident batch; basefc refuses a mapped batch."""
    from xcltk_b200 import lib
    b = baf_batch
    p = gpu_params(Conf(min_include=0), False)
    t0, st0 = gpu_ctx.baf_pileup(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 1000, p)
    mapped = gpu_ctx.map_reads(b.host)
    t1, st1 = gpu_ctx.baf_pileup(mapped, b.snp_gid, b.snp_pos, b.cell_keys, 1000, p)
    assert np.array_equal(t0, t1) and t0.sum() > 1000
    keep = (t0.sum(axis=1) >= 1).astype(np.uint8)
    a = gpu_ctx.baf_count(st0, b.reg_ptr, b.reg_snp, b.hap_of, keep, True)
    c = gpu_ctx.baf_count(st1, b.reg_ptr, b.reg_snp, b.hap_of, keep, True)
    for x, y in zip(a, c):
        assert all(np.array_equal(u, v) for u, v in zip(x[:3], y[:3]))
    with pytest.raises(lib.XgError):
        gpu_ctx.basefc(mapped, b.gid, b.beg, b.end, b.cell_keys, 1000, gpu_params(Conf()))
    st0.close()
    st1.close()
    mapped.close()


def test_basefc_full_size_properties(gpu_ctx):
    """Bench-scale batch (config 3 shape, 50M reads): idempotence and per-contig additivity --
    counting each contig's features separately and concatenating equals the whole run."""
    from xcltk_b200 import workload
    n = int(float(os.environ.get("XG_TEST_BIG_READS", "5e7")))
    w = workload.make_basefc_workload(gpu_ctx, n, 10000, 60000, seed=13)
    p = gpu_params(Conf())
    a = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 10000, p)[:3]]
    b = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 10000, p)[:3]]
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert int(a[2].sum()) <= int(n * 1.5) and len(a[2]) > n // 10
    rows, cols, vals = [], [], []
    for g in np.unique(w.gid):
        sel = np.nonzero(w.gid == g)[0]
        r, c, v, _ = gpu_ctx.basefc(w.dreads, w.gid[sel], w.beg[sel], w.end[sel], w.cell_keys, 10000, p)
        rows.append(sel[r])
        cols.append(np.array(c))
        vals.append(np.array(v))
    rows, cols, vals = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    order = np.lexsort((cols, rows))
    assert np.array_equal(rows[order], a[0]) and np.array_equal(cols[order], a[1]) and np.array_equal(vals[order], a[2])


def test_basefc_row_segments_equal_sorted_result(gpu_ctx, fc_batch, tmp_path):
    """the rows layouts: rows in completion order, copied out under the kernels --
    the same matrix as the sorted result, from HBM and streamed from the host, on the first call
    (no size hint: one copy at the end) and on repeated ones (per-epoch copies); and the
    Matrix-Market text written from it is the one written from the sorted CSR."""
    from xcltk_b200 import engine, lib
    w, p = fc_batch, gpu_params(Conf())
    ref = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, p)[:3]]
    for k in range(3):
        seg = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, p, segments=True)
        assert isinstance(seg, lib.RowSegments) and seg.nnz == len(ref[2])
        for a, b in zip(seg.to_sorted(), ref):
            assert np.array_equal(a, b)
    seg_h = gpu_ctx.basefc_host(w.host, w.gid, w.beg, w.end, w.cell_keys, 2000, p, segments=True)
    for a, b in zip(seg_h.to_sorted(), ref):
        assert np.array_equal(a, b)
    # narrow entries (column | count << 16), resident and streamed, and the text written from them
    for call, src in ((gpu_ctx.basefc, w.dreads), (gpu_ctx.basefc_host, w.host)):
        for k in range(2):
            seg_n = call(src, w.gid, w.beg, w.end, w.cell_keys, 2000, p, segments="narrow")
            assert seg_n.cv16 is not None and seg_n.nnz == len(ref[2])
            for a, b in zip(seg_n.to_sorted(), ref):
                assert np.array_equal(a, b)
    # 16-bit entries (column delta | small count; first of a row, wide gaps and large counts in the side list)
    for call, src in ((gpu_ctx.basefc, w.dreads), (gpu_ctx.basefc_host, w.host)):
        for k in range(2):
            seg_t = call(src, w.gid, w.beg, w.end, w.cell_keys, 2000, p, segments="tiny")
            assert seg_t.tiny is not None and seg_t.tiny.dtype == np.uint16 and seg_t.nnz == len(ref[2])
            n_rows_nz = int((np.asarray(seg_t.row_cnt) > 0).sum())
            assert n_rows_nz <= len(seg_t.over[0]) < seg_t.nnz // 4         # every row start, few others
            for a, b in zip(seg_t.to_sorted(), ref):
                assert np.array_equal(a, b)
    # a smaller and a larger problem after the hint was set
    for sel in (slice(0, len(w.gid) // 3), slice(None)):
        seg = gpu_ctx.basefc(w.dreads, w.gid[sel], w.beg[sel], w.end[sel], w.cell_keys, 2000, p, segments=True)
        r = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid[sel], w.beg[sel], w.end[sel], w.cell_keys, 2000, p)[:3]]
        for a, b in zip(seg.to_sorted(), r):
            assert np.array_equal(a, b)
    n = len(w.gid)
    emitted = np.zeros(n, dtype=bool)
    emitted[ref[0]] = True
    emitted[::7] = True
    engine.write_mtx(str(tmp_path / "a.mtx"), n, ref[0], ref[1], ref[2], emitted, 2000)
    out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
    lib.write_mtx_rows(str(tmp_path / "b.mtx"), seg, out_row, int(emitted.sum()))
    assert open(str(tmp_path / "a.mtx"), "rb").read() == open(str(tmp_path / "b.mtx"), "rb").read()
    lib.write_mtx_rows(str(tmp_path / "c.mtx"), seg_n, out_row, int(emitted.sum()))
    assert open(str(tmp_path / "a.mtx"), "rb").read() == open(str(tmp_path / "c.mtx"), "rb").read()
    lib.write_mtx_rows(str(tmp_path / "d.mtx"), seg_t, out_row, int(emitted.sum()), n_threads=3)
    assert open(str(tmp_path / "a.mtx"), "rb").read() == open(str(tmp_path / "d.mtx"), "rb").read()
    # ... and the text formatted on the device from the staging area of the last call (every result layout)
    for k, mode in enumerate((True, "narrow", "tiny")):
        gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, p, segments=mode)
        gpu_ctx.basefc_write_mtx(str(tmp_path / ("g%d.mtx" % k)), out_row, int(emitted.sum()), n_threads=2 + k)
        assert open(str(tmp_path / "a.mtx"), "rb").read() == open(str(tmp_path / ("g%d.mtx" % k)), "rb").read()
    gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, p)          # a sorted result leaves no staged rows
    with pytest.raises(lib.XgError):
        gpu_ctx.basefc_write_mtx(str(tmp_path / "x.mtx"), out_row, int(emitted.sum()))
    seg = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 2000, p, segments=True)
    with pytest.raises(lib.XgError):                      # a non-empty row without an output row
        gpu_ctx.basefc_write_mtx(str(tmp_path / "x.mtx"), np.zeros(n, np.int32), 0)


def test_basefc_row_segments_degenerate_inputs(gpu_ctx, fc_batch):
    """no features; only features that fetch nothing (unknown contig, empty window): empty rows"""
    w, p = fc_batch, gpu_params(Conf())
    z = np.zeros(0, dtype=np.int32)
    seg = gpu_ctx.basefc(w.dreads, z, z, z, w.cell_keys, 2000, p, segments=True)
    assert seg.nnz == 0 and len(seg.row_cnt) == 0
    gid = np.array([-1, int(w.gid[0]), -1], dtype=np.int32)
    beg = np.array([0, 5, 10], dtype=np.int32)
    end = np.array([100, 5, 20], dtype=np.int32)
    seg = gpu_ctx.basefc(w.dreads, gid, beg, end, w.cell_keys, 2000, p, segments=True)
    ref = gpu_ctx.basefc(w.dreads, gid, beg, end, w.cell_keys, 2000, p)
    assert seg.nnz == len(ref[2]) == 0 and list(seg.row_cnt) == [0, 0, 0]
    # one real feature between two empty ones
    gid = np.array([-1, int(w.gid[5]), -1], dtype=np.int32)
    beg = np.array([0, int(w.beg[5]), 10], dtype=np.int32)
    end = np.array([100, int(w.end[5]), 20], dtype=np.int32)
    seg = gpu_ctx.basefc(w.dreads, gid, beg, end, w.cell_keys, 2000, p, segments=True)
    ref = [np.array(x) for x in gpu_ctx.basefc(w.dreads, gid, beg, end, w.cell_keys, 2000, p)[:3]]
    for a, b in zip(seg.to_sorted(), ref):
        assert np.array_equal(a, b)


def test_baf_full_size_properties(gpu_ctx):
    """Bench-scale baf batch (config 2 shape: 50M reads, 5 000 cells, 200 000 SNPs): the run is
    reproducible; AD entries sit on DP entries and never exceed them; counting the regions in two halves and stacking the rows equals the whole
    run; dropping every SNP empties the matrices."""
    from xcltk_b200 import workload
    n = int(float(os.environ.get("XG_TEST_BIG_READS", "5e7")))
    b = workload.make_baf_workload(gpu_ctx, n, 5000, 200000, seed=17)
    p = gpu_params(Conf(min_include=0), False)

    def run(reg_ptr, reg_snp, keep=None):
        totals, st = gpu_ctx.baf_pileup(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 5000, p)
        k = ((totals[:, :5].sum(axis=1) >= 1).astype(np.uint8)) if keep is None else keep
        out = gpu_ctx.baf_count(st, reg_ptr, reg_snp, b.hap_of, k, True)
        st.close()
        return totals, [[np.array(x) for x in m[:3]] for m in out]

    totals, (ad, dp, oth) = run(b.reg_ptr, b.reg_snp)
    totals2, (ad2, dp2, oth2) = run(b.reg_ptr, b.reg_snp)
    assert np.array_equal(totals, totals2)
    for x, y in zip((ad, dp, oth), (ad2, dp2, oth2)):
        assert all(np.array_equal(u, v) for u, v in zip(x, y))
    assert len(dp[2]) > 1000 and int(totals.sum()) > 0       # (regions overlap: a SNP counts in each of them)
    n_cols = 5000
    key_dp = dp[0].astype(np.int64) * n_cols + dp[1]
    key_ad = ad[0].astype(np.int64) * n_cols + ad[1]
    pos = np.searchsorted(key_dp, key_ad)
    assert np.all(pos < len(key_dp)) and np.array_equal(key_dp[pos], key_ad)      # AD ⊂ DP
    assert np.all(ad[2] <= dp[2][pos]) and np.all(ad[2] > 0) and np.all(dp[2] > 0)
    # two halves of the regions, rows stacked
    n_reg = len(b.reg_ptr) - 1
    h = n_reg // 2
    parts = []
    for lo, hi in ((0, h), (h, n_reg)):
        rp = (b.reg_ptr[lo:hi + 1] - b.reg_ptr[lo]).astype(np.int64)
        rs = b.reg_snp[b.reg_ptr[lo]:b.reg_ptr[hi]]
        _, mats = run(rp, rs)
        parts.append([(m[0] + lo, m[1], m[2]) for m in mats])
    for k, whole in enumerate((ad, dp, oth)):
        for j in range(3):
            assert np.array_equal(np.concatenate([parts[0][k][j], parts[1][k][j]]), whole[j])
    _, (ad0, dp0, oth0) = run(b.reg_ptr, b.reg_snp, keep=np.zeros(len(b.snp_gid), dtype=np.uint8))
    assert len(ad0[2]) == len(dp0[2]) == len(oth0[2]) == 0


def test_basefc_narrow_entries_with_large_counts(gpu_ctx):
    """sample mode, one column: every count is far beyond 16 bits and goes through the side list;
    and more than 65536 columns switch the packing off"""
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 3000000, 50, 33472, seed=5, chroms={"20", "21", "22"})
    conf = Conf()
    conf.use_barcodes = lambda: False                      # every read -> column of its BAM (one BAM: column 0)
    p = gpu_params(conf)
    # whole-contig windows next to the genes: hundreds of thousands of molecules per entry
    g = np.unique(w.gid).astype(np.int32)
    gid = np.concatenate([g, w.gid[:300]]).astype(np.int32)
    beg = np.concatenate([np.zeros(len(g), np.int32), w.beg[:300]]).astype(np.int32)
    end = np.concatenate([np.full(len(g), 250000000, np.int32), w.end[:300]]).astype(np.int32)
    ref = [np.array(x) for x in gpu_ctx.basefc(w.dreads, gid, beg, end, None, 1, p)[:3]]
    assert ref[2].max() > 70000 and ref[2].min() < 65535
    seg = gpu_ctx.basefc(w.dreads, gid, beg, end, None, 1, p, segments="narrow")
    assert seg.cv16 is not None and len(seg.over[0]) == int((ref[2] >= 65535).sum()) > 0
    for a, b in zip(seg.to_sorted(), ref):
        assert np.array_equal(a, b)
    p2 = gpu_params(Conf())
    seg = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, np.arange(1, 70001, dtype=np.uint64) << np.uint64(40), 70000, p2,
                         segments="narrow")
    assert seg.cv16 is None                                # too many columns for 16 bits
    # the 16-bit layout: counts in the tens of thousands all go through the side list; 70 000 columns are fine
    seg = gpu_ctx.basefc(w.dreads, gid, beg, end, None, 1, p, segments="tiny")
    assert seg.tiny is not None and len(seg.over[0]) >= int((ref[2] > 15).sum())
    for a, b in zip(seg.to_sorted(), ref):
        assert np.array_equal(a, b)
    keys70k = np.arange(1, 70001, dtype=np.uint64) << np.uint64(40)
    r70 = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, keys70k, 70000, p2)[:3]]
    seg = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, keys70k, 70000, p2, segments="tiny")
    assert seg.tiny is not None
    for a, b in zip(seg.to_sorted(), r70):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("world", [2, 5])
def test_genomic_chunks_of_one_library_give_the_unsharded_rows(gpu_ctx, world):
    """bench.py --scaling strong on one GPU: every chunk (its features + the reads that can overlap them, generated
    as a slice of the same library) yields exactly its rows of the unsharded basefc and baf matrices."""
    from xcltk_b200 import workload
    chroms = {"19", "20", "21", "22"}
    conf = Conf()
    full = workload.make_basefc_workload(gpu_ctx, 1200000, 400, 9000, seed=31, chroms=chroms)
    f_row, f_col, f_val, _ = gpu_ctx.basefc(full.dreads, full.gid, full.beg, full.end, full.cell_keys, 400, gpu_params(conf))
    key_full = {}
    for r, c, v in zip(f_row.tolist(), f_col.tolist(), f_val.tolist()):
        key_full.setdefault(r, []).append((c, v))
    seen_rows, held = set(), 0
    for rank in range(world):
        w = workload.make_basefc_workload(gpu_ctx, 1200000, 400, 9000, seed=31, chroms=chroms, part=(rank, world))
        assert np.array_equal(w.cell_keys, full.cell_keys)
        held += w.n_reads
        row, col, val, _ = gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 400, gpu_params(conf))
        got = {}
        for r, c, v in zip(row.tolist(), col.tolist(), val.tolist()):
            got.setdefault(int(w.feat_index[r]), []).append((c, v))
        for k, g in enumerate(w.feat_index.tolist()):
            assert g not in seen_rows
            seen_rows.add(g)
            assert got.get(g, []) == key_full.get(g, []), (rank, k, g)
        w.dreads.close()
    assert seen_rows == set(range(len(full.gid)))
    assert held < 1200000 * 1.2                         # halos are small next to the chunks
    full.dreads.close()

    # baf: regions follow their chunk, the SNP table is shared
    fb = workload.make_baf_workload(gpu_ctx, 600000, 300, 4000, seed=33, chroms=chroms)
    totals, st = gpu_ctx.baf_pileup(fb.dreads, fb.snp_gid, fb.snp_pos, fb.cell_keys, 300, fb.params)
    keep = (totals.sum(axis=1) >= 1).astype(np.uint8)
    full_m = gpu_ctx.baf_count(st, fb.reg_ptr, fb.reg_snp, fb.hap_of, keep, True)
    st.close()
    full_rows = [{} for _ in range(3)]
    for k in range(3):
        for r, c, v in zip(full_m[k][0].tolist(), full_m[k][1].tolist(), full_m[k][2].tolist()):
            full_rows[k].setdefault(r, []).append((c, v))
    for rank in range(world):
        w = workload.make_baf_workload(gpu_ctx, 600000, 300, 4000, seed=33, chroms=chroms, part=(rank, world))
        totals, st = gpu_ctx.baf_pileup(w.dreads, w.snp_gid, w.snp_pos, w.cell_keys, 300, w.params)
        keep = (totals.sum(axis=1) >= 1).astype(np.uint8)
        m = gpu_ctx.baf_count(st, w.reg_ptr, w.reg_snp, w.hap_of, keep, True)
        st.close()
        for k in range(3):
            got = {}
            for r, c, v in zip(m[k][0].tolist(), m[k][1].tolist(), m[k][2].tolist()):
                got.setdefault(int(w.feat_index[r]), []).append((c, v))
            for g in w.feat_index.tolist():
                assert got.get(g, []) == full_rows[k].get(g, []), (rank, k, g)
        w.dreads.close()
    fb.dreads.close()
