"""The packed rows layouts of basefc and the device Matrix-Market writer at their switches.  Every rows layout
(segments=True / "narrow" / "tiny", resident and through basefc_host) is compared with the CSR result of the same
call, the CSR result with oracle.basefc where the shape allows, and the device text byte for byte with the text
engine.write_mtx writes from the CSR result.

  narrow  column | count << 16: packed up to 65 536 columns; a count >= 65 535 goes to the side list
  tiny    (column - previous column - 1) << 4 | count: a gap of up to 4 095 columns (d <= 4094) and counts 1..15
          pack; the first entry of a row, wider gaps and larger counts go to the side list; more than 2^23
          side-list entries give plain 32-bit entries instead
  text    mtx_digits at every decimal width of rows, columns and counts; 32 MB pinned chunks through 1, 2 or 8
          writer threads"""

import hashlib

import numpy as np
import pytest

from recsets import build, cell_keys, umi_keys
from xcltk_b200 import engine, lib

pytestmark = pytest.mark.gpu

LAYOUTS = (True, "narrow", "tiny")
TINY_OVER_CAP = 1 << 23


class Conf(object):
    min_mapq, min_len, min_include = 0, 1, 1
    incl_flag, excl_flag, no_orphan = 0, 0, False
    barcodes = True

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return self.barcodes

    def use_umi(self):
        return True


def tiny_escapes(row, col, val):
    """Entries the 16-bit layout cannot pack: first of its row, d = column - previous - 1 > 4094, count not in 1..15."""
    row, col, val = (np.asarray(x, np.int64) for x in (row, col, val))
    first = np.ones(len(row), bool)
    first[1:] = row[1:] != row[:-1]
    d = np.zeros(len(row), np.int64)
    d[1:] = col[1:] - col[:-1] - 1
    return int((first | (d > 4094) | (val < 1) | (val > 15)).sum())


def check_layouts(ctx, src, call, gid, beg, end, keys, n_cols, params, ref):
    """Every rows layout of one call == the CSR result `ref`; returns {layout: RowSegments}."""
    out = {}
    for mode in LAYOUTS:
        seg = call(src, gid, beg, end, keys, n_cols, params, segments=mode)
        assert isinstance(seg, lib.RowSegments) and seg.nnz == len(ref[2])
        for a, b in zip(seg.to_sorted(), ref):
            assert np.array_equal(a, b), mode
        out[mode] = seg
    return out


def sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as fp:
        for blk in iter(lambda: fp.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()


def check_text(ctx, tmp_path, reads_src, gid, beg, end, keys, n_cols, params, ref, emitted, threads):
    """The device text of every rows layout (n_threads each of `threads`) == engine.write_mtx of the CSR result."""
    n = len(gid)
    a = str(tmp_path / "csr.mtx")
    engine.write_mtx(a, n, ref[0], ref[1], ref[2], emitted, n_cols)
    want, size = sha(a), (tmp_path / "csr.mtx").stat().st_size
    out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
    for mode in LAYOUTS:
        ctx.basefc(reads_src, gid, beg, end, keys, n_cols, params, segments=mode)
        for t in threads:
            b = str(tmp_path / "dev.mtx")
            ctx.basefc_write_mtx(b, out_row, int(emitted.sum()), n_threads=t)
            assert sha(b) == want, (mode, t)
    return size


# ------------------------------------------------------------------------------------------ exact boundaries
def boundary_batch(n_cols):
    """Feature k covers [10000 k, 10000 k + 500); its reads sit inside it.  (feature, column, count) entries:
    gaps of exactly 4 095 and 4 096 columns and a wide one, counts 15 / 16 and 65 534 / 65 535, column n_cols - 1."""
    plan = [(0, 0, 1), (0, 4095, 2), (0, 8191, 3), (0, 8191 + 10000, 1),          # d = 4094, 4095, 9999
            (1, 5, 1), (1, 6, 15), (1, 7, 16), (1, 4102, 2),                       # d = 0, 0, 4094
            (2, 0, 1), (2, n_cols - 1, 1),
            (4, 7, 65534), (4, 8, 65535), (4, 9, 1)]                               # (feature 3: no reads)
    cell = np.concatenate([np.full(v, c, np.int64) for _, c, v in plan])
    feat = np.concatenate([np.full(v, f, np.int64) for f, _, v in plan])
    pos = feat * 10000 + 100 + (np.arange(len(cell)) % 300)
    order = np.argsort(pos, kind="stable")
    pos, cell = pos[order], cell[order]
    n = len(pos)
    ck = cell_keys(n_cols)
    reads = build(pos, ck[cell], umi_keys(n), [(0, 0, 0, n)], end=pos + 50)
    beg = np.arange(5, dtype=np.int32) * 10000
    return reads, ck, np.zeros(5, np.int32), beg, beg + 500


@pytest.mark.parametrize("n_cols", [65536, 65537])
def test_packed_layouts_at_their_boundaries(gpu_ctx, tmp_path, n_cols):
    from oracle import oracle
    reads, ck, gid, beg, end = boundary_batch(n_cols)
    conf = Conf()
    p = engine.make_params(conf, reads.max_aln_len, True)
    d = gpu_ctx.upload(reads)
    try:
        ref = [np.array(x) for x in gpu_ctx.basefc(d, gid, beg, end, ck, n_cols, p)[:3]]
        o = oracle.basefc(reads, gid, beg, end, ck, n_cols, oracle.params(conf), 4)
        assert all(np.array_equal(a, b) for a, b in zip(ref, o))
        assert ref[2].tolist() == [1, 2, 3, 1, 1, 15, 16, 2, 1, 1, 65534, 65535, 1]
        assert ref[1].max() == n_cols - 1
        host = d.download()             # a pinned copy of the batch for the streamed path
        for call, src in ((gpu_ctx.basefc, d), (gpu_ctx.basefc_host, host)):
            seg = check_layouts(gpu_ctx, src, call, gid, beg, end, ck, n_cols, p, ref)
            if n_cols <= 65536:         # narrow stays packed; exactly the count 65 535 is in the side list
                assert seg["narrow"].cv16 is not None and len(seg["narrow"].over[0]) == 1
                assert int(seg["narrow"].over[1][0]) == 65535
            else:
                assert seg["narrow"].cv16 is None
            t = seg["tiny"]
            assert t.tiny is not None and len(t.over[0]) == tiny_escapes(*ref)
            assert len(t.over[0]) == 9                   # 4 row starts; d = 4095 and 9999; n_cols - 1; 16; 65535
        host.close()
        emitted = np.ones(5, bool)
        check_text(gpu_ctx, tmp_path, d, gid, beg, end, ck, n_cols, p, ref, emitted, (1, 3))
    finally:
        d.close()


# ------------------------------------------------------------------------------------------ decimal widths
def widths_batch():
    """Rows, 1-based columns and counts at both sides of every decimal width.  Barcode mode: feature F_k has 10^k - 1
    molecules in column 10^k - 2 and 10^k in column 10^k - 1 (1-based 10^k - 1 and 10^k), k = 1..5.  Sample mode:
    features S_1..S_3 hold 999 999, 1 000 000 and 1 000 001 molecules.  The features sit at input rows 10^j - 2 and
    10^j - 1 (output rows 10^j - 1, 10^j), after rows that fetch nothing; every row is emitted."""
    cells, poss = [], []
    for k in range(1, 6):
        for c, v in ((10 ** k - 2, 10 ** k - 1), (10 ** k - 1, 10 ** k)):
            cells.append(np.full(v, c, np.int64))
            poss.append(k * 10000 + 100 + np.arange(v) % 200)
    n_bc = sum(len(c) for c in cells)
    s_pos = np.concatenate([np.full(999999, 100000), [120000, 130000]]).astype(np.int64)
    pos = np.concatenate(poss + [s_pos])
    cell = np.concatenate(cells + [np.full(len(s_pos), -1, np.int64)])
    order = np.argsort(pos, kind="stable")
    pos, cell = pos[order], cell[order]
    n_cols = 100000
    ck = cell_keys(n_cols)
    keys = np.where(cell >= 0, ck[np.maximum(cell, 0)], cell_keys(1, salt=n_cols + 7)[0])     # S reads: unlisted cell
    n = len(pos)
    reads = build(pos, keys, umi_keys(n), [(0, 0, 0, n)], end=pos + 50)
    real = [(k * 10000, k * 10000 + 500) for k in range(1, 6)] + [(100000, 100100), (100000, 120100), (100000, 130100)]
    slots = sorted({10 ** j - 2 for j in range(1, 7)} | {10 ** j - 1 for j in range(1, 7)})
    n_rows = slots[-1] + 3
    gid = np.full(n_rows, -1, np.int32)
    beg = np.zeros(n_rows, np.int32)
    end = np.full(n_rows, 100, np.int32)
    for i, r in enumerate(slots):
        gid[r], (beg[r], end[r]) = 0, real[i % len(real)]
    assert n_bc > 200000
    return reads, ck, n_cols, gid, beg, end


def test_device_mtx_text_at_every_decimal_width(gpu_ctx, tmp_path):
    from oracle import oracle
    reads, ck, n_cols, gid, beg, end = widths_batch()
    emitted = np.ones(len(gid), bool)
    d = gpu_ctx.upload(reads)
    try:
        for conf, keys, nc in ((Conf(), ck, n_cols), (Conf(barcodes=False), None, 1)):
            p = engine.make_params(conf, reads.max_aln_len, True)
            ref = [np.array(x) for x in gpu_ctx.basefc(d, gid, beg, end, keys, nc, p)[:3]]
            o = oracle.basefc(reads, gid, beg, end, keys, nc, oracle.params(conf), 4)
            assert all(np.array_equal(a, b) for a, b in zip(ref, o))
            vals = set(ref[2].tolist())
            if keys is not None:            # every width of columns (1-based) and counts
                assert {9, 10, 99, 100, 999, 1000, 9999, 10000, 99999, 100000} <= vals
                assert {9, 10, 99, 100, 999, 1000, 9999, 10000, 99999, 100000} <= set((ref[1] + 1).tolist())
            else:
                assert {999999, 1000000, 1000001} <= vals
                rows = set((ref[0] + 1).tolist())   # output row = input row + 1: every row is emitted
                assert {9, 10, 99, 100, 999, 1000, 9999, 10000, 99999, 100000, 999999, 1000000} <= rows
            check_layouts(gpu_ctx, d, gpu_ctx.basefc, gid, beg, end, keys, nc, p, ref)
            check_text(gpu_ctx, tmp_path, d, gid, beg, end, keys, nc, p, ref, emitted, (1, 8))
    finally:
        d.close()


# ------------------------------------------------------------------------------------------ wide matrices
SPREAD = 4096
N_CELLS = 1000


@pytest.fixture(scope="module")
def wide(gpu_ctx):
    """3 * 10^7 synthetic reads, 1 000 cells, 60 000 features; the key list places cell k at column 4096 k, the other
    columns hold keys that match no read."""
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 30000000, N_CELLS, 60000, seed=41)
    w.wide_keys = cell_keys(N_CELLS * SPREAD)
    w.wide_keys[::SPREAD] = w.cell_keys
    w.conf = Conf(min_mapq=20, min_len=30, min_include=0.9, excl_flag=772, no_orphan=True)
    w.p = engine.make_params(w.conf, 91, True)
    w.ref = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, N_CELLS, w.p)[:3]]
    yield w
    w.dreads.close()


def test_wide_matrix_side_list_overflow(gpu_ctx, wide):
    """Columns 4 096 apart: no entry is on the 16-bit grid, so the side list of the tiny layout overflows and the call
    comes back in plain 32-bit entries; the matrix is the compact one with its columns times 4 096.  (4 096 000
    columns: more than a segment feature's cell bitmap holds -- such a call used to fail before counting.)"""
    w = wide
    n_cols = N_CELLS * SPREAD
    ref = [w.ref[0], w.ref[1] * SPREAD, w.ref[2]]
    assert len(ref[2]) > TINY_OVER_CAP
    got = [np.array(x) for x in gpu_ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.wide_keys, n_cols, w.p)[:3]]
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    host = w.dreads.download()
    try:
        for call, src in ((gpu_ctx.basefc, w.dreads), (gpu_ctx.basefc_host, host)):
            seg = check_layouts(gpu_ctx, src, call, w.gid, w.beg, w.end, w.wide_keys, n_cols, w.p, ref)
            assert seg["narrow"].cv16 is None                              # > 65 536 columns
            assert seg["tiny"].tiny is None and seg["tiny"].cv16 is None    # side list full: plain entries
    finally:
        host.close()


def test_device_mtx_text_of_a_large_matrix(gpu_ctx, wide, tmp_path):
    """Hundreds of MB of text: many 32 MB chunks through one buffer (1 thread), a ring of 2, and of 8."""
    w = wide
    n_cols = N_CELLS * SPREAD
    ref = [w.ref[0], w.ref[1] * SPREAD, w.ref[2]]
    emitted = np.zeros(len(w.gid), bool)
    emitted[ref[0]] = True
    emitted[::5] = True                                  # and empty rows
    size = check_text(gpu_ctx, tmp_path, w.dreads, w.gid, w.beg, w.end, w.wide_keys, n_cols, w.p, ref, emitted,
                      (1, 2, 8))
    assert size > 3 * (32 << 20)
