"""ctypes binding of include/xcltk_b200.h (the C-ABI boundary).

The product path has no CPU fallback: if the library cannot be built/loaded or no CUDA
device is present, the device entry points raise `XgError`.
"""

import ctypes as C
import os

import numpy as np

from . import build as _build

XG_KEY_EMPTY = 0
XG_KEY_NONE = 0xFFFFFFFFFFFFFFFF
XG_KEY_NOMATCH = 0xFFFFFFFFFFFFFFFE
XG_TILE = 1024

c_i32p = C.POINTER(C.c_int32)
c_u32p = C.POINTER(C.c_uint32)
c_u16p = C.POINTER(C.c_uint16)
c_i64p = C.POINTER(C.c_int64)
c_u64p = C.POINTER(C.c_uint64)
c_u8p = C.POINTER(C.c_uint8)


XG_E_UNSUPPORTED = -7

# result layouts of xg_basefc (include/xcltk_b200.h), by Context.basefc's `segments`
XG_LAYOUT_CSR, XG_LAYOUT_ROWS, XG_LAYOUT_ROWS_NARROW, XG_LAYOUT_ROWS_TINY = 0, 1, 2, 3


class XgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("xcltk_b200 error %d: %s" % (code, msg))
        self.code = code


class Run(C.Structure):
    _fields_ = [("bam_idx", C.c_int32), ("gid", C.c_int32), ("rec_beg", C.c_int64), ("rec_end", C.c_int64)]


class Tile(C.Structure):
    _fields_ = [("rec_beg", C.c_int64), ("n_rec", C.c_int32), ("run", C.c_int32),
                ("first_pos", C.c_int32), ("max_end", C.c_int32)]


class Reads(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_cigar", C.c_int64), ("n_seq_words", C.c_int64),
                ("n_runs", C.c_int32), ("n_tiles", C.c_int32), ("max_aln_len", C.c_int32),
                ("max_span", C.c_int32), ("n_records_seen", C.c_int64),
                ("pos_end", c_i32p), ("fmq", c_u32p), ("cig_off", c_u32p), ("keys", c_u64p),
                ("seq_off", c_u32p), ("cigar", c_u32p), ("seq", c_u32p),
                ("runs", C.POINTER(Run)), ("tiles", C.POINTER(Tile))]


class Params(C.Structure):
    _fields_ = [("min_mapq", C.c_int32), ("min_len", C.c_int32), ("incl_flag", C.c_uint32),
                ("excl_flag", C.c_uint32), ("no_orphan", C.c_int32), ("use_cell_tag", C.c_int32),
                ("need_umi_tag", C.c_int32), ("min_incl_tab", c_i32p), ("min_incl_tab_len", C.c_int32),
                ("min_incl_len", C.c_int32)]


class Features(C.Structure):
    _fields_ = [("n", C.c_int32), ("gid", c_i32p), ("beg", c_i32p), ("end", c_i32p)]


class Barcodes(C.Structure):
    _fields_ = [("n", C.c_int32), ("keys", c_u64p), ("n_samples", C.c_int32)]


class Coo(C.Structure):
    _fields_ = [("nnz", C.c_int64), ("n_rows", C.c_int32), ("n_cols", C.c_int32),
                ("col", c_i32p), ("val", c_i32p), ("row_ptr", c_i64p),
                ("row_beg", c_i64p), ("row_cnt", c_i32p),
                ("colval16", c_u32p), ("n_over", C.c_int64), ("over_idx", c_i64p), ("over_val", c_i32p),
                ("coldelta16", c_u16p), ("over_col", c_i32p)]


class Snps(C.Structure):
    _fields_ = [("n", C.c_int32), ("gid", c_i32p), ("pos", c_i32p)]


class SnpFilter(C.Structure):
    _fields_ = [("ref_idx", c_u8p), ("alt_idx", c_u8p), ("min_count", C.c_double), ("min_maf", C.c_double)]


class SynthParams(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_cells", C.c_int32), ("read_len", C.c_int32),
                ("want_seq", C.c_int32), ("seed", C.c_uint64),
                ("n_spans", C.c_int32), ("span_gid", c_i32p), ("span_beg", c_i32p), ("span_end", c_i32p),
                ("n_snps", C.c_int32), ("snp_gid", c_i32p), ("snp_pos", c_i32p),
                ("snp_ref", c_u8p), ("snp_alt", c_u8p), ("snp_ref_hap", c_u8p),
                ("first_read", C.c_int64), ("total_reads", C.c_int64)]


# every symbol include/xcltk_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "xg_keyspace_create": (_P, []),
    "xg_keyspace_destroy": (None, [_P]),
    "xg_key_encode": (C.c_uint64, [_P, C.c_char_p, C.c_int64]),
    "xg_key_decode": (C.c_int64, [_P, C.c_uint64, C.c_char_p, C.c_int64]),
    "xg_keyspace_n_interned": (C.c_int64, [_P]),
    "xg_bam_header_read": (C.c_int, [C.c_char_p, C.POINTER(_P)]),
    "xg_bam_header_n_ref": (C.c_int32, [_P]),
    "xg_bam_header_ref_name": (C.c_char_p, [_P, C.c_int32]),
    "xg_bam_header_ref_len": (C.c_int64, [_P, C.c_int32]),
    "xg_bam_header_free": (None, [_P]),
    "xg_decode_bams": (C.c_int, [C.c_int32, C.POINTER(C.c_char_p), C.POINTER(c_i32p), c_i32p,
                                 C.c_char_p, C.c_char_p, C.c_int32, C.c_int32, _P,
                                 C.POINTER(C.POINTER(Reads))]),
    "xg_reads_free": (None, [C.POINTER(Reads)]),
    "xg_host_last_error": (C.c_char_p, []),
    "xg_write_mtx_rows": (C.c_int, [C.c_char_p, C.c_int32, c_i64p, c_i32p, c_i32p, C.c_int32, C.c_int32, c_i32p,
                                    c_i32p, C.c_int32]),
    "xg_write_mtx_rows16": (C.c_int, [C.c_char_p, C.c_int32, c_i64p, c_i32p, c_i32p, C.c_int32, C.c_int32, c_u32p,
                                      C.c_int64, c_i64p, c_i32p, C.c_int32]),
    "xg_write_mtx_rows_tiny": (C.c_int, [C.c_char_p, C.c_int32, c_i64p, c_i32p, c_i32p, C.c_int32, C.c_int32, c_u16p,
                                         C.c_int64, c_i64p, c_i32p, c_i32p, C.c_int32]),
    "xg_write_mtx": (C.c_int, [C.c_char_p, C.c_int32, c_i64p, c_i32p, C.c_int32, C.c_int32, c_i32p, c_i32p,
                               C.c_int32]),
    "xg_create": (C.c_int, [C.c_int32, C.POINTER(_P)]),
    "xg_destroy": (None, [_P]),
    "xg_last_error": (C.c_char_p, [_P]),
    "xg_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "xg_upload_reads": (C.c_int, [_P, C.POINTER(Reads), C.POINTER(_P)]),
    "xg_map_reads": (C.c_int, [_P, C.POINTER(Reads), C.POINTER(_P)]),
    "xg_download_reads": (C.c_int, [_P, _P, C.POINTER(C.POINTER(Reads))]),
    "xg_dreads_free": (None, [_P, _P]),
    "xg_dreads_n": (C.c_int64, [_P]),
    "xg_dreads_info": (None, [_P, c_i64p]),
    "xg_dreads_index": (None, [_P, C.POINTER(Run), C.POINTER(Tile)]),
    "xg_decode_bams_device": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(c_i32p), c_i32p,
                                        C.c_char_p, C.c_char_p, C.c_int32, _P, C.POINTER(_P), c_i64p]),
    "xg_bgzf_inflate_device": (C.c_int, [_P, C.c_char_p, c_u8p, C.c_int64, c_i64p]),
    "xg_coo_free": (None, [C.POINTER(Coo)]),
    "xg_basefc": (C.c_int, [_P, _P, C.POINTER(Features), C.POINTER(Barcodes), C.POINTER(Params), C.c_int32,
                            C.POINTER(C.POINTER(Coo))]),
    "xg_basefc_host": (C.c_int, [_P, C.POINTER(Reads), C.POINTER(Features), C.POINTER(Barcodes), C.POINTER(Params),
                                 C.c_int32, C.POINTER(C.POINTER(Coo))]),
    "xg_baf_pileup": (C.c_int, [_P, _P, C.POINTER(Snps), C.POINTER(Barcodes), C.POINTER(Params),
                                c_i64p, C.POINTER(_P)]),
    "xg_baf_count": (C.c_int, [_P, _P, C.c_int32, c_i64p, c_i32p, c_u8p, c_u8p, C.c_int32,
                               C.POINTER(C.POINTER(Coo)), C.POINTER(C.POINTER(Coo)),
                               C.POINTER(C.POINTER(Coo))]),
    "xg_baf_state_free": (None, [_P, _P]),
    "xg_basefc_write_mtx_device": (C.c_int, [_P, C.c_char_p, C.c_int32, c_i32p, C.c_int32, C.c_int32]),
    "xg_baf_fc": (C.c_int, [_P, _P, C.POINTER(Snps), C.POINTER(Barcodes), C.POINTER(Params), C.POINTER(SnpFilter),
                            C.c_int32, c_i64p, c_i32p, c_u8p, C.c_int32, c_i64p, c_u8p,
                            C.POINTER(C.POINTER(Coo)), C.POINTER(C.POINTER(Coo)), C.POINTER(C.POINTER(Coo))]),
    "xg_synth_reads": (C.c_int, [_P, C.POINTER(SynthParams), C.POINTER(_P), c_u64p]),
    "xg_synth_read_index": (C.c_int64, [C.POINTER(SynthParams), C.c_int32, C.c_int32]),
    "xg_write_bam": (C.c_int, [C.c_char_p, C.POINTER(Reads), C.c_int32, C.POINTER(C.c_char_p), c_i64p, _P,
                               C.c_char_p, C.c_char_p, C.c_int32, C.c_int32, C.c_int32]),
    "xg_decode_bams_device_range": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(c_i32p), c_i32p,
                                              C.c_char_p, C.c_char_p, C.c_int32, _P, c_i64p, c_i64p,
                                              C.POINTER(_P), C.POINTER(C.c_int64)]),
    "xg_bgzf_block_index": (C.c_int, [C.c_char_p, C.POINTER(c_i64p), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                      C.POINTER(C.c_int32)]),
    "xg_free_array": (None, [_P]),
    "xg_bam_block_probe": (C.c_int, [C.c_char_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "xg_last_timing": (None, [_P, C.POINTER(C.c_double)]),
    "xg_version": (C.c_char_p, []),
}

_lib = None


def lib_path():
    return _build.LIB


def load(rebuild=True):
    """Load (building first if sources are newer) and type every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if rebuild:
        try:
            path = _build.build()
        except Exception as ex:
            # A library that is older than its sources must not stand in for them: only when there is no compiler
            # (a box that got the prebuilt file) and the file exists is it loaded as it is.
            import shutil
            have_nvcc = bool(os.environ.get("NVCC") or shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc"))
            if have_nvcc or not os.path.exists(path):
                raise
            import logging
            logging.getLogger(__name__).warning("no compiler here (%s); loading the prebuilt %s", ex, path)
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)           # AttributeError = missing export: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def as_ptr(arr, ptype):
    return arr.ctypes.data_as(ptype)


def np_view(ptr, n, dtype):
    """Zero-copy numpy view of library-owned memory (valid until the owner is freed)."""
    if n <= 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    t = np.dtype(dtype)
    buf = (C.c_char * (n * t.itemsize)).from_address(C.addressof(ptr.contents))
    return np.frombuffer(buf, dtype=t, count=n)


class KeySpace(object):
    def __init__(self):
        self.lib = load()
        self.h = self.lib.xg_keyspace_create()

    def encode(self, s):
        b = s.encode("utf8") if isinstance(s, str) else bytes(s)
        return int(self.lib.xg_key_encode(self.h, b, len(b)))

    def decode(self, key):
        buf = C.create_string_buffer(4096)
        n = self.lib.xg_key_decode(self.h, C.c_uint64(key), buf, 4096)
        if n < 0:
            return None
        return buf.raw[:n].decode("utf8", "replace")

    def n_interned(self):
        return int(self.lib.xg_keyspace_n_interned(self.h))

    def close(self):
        if self.h:
            self.lib.xg_keyspace_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bam_references(path):
    """[(name, length)] of a BAM header (pysam: AlignmentFile.references / .lengths)."""
    lib = load()
    h = _P()
    rc = lib.xg_bam_header_read(path.encode(), C.byref(h))
    if rc != 0:
        raise XgError(rc, lib.xg_host_last_error().decode())
    try:
        n = lib.xg_bam_header_n_ref(h)
        return [(lib.xg_bam_header_ref_name(h, i).decode(), int(lib.xg_bam_header_ref_len(h, i)))
                for i in range(n)]
    finally:
        lib.xg_bam_header_free(h)


class HostReads(object):
    """A decoded batch (library-owned host memory) with numpy views."""

    def __init__(self, ptr):
        self.lib = load()
        self.ptr = ptr
        r = ptr.contents
        self.n = int(r.n_reads)
        self.n_records_seen = int(r.n_records_seen)
        self.max_aln_len = int(r.max_aln_len)
        self.max_span = int(r.max_span)
        self.pos_end = np_view(r.pos_end, 2 * self.n, np.int32).reshape(-1, 2)
        self.fmq = np_view(r.fmq, self.n, np.uint32)
        self.cig_off = np_view(r.cig_off, self.n, np.uint32)
        self.keys = np_view(r.keys, 2 * self.n, np.uint64).reshape(-1, 2)
        self.cigar = np_view(r.cigar, int(r.n_cigar), np.uint32)
        self.has_seq = bool(r.seq_off) and bool(r.seq)
        self.seq_off = np_view(r.seq_off, self.n, np.uint32) if self.has_seq else None
        self.seq = np_view(r.seq, int(r.n_seq_words), np.uint32) if self.has_seq else None
        self.runs = [(x.bam_idx, x.gid, x.rec_beg, x.rec_end) for x in
                     (r.runs[i] for i in range(r.n_runs))]
        self.n_tiles = int(r.n_tiles)

    def tiles(self):
        r = self.ptr.contents
        return [(t.rec_beg, t.n_rec, t.run, t.first_pos, t.max_end) for t in
                (r.tiles[i] for i in range(r.n_tiles))]

    def nbytes(self):
        r = self.ptr.contents
        b = self.n * (8 + 4 + 4 + 16) + int(r.n_cigar) * 4
        if self.has_seq:
            b += self.n * 4 + int(r.n_seq_words) * 4
        return b

    def close(self):
        if self.ptr is not None:
            for a in ("pos_end", "fmq", "cig_off", "keys", "cigar", "seq_off", "seq"):
                setattr(self, a, None)
            self.lib.xg_reads_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def decode_bams(paths, tid_maps, cell_tag, umi_tag, want_seq, keyspace, n_threads=0):
    lib = load()
    n = len(paths)
    cpaths = (C.c_char_p * n)(*[p.encode() for p in paths])
    maps = [np.ascontiguousarray(m, dtype=np.int32) for m in tid_maps]
    cmaps = (c_i32p * n)(*[as_ptr(m, c_i32p) for m in maps])
    lens = np.array([len(m) for m in maps], dtype=np.int32)
    out = C.POINTER(Reads)()
    rc = lib.xg_decode_bams(n, cpaths, cmaps, as_ptr(lens, c_i32p),
                            cell_tag.encode() if cell_tag else None,
                            umi_tag.encode() if umi_tag else None,
                            1 if want_seq else 0, n_threads, keyspace.h, C.byref(out))
    if rc != 0:
        raise XgError(rc, lib.xg_host_last_error().decode())
    return HostReads(out)


def write_mtx(path, row_ptr, out_row, n_rows_out, n_cols, col, val, n_threads=0):
    """CSR (all input rows) -> MatrixMarket text; out_row[r] = 1-based output row or 0."""
    lib = load()
    row_ptr = np.ascontiguousarray(row_ptr, dtype=np.int64)
    out_row = np.ascontiguousarray(out_row, dtype=np.int32)
    col = np.ascontiguousarray(col, dtype=np.int32)
    val = np.ascontiguousarray(val, dtype=np.int32)
    if len(col) == 0:
        col = np.zeros(1, dtype=np.int32)
        val = np.zeros(1, dtype=np.int32)
    rc = lib.xg_write_mtx(path.encode(), len(row_ptr) - 1, as_ptr(row_ptr, c_i64p), as_ptr(out_row, c_i32p),
                          int(n_rows_out), int(n_cols), as_ptr(col, c_i32p), as_ptr(val, c_i32p), n_threads)
    if rc != 0:
        raise XgError(rc, lib.xg_host_last_error().decode())


class _CooOwner(object):
    """Keeps a library-owned xg_coo alive while numpy views of it exist."""

    def __init__(self, lib, pcoo, ctx_obj=None):
        self.lib, self.pcoo, self.ctx_obj = lib, pcoo, ctx_obj   # ctx_obj: the Context must outlive us

    def __del__(self):
        try:
            self.lib.xg_coo_free(self.pcoo)
        except Exception:
            pass


class _View(np.ndarray):
    """ndarray view that carries a reference to the owner of its memory."""
    _owner = None

    def __array_finalize__(self, obj):
        self._owner = getattr(obj, "_owner", None)


class LazyRows(object):
    """Row indices of a CSR result, expanded from row_ptr on first use (np.asarray(rows),
    rows[...], len(rows)); the library then ships col / val / row_ptr only."""

    def __init__(self, row_ptr, nnz):
        self._ptr, self._n, self._rows = row_ptr, nnz, None

    def __len__(self):
        return self._n

    def __array__(self, dtype=None, copy=None):
        if self._rows is None:
            counts = np.diff(self._ptr)
            self._rows = np.repeat(np.arange(len(counts), dtype=np.int32), counts)
        return self._rows if dtype is None else self._rows.astype(dtype)

    def __getitem__(self, k):
        return np.asarray(self)[k]

    def tolist(self):
        return np.asarray(self).tolist()

    def astype(self, dtype):
        return np.asarray(self).astype(dtype)


class RowSegments(object):
    """basefc result with the rows in the order the device completed them (the rows layouts of
    xg_basefc): row r is entries [row_beg[r], row_beg[r] + row_cnt[r]), sorted by col.  The
    entries are either `col` / `val` (int32 each) or, in the narrow layout, `cv16` (uint32:
    column | count << 16, counts >= 65535 in the side list `over`); `.col` / `.val` unpack on
    demand.  This is what the Matrix-Market writer consumes (write_mtx_rows); to_sorted() gives
    (row, col, val) sorted by (row, col) for everything else."""

    def __init__(self, row_beg, row_cnt, col, val, shape, cv16=None, over=None, tiny=None):
        """tiny: the 16-bit layout (XG_LAYOUT_ROWS_TINY): (column - previous column of the row - 1) << 4 | count per entry,
        0 = the entry is in the side list `over` = (idx, val, col) -- every row's first entry is."""
        self.row_beg, self.row_cnt, self.shape = row_beg, row_cnt, shape
        self._col, self._val, self.cv16, self.over, self.tiny = col, val, cv16, over, tiny
        self.nnz = len(tiny) if tiny is not None else len(val) if cv16 is None else len(cv16)

    def _unpack_tiny(self):
        w = np.asarray(self.tiny)
        n = len(w)
        val = (w & np.uint16(15)).astype(np.int32)
        if n == 0:
            self._col, self._val = np.zeros(0, np.int32), val
            return
        step = (w >> np.uint16(4)).astype(np.int64) + 1
        esc = w == 0
        step[esc] = 0
        run = np.cumsum(step)
        idx, oval, ocol = self.over
        if int(esc.sum()) != len(idx):
            raise XgError(-1, "16-bit result layout: side list does not match the escape words")
        off = np.zeros(n, dtype=np.int64)
        off[idx] = ocol.astype(np.int64) - run[idx]
        last = np.maximum.accumulate(np.where(esc, np.arange(n, dtype=np.int64), 0))     # entry 0 starts a row
        val[idx] = oval
        self._col, self._val = (run + off[last]).astype(np.int32), val

    @property
    def col(self):
        if self._col is None:
            if self.tiny is not None:
                self._unpack_tiny()
            else:
                self._col = (np.asarray(self.cv16) & np.uint32(0xffff)).astype(np.int32)
        return self._col

    @property
    def val(self):
        if self._val is None:
            if self.tiny is not None:
                self._unpack_tiny()
                return self._val
            v = (np.asarray(self.cv16) >> np.uint32(16)).astype(np.int32)
            if self.over is not None and len(self.over[0]):
                v[self.over[0]] = self.over[1]
            self._val = v
        return self._val

    def to_sorted(self):
        cnt = self.row_cnt.astype(np.int64)
        row = np.repeat(np.arange(len(cnt), dtype=np.int32), cnt)
        ptr = np.concatenate([[0], np.cumsum(cnt)])
        src = np.repeat(self.row_beg - ptr[:-1], cnt) + np.arange(int(ptr[-1]), dtype=np.int64)
        return row, np.asarray(self.col)[src], np.asarray(self.val)[src]


def write_mtx_rows(path, seg, out_row, n_rows_out, n_threads=0):
    """RowSegments -> MatrixMarket text (xg_write_mtx_rows / xg_write_mtx_rows16)."""
    lib = load()
    out_row = np.ascontiguousarray(out_row, dtype=np.int32)
    args = (path.encode(), len(seg.row_cnt), as_ptr(seg.row_beg, c_i64p), as_ptr(seg.row_cnt, c_i32p),
            as_ptr(out_row, c_i32p), int(n_rows_out), int(seg.shape[1]))
    if seg.tiny is not None:
        tw = seg.tiny if seg.nnz else np.zeros(1, dtype=np.uint16)
        oi = np.ascontiguousarray(seg.over[0], dtype=np.int64)
        ov = np.ascontiguousarray(seg.over[1], dtype=np.int32)
        oc = np.ascontiguousarray(seg.over[2], dtype=np.int32)
        rc = lib.xg_write_mtx_rows_tiny(*args, as_ptr(tw, c_u16p), len(oi), as_ptr(oi, c_i64p) if len(oi) else None,
                                        as_ptr(oc, c_i32p) if len(oi) else None, as_ptr(ov, c_i32p) if len(oi) else None,
                                        n_threads)
    elif seg.cv16 is not None:
        cv = seg.cv16 if seg.nnz else np.zeros(1, dtype=np.uint32)
        oi = np.ascontiguousarray(seg.over[0], dtype=np.int64) if seg.over is not None else np.zeros(0, np.int64)
        ov = np.ascontiguousarray(seg.over[1], dtype=np.int32) if seg.over is not None else np.zeros(0, np.int32)
        rc = lib.xg_write_mtx_rows16(*args, as_ptr(cv, c_u32p), len(oi), as_ptr(oi, c_i64p) if len(oi) else None,
                                     as_ptr(ov, c_i32p) if len(ov) else None, n_threads)
    else:
        col, val = seg.col, seg.val
        if seg.nnz == 0:
            col = np.zeros(1, dtype=np.int32)
            val = np.zeros(1, dtype=np.int32)
        rc = lib.xg_write_mtx_rows(*args, as_ptr(col, c_i32p), as_ptr(val, c_i32p), n_threads)
    if rc != 0:
        raise XgError(rc, lib.xg_host_last_error().decode())


def _take(lib, pcoo, ctx_obj, views, copy):
    """Copies of `views` with the result freed at once, or views that keep it alive (a _CooOwner)."""
    if copy:
        out = [v.copy() for v in views]
        lib.xg_coo_free(pcoo)
        return out
    owner = _CooOwner(lib, pcoo, ctx_obj)
    out = [v.view(_View) for v in views]
    for v in out:
        v._owner = owner
    return out


def coo_to_numpy(lib, pcoo, copy_below=1 << 16, ctx_obj=None):
    """(row, col, val, shape) with `row` a LazyRows (expanded from row_ptr on use), or a RowSegments for the rows
    layouts.  Large results are zero-copy views of the library's pinned buffers (released when the last view dies);
    small ones are copied and freed at once."""
    m = pcoo.contents
    nnz = int(m.nnz)
    shape = (int(m.n_rows), int(m.n_cols))
    copy = nnz <= copy_below
    if not bool(m.row_beg):                   # CSR
        row_ptr = np_view(m.row_ptr, shape[0] + 1, np.int64).copy()
        col, val = _take(lib, pcoo, ctx_obj, [np_view(m.col, nnz, np.int32), np_view(m.val, nnz, np.int32)], copy)
        return LazyRows(row_ptr, nnz), col, val, shape
    row_beg = np_view(m.row_beg, shape[0], np.int64).copy()
    row_cnt = np_view(m.row_cnt, shape[0], np.int32).copy()
    n_over = int(m.n_over)
    if bool(m.coldelta16):                    # 16-bit entries; the side list holds about one entry per row
        tiny, idx, oval, ocol = _take(lib, pcoo, ctx_obj, [
            np_view(m.coldelta16, nnz, np.uint16), np_view(m.over_idx, n_over, np.int64),
            np_view(m.over_val, n_over, np.int32), np_view(m.over_col, n_over, np.int32)], copy)
        return RowSegments(row_beg, row_cnt, None, None, shape, over=(idx, oval, ocol), tiny=tiny)
    if bool(m.colval16):                      # narrow entries
        over = (np_view(m.over_idx, n_over, np.int64).copy(), np_view(m.over_val, n_over, np.int32).copy())
        cv, = _take(lib, pcoo, ctx_obj, [np_view(m.colval16, nnz, np.uint32)], copy)
        return RowSegments(row_beg, row_cnt, None, None, shape, cv16=cv, over=over)
    col, val = _take(lib, pcoo, ctx_obj, [np_view(m.col, nnz, np.int32), np_view(m.val, nnz, np.int32)], copy)
    return RowSegments(row_beg, row_cnt, col, val, shape)


class Context(object):
    """One per GPU (include/xcltk_b200.h: xg_ctx)."""

    def __init__(self, device=0):
        self.lib = load()
        self.device = device
        self.h = _P()
        rc = self.lib.xg_create(device, C.byref(self.h))
        if rc != 0:
            msg = self.lib.xg_last_error(self.h).decode() if self.h else "xg_create failed"
            if self.h:
                self.lib.xg_destroy(self.h)
                self.h = None
            raise XgError(rc, msg)

    def _check(self, rc):
        if rc != 0:
            raise XgError(rc, self.lib.xg_last_error(self.h).decode())

    def upload(self, host_reads):
        d = _P()
        self._check(self.lib.xg_upload_reads(self.h, host_reads.ptr, C.byref(d)))
        return DeviceReads(self, d)

    def decode_bams(self, paths, tid_maps, cell_tag, umi_tag, want_seq, keyspace=None, ranges=None):
        """BGZF inflate + BAM parse on the device (xg_decode_bams_device).  Returns
        (DeviceReads, n_records_seen), or None when the files need the host decoder.
        keyspace: interns the cell / UMI values that do not pack into 63 bits (query names,
        free-text barcodes); without it such files are left to the host decoder.
        ranges: [(lo, hi)] byte offsets of BGZF block starts per BAM -- only those blocks are decoded
        (xg_decode_bams_device_range; see bgzf_block_index / bam_block_probe)."""
        n = len(paths)
        cpaths = (C.c_char_p * n)(*[p.encode() for p in paths])
        maps = [np.ascontiguousarray(m, dtype=np.int32) for m in tid_maps]
        cmaps = (c_i32p * n)(*[as_ptr(m, c_i32p) for m in maps])
        lens = np.array([len(m) for m in maps], dtype=np.int32)
        d = _P()
        seen = C.c_int64(0)
        args = (self.h, n, cpaths, cmaps, as_ptr(lens, c_i32p), cell_tag.encode() if cell_tag else None,
                umi_tag.encode() if umi_tag else None, 1 if want_seq else 0,
                keyspace.h if keyspace is not None else None)
        if ranges is None:
            rc = self.lib.xg_decode_bams_device(*args, C.byref(d), C.byref(seen))
        else:
            lo = np.array([r[0] for r in ranges], dtype=np.int64)
            hi = np.array([r[1] for r in ranges], dtype=np.int64)
            rc = self.lib.xg_decode_bams_device_range(*args, as_ptr(lo, c_i64p), as_ptr(hi, c_i64p), C.byref(d),
                                                      C.byref(seen))
        if rc == XG_E_UNSUPPORTED:
            self.decode_fallback_reason = self.lib.xg_last_error(self.h).decode()
            return None
        self._check(rc)
        return DeviceReads(self, d), int(seen.value)

    def bgzf_inflate(self, path):
        """Inflate a BGZF file on the device; returns the bytes (validation of the inflate kernel)."""
        n = C.c_int64(0)
        self._check(self.lib.xg_bgzf_inflate_device(self.h, path.encode(), None, 0, C.byref(n)))
        out = np.empty(max(1, n.value), dtype=np.uint8)
        self._check(self.lib.xg_bgzf_inflate_device(self.h, path.encode(), as_ptr(out, c_u8p), n.value, C.byref(n)))
        return out[:n.value]

    def map_reads(self, host_reads):
        """Zero-copy batch for baf: only pos/end go to HBM; `host_reads` must stay alive."""
        d = _P()
        self._check(self.lib.xg_map_reads(self.h, host_reads.ptr, C.byref(d)))
        dr = DeviceReads(self, d)
        dr._host = host_reads
        return dr

    def timing(self):
        t = (C.c_double * 16)()
        self.lib.xg_last_timing(self.h, t)
        return list(t)

    def _basefc(self, entry, reads, gid, beg, end, cell_keys, n_samples, params, segments):
        gid = np.ascontiguousarray(gid, dtype=np.int32)
        beg = np.ascontiguousarray(beg, dtype=np.int32)
        end = np.ascontiguousarray(end, dtype=np.int32)
        keys = np.ascontiguousarray(cell_keys if cell_keys is not None else [], dtype=np.uint64)
        f = Features(len(gid), as_ptr(gid, c_i32p), as_ptr(beg, c_i32p), as_ptr(end, c_i32p))
        b = Barcodes(len(keys), as_ptr(keys, c_u64p), n_samples)
        if not segments:
            layout = XG_LAYOUT_CSR
        else:
            layout = {"narrow": XG_LAYOUT_ROWS_NARROW, "tiny": XG_LAYOUT_ROWS_TINY}.get(segments, XG_LAYOUT_ROWS)
        out = C.POINTER(Coo)()
        self._check(entry(self.h, reads, C.byref(f), C.byref(b), C.byref(params.c), layout, C.byref(out)))
        return coo_to_numpy(self.lib, out, ctx_obj=self)

    def basefc(self, dreads, gid, beg, end, cell_keys, n_samples, params, segments=False):
        """(row, col, val, shape) sorted by (row, col); segments=True: a RowSegments (rows in
        completion order, copied out while the counting is still running); segments="narrow": the
        same with 32-bit packed entries when there are at most 65536 columns; segments="tiny": 16-bit entries
        (column delta | small count) + a side list -- a quarter of the bytes, for matrices of small counts."""
        return self._basefc(self.lib.xg_basefc, dreads.h, gid, beg, end, cell_keys, n_samples, params, segments)

    def basefc_write_mtx(self, path, out_row, n_rows_out, n_threads=0):
        """Matrix-Market text of the LAST basefc(..., segments=...) result of this context, formatted on the device
        from the rows still in its staging area (xg_basefc_write_mtx_device): out_row[r] = 1-based output row of
        input row r, 0 = not emitted."""
        out_row = np.ascontiguousarray(out_row, dtype=np.int32)
        self._check(self.lib.xg_basefc_write_mtx_device(self.h, path.encode(), len(out_row), as_ptr(out_row, c_i32p),
                                                        int(n_rows_out), int(n_threads)))

    def basefc_host(self, host_reads, gid, beg, end, cell_keys, n_samples, params, segments=False):
        """basefc straight from a pinned host batch: H2D streamed under the counting kernels."""
        return self._basefc(self.lib.xg_basefc_host, host_reads.ptr, gid, beg, end, cell_keys, n_samples, params,
                            segments)

    def baf_pileup(self, dreads, gid, pos, cell_keys, n_samples, params, reuse_totals=False):
        """reuse_totals: the returned totals array is the context's own buffer, overwritten by the next pileup."""
        gid = np.ascontiguousarray(gid, dtype=np.int32)
        pos = np.ascontiguousarray(pos, dtype=np.int32)
        keys = np.ascontiguousarray(cell_keys if cell_keys is not None else [], dtype=np.uint64)
        s = Snps(len(gid), as_ptr(gid, c_i32p), as_ptr(pos, c_i32p))
        b = Barcodes(len(keys), as_ptr(keys, c_u64p), n_samples)
        # the library fills every entry; the array is reused from call to call (fresh pages cost more than the
        # copy itself) -- callers that keep the totals across pileups copy them
        totals = getattr(self, "_totals_buf", None) if reuse_totals else None
        if totals is None or totals.shape[0] != len(gid):
            totals = np.zeros((len(gid), 5), dtype=np.int64)
            if reuse_totals:
                self._totals_buf = totals
        st = _P()
        self._check(self.lib.xg_baf_pileup(self.h, dreads.h, C.byref(s), C.byref(b), C.byref(params.c),
                                           as_ptr(totals, c_i64p), C.byref(st)))
        return totals, BafState(self, st)

    def baf_count(self, state, reg_ptr, reg_snp, hap_of, keep, no_dup_hap):
        reg_ptr = np.ascontiguousarray(reg_ptr, dtype=np.int64)
        reg_snp = np.ascontiguousarray(reg_snp, dtype=np.int32)
        hap_of = np.ascontiguousarray(hap_of, dtype=np.uint8)
        keep = np.ascontiguousarray(keep, dtype=np.uint8)
        ad, dp, oth = C.POINTER(Coo)(), C.POINTER(Coo)(), C.POINTER(Coo)()
        self._check(self.lib.xg_baf_count(self.h, state.h, len(reg_ptr) - 1, as_ptr(reg_ptr, c_i64p),
                                          as_ptr(reg_snp, c_i32p), as_ptr(hap_of, c_u8p),
                                          as_ptr(keep, c_u8p), 1 if no_dup_hap else 0,
                                          C.byref(ad), C.byref(dp), C.byref(oth)))
        return tuple(coo_to_numpy(self.lib, m, ctx_obj=self) for m in (ad, dp, oth))

    def baf_fc(self, dreads, gid, pos, cell_keys, n_samples, params, ref_idx, alt_idx, min_count, min_maf,
               reg_ptr, reg_snp, hap_of, no_dup_hap, want_totals=False, want_keep=False):
        """Pileup, the SNP filter on the device and the region count in one library call (xg_baf_fc).
        Returns (ad, dp, oth[, totals][, keep])."""
        gid = np.ascontiguousarray(gid, dtype=np.int32)
        pos = np.ascontiguousarray(pos, dtype=np.int32)
        keys = np.ascontiguousarray(cell_keys if cell_keys is not None else [], dtype=np.uint64)
        ref_idx = np.ascontiguousarray(ref_idx, dtype=np.uint8)
        alt_idx = np.ascontiguousarray(alt_idx, dtype=np.uint8)
        reg_ptr = np.ascontiguousarray(reg_ptr, dtype=np.int64)
        reg_snp = np.ascontiguousarray(reg_snp, dtype=np.int32)
        hap_of = np.ascontiguousarray(hap_of, dtype=np.uint8)
        if len(ref_idx) != len(gid) or len(alt_idx) != len(gid) or hap_of.size != 8 * len(gid):
            raise ValueError("baf_fc: per-SNP arrays of different lengths")
        s = Snps(len(gid), as_ptr(gid, c_i32p), as_ptr(pos, c_i32p))
        b = Barcodes(len(keys), as_ptr(keys, c_u64p), n_samples)
        f = SnpFilter(as_ptr(ref_idx, c_u8p), as_ptr(alt_idx, c_u8p), float(min_count), float(min_maf))
        totals = np.zeros((len(gid), 5), dtype=np.int64) if want_totals else None
        keep = np.zeros(len(gid), dtype=np.uint8) if want_keep else None
        ad, dp, oth = C.POINTER(Coo)(), C.POINTER(Coo)(), C.POINTER(Coo)()
        self._check(self.lib.xg_baf_fc(self.h, dreads.h, C.byref(s), C.byref(b), C.byref(params.c), C.byref(f),
                                       len(reg_ptr) - 1, as_ptr(reg_ptr, c_i64p), as_ptr(reg_snp, c_i32p),
                                       as_ptr(hap_of, c_u8p), 1 if no_dup_hap else 0,
                                       as_ptr(totals, c_i64p) if want_totals else None,
                                       as_ptr(keep, c_u8p) if want_keep else None,
                                       C.byref(ad), C.byref(dp), C.byref(oth)))
        out = tuple(coo_to_numpy(self.lib, m, ctx_obj=self) for m in (ad, dp, oth))
        if want_totals:
            out += (totals,)
        if want_keep:
            out += (keep,)
        return out

    def synth_reads(self, n_reads, n_cells, span_gid, span_beg, span_end, seed=7, read_len=91,
                    want_seq=False, snps=None, first_read=0, total_reads=0):
        """total_reads > 0: only reads [first_read, first_read + n_reads) of a library of total_reads."""
        sg = np.ascontiguousarray(span_gid, dtype=np.int32)
        sb = np.ascontiguousarray(span_beg, dtype=np.int32)
        se = np.ascontiguousarray(span_end, dtype=np.int32)
        p = SynthParams()
        p.n_reads, p.n_cells, p.read_len, p.want_seq, p.seed = n_reads, n_cells, read_len, int(want_seq), seed
        p.n_spans, p.span_gid, p.span_beg, p.span_end = len(sg), as_ptr(sg, c_i32p), as_ptr(sb, c_i32p), as_ptr(se, c_i32p)
        p.first_read, p.total_reads = int(first_read), int(total_reads)
        keep = [sg, sb, se]
        if snps is not None:
            arrs = [np.ascontiguousarray(snps[0], dtype=np.int32), np.ascontiguousarray(snps[1], dtype=np.int32)] + \
                   [np.ascontiguousarray(a, dtype=np.uint8) for a in snps[2:5]]
            keep += arrs
            p.n_snps = len(arrs[0])
            p.snp_gid, p.snp_pos = as_ptr(arrs[0], c_i32p), as_ptr(arrs[1], c_i32p)
            p.snp_ref, p.snp_alt, p.snp_ref_hap = (as_ptr(a, c_u8p) for a in arrs[2:5])
        bk = np.zeros(n_cells, dtype=np.uint64)
        d = _P()
        self._check(self.lib.xg_synth_reads(self.h, C.byref(p), C.byref(d), as_ptr(bk, c_u64p)))
        return DeviceReads(self, d), bk

    def close(self):
        if self.h:
            self.lib.xg_destroy(self.h)
            self.h = None

    def synth_read_index(self, n_total, span_gid, span_beg, span_end, gid, pos, seed=7):
        return synth_read_index(n_total, span_gid, span_beg, span_end, gid, pos, seed)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bgzf_block_index(path):
    """(offsets of every BGZF block + the file size, block of the first record, starts-at-a-block-boundary)."""
    lib = load()
    p, n, first, al = c_i64p(), C.c_int64(0), C.c_int64(0), C.c_int32(0)
    rc = lib.xg_bgzf_block_index(path.encode(), C.byref(p), C.byref(n), C.byref(first), C.byref(al))
    if rc != 0:
        raise XgError(rc, lib.xg_host_last_error().decode())
    off = np.ctypeslib.as_array(p, shape=(n.value + 1,)).copy()
    lib.xg_free_array(C.cast(p, _P))
    return off, int(first.value), bool(al.value)


def bam_block_probe(path, offset):
    """(tid, pos) of the record at the beginning of the BGZF block at `offset`; tid -2: no record there."""
    lib = load()
    tid, pos = C.c_int32(0), C.c_int32(0)
    rc = lib.xg_bam_block_probe(path.encode(), int(offset), C.byref(tid), C.byref(pos))
    if rc != 0:
        raise XgError(rc, lib.xg_host_last_error().decode())
    return int(tid.value), int(pos.value)


def write_bam(path, host_reads, contigs, keyspace=None, cell_tag="CB", umi_tag="UB", level=1, n_threads=0,
              name_from_umi=False):
    """HostReads -> BAM file (xg_write_bam).  contigs: [(name, length)] in gid order."""
    lib = load()
    names = (C.c_char_p * len(contigs))(*[c[0].encode() for c in contigs])
    lens = np.array([c[1] for c in contigs], dtype=np.int64)
    rc = lib.xg_write_bam(path.encode(), host_reads.ptr, len(contigs), names, as_ptr(lens, c_i64p),
                          keyspace.h if keyspace is not None else None,
                          cell_tag.encode() if cell_tag else None, umi_tag.encode() if umi_tag else None,
                          1 if name_from_umi else 0, level, n_threads)
    if rc != 0:
        raise XgError(rc, lib.xg_host_last_error().decode())


def synth_read_index(n_total, span_gid, span_beg, span_end, gid, pos, seed=7):
    """First read of the synthetic library (xg_synth_reads) at or after (gid, pos).  Host only."""
    sg = np.ascontiguousarray(span_gid, dtype=np.int32)
    sb = np.ascontiguousarray(span_beg, dtype=np.int32)
    se = np.ascontiguousarray(span_end, dtype=np.int32)
    p = SynthParams()
    p.n_reads, p.seed = int(n_total), seed
    p.n_spans, p.span_gid, p.span_beg, p.span_end = len(sg), as_ptr(sg, c_i32p), as_ptr(sb, c_i32p), as_ptr(se, c_i32p)
    return int(load().xg_synth_read_index(C.byref(p), int(gid), int(pos)))


class DeviceReads(object):
    def __init__(self, ctx, h):
        self.ctx, self.h = ctx, h

    @property
    def n(self):
        return int(self.ctx.lib.xg_dreads_n(self.h))

    def info(self):
        v = (C.c_int64 * 8)()
        self.ctx.lib.xg_dreads_info(self.h, v)
        return dict(zip(("n_reads", "n_cigar", "n_seq_words", "n_runs", "n_tiles", "max_aln_len", "max_span",
                         "bytes"), [int(x) for x in v]))

    def index(self):
        """(runs, tiles) as the host decoder reports them: [(bam_idx, gid, rec_beg, rec_end)],
        [(rec_beg, n_rec, run, first_pos, max_end)]."""
        i = self.info()
        runs = (Run * max(1, i["n_runs"]))()
        tiles = (Tile * max(1, i["n_tiles"]))()
        self.ctx.lib.xg_dreads_index(self.h, runs, tiles)
        return ([(x.bam_idx, x.gid, x.rec_beg, x.rec_end) for x in runs[:i["n_runs"]]],
                [(t.rec_beg, t.n_rec, t.run, t.first_pos, t.max_end) for t in tiles[:i["n_tiles"]]])

    def download(self):
        out = C.POINTER(Reads)()
        self.ctx._check(self.ctx.lib.xg_download_reads(self.ctx.h, self.h, C.byref(out)))
        return HostReads(out)

    def close(self):
        if self.h and self.ctx.h:
            self.ctx.lib.xg_dreads_free(self.ctx.h, self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BafState(object):
    def __init__(self, ctx, h):
        self.ctx, self.h = ctx, h

    def close(self):
        if self.h and self.ctx.h:
            self.ctx.lib.xg_baf_state_free(self.ctx.h, self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ParamsBox(object):
    """xg_params plus the numpy array that backs min_incl_tab."""

    def __init__(self, min_mapq, min_len, incl_flag, excl_flag, no_orphan, use_cell_tag,
                 need_umi_tag, incl_tab=None, incl_len=0):
        self.tab = None if incl_tab is None else np.ascontiguousarray(incl_tab, dtype=np.int32)
        self.c = Params(int(min_mapq), int(min_len), int(incl_flag), int(excl_flag), int(bool(no_orphan)),
                        int(bool(use_cell_tag)), int(bool(need_umi_tag)),
                        as_ptr(self.tab, c_i32p) if self.tab is not None else None,
                        len(self.tab) if self.tab is not None else 0, int(incl_len))


class ArrayReads(object):
    """xg_reads assembled from caller-owned numpy arrays (same duck type as HostReads: `.ptr`
    for xg_upload_reads).  Used for record batches that do not come from xg_decode_bams."""

    def __init__(self, pos_end, fmq, cig_off, keys, cigar, runs, seq_off=None, seq=None,
                 max_aln_len=0, max_span=0):
        n = len(fmq)
        self.n = n
        a = self._arrays = {
            "pos_end": np.ascontiguousarray(pos_end, dtype=np.int32).reshape(-1),
            "fmq": np.ascontiguousarray(fmq, dtype=np.uint32),
            "cig_off": np.ascontiguousarray(cig_off, dtype=np.uint32),
            "keys": np.ascontiguousarray(keys, dtype=np.uint64).reshape(-1),
            "cigar": np.ascontiguousarray(cigar if len(cigar) else [0], dtype=np.uint32),
        }
        assert len(a["cig_off"]) == n + 1 and len(a["pos_end"]) == 2 * n and len(a["keys"]) == 2 * n
        self.has_seq = seq_off is not None and seq is not None
        if self.has_seq:
            a["seq_off"] = np.ascontiguousarray(seq_off, dtype=np.uint32)
            a["seq"] = np.ascontiguousarray(seq if len(seq) else [0], dtype=np.uint32)
        run_arr = (Run * max(1, len(runs)))()
        tiles = []
        pe = a["pos_end"].reshape(-1, 2)
        for k, (bam_idx, gid, rb, re_) in enumerate(runs):
            run_arr[k] = Run(int(bam_idx), int(gid), int(rb), int(re_))
            for s in range(int(rb), int(re_), XG_TILE):
                e = min(s + XG_TILE, int(re_))
                tiles.append(Tile(s, e - s, k, int(pe[s, 0]), int(pe[s:e, 1].max())))
        tile_arr = (Tile * max(1, len(tiles)))(*tiles)
        self._keep = (run_arr, tile_arr)
        self.runs = [tuple(int(x) for x in r) for r in runs]
        self.pos_end, self.fmq, self.keys = pe, a["fmq"], a["keys"].reshape(-1, 2)
        self.max_aln_len, self.max_span = int(max_aln_len), int(max_span)
        r = Reads()
        r.n_reads, r.n_cigar = n, len(cigar)
        r.n_seq_words = len(seq) if self.has_seq else 0
        r.n_runs, r.n_tiles = len(runs), len(tiles)
        r.max_aln_len, r.max_span, r.n_records_seen = int(max_aln_len), int(max_span), n
        r.pos_end, r.fmq = as_ptr(a["pos_end"], c_i32p), as_ptr(a["fmq"], c_u32p)
        r.cig_off, r.keys = as_ptr(a["cig_off"], c_u32p), as_ptr(a["keys"], c_u64p)
        r.cigar = as_ptr(a["cigar"], c_u32p)
        if self.has_seq:
            r.seq_off, r.seq = as_ptr(a["seq_off"], c_u32p), as_ptr(a["seq"], c_u32p)
        r.runs, r.tiles = C.cast(run_arr, C.POINTER(Run)), C.cast(tile_arr, C.POINTER(Tile))
        self._struct = r
        self.ptr = C.pointer(r)

    def nbytes(self):
        return sum(v.nbytes for v in self._arrays.values())

    def close(self):
        pass
