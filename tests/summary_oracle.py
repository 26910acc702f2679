"""ctypes front end of tests/summary_oracle.c: orc_basefc_summary, the CPU oracle of basefc's read-assignment summary
(xg_basefc_summary).  Test infrastructure only: compiled on first use into a temporary directory, together with the
basefc oracle it builds on (oracle/xg_oracle.c, included unchanged)."""

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "summary_oracle.c")
FATES = ("mapq", "flag", "no_umi", "short", "not_included", "one_feature", "multi_feature")

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u64p = C.POINTER(C.c_uint64)

_lib = None


def load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="xg_summary_oracle_"), "libsummary_oracle.so")
        base = ["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-o", out, SRC]
        if subprocess.run(base[:-3] + ["-fopenmp"] + base[-3:], capture_output=True).returncode != 0:
            subprocess.run(base, check=True, capture_output=True)
        _lib = C.CDLL(out)
        _lib.orc_basefc_summary.restype = C.c_int
    return _lib


def _ptr(a, t):
    return a.ctypes.data_as(t)


def summary(host_reads, gid, beg, end, cell_keys, n_samples, par, own=None, n_threads=8):
    """(n_samples + 1, 7) int64: the records in range of a feature per column (last row: no listed cell) and fate.
    par: oracle.params(conf); own: None or (gid_lo, pos_lo, gid_hi, pos_hi)."""
    lib = load()
    g, b, e = (np.ascontiguousarray(a, dtype=np.int32) for a in (gid, beg, end))
    keys = np.ascontiguousarray(cell_keys if cell_keys is not None else [], dtype=np.uint64)
    own_arr = None if own is None else np.ascontiguousarray(own, dtype=np.int32)
    out = np.zeros((n_samples + 1, len(FATES)), dtype=np.int64)
    rc = lib.orc_basefc_summary(host_reads.ptr, C.c_int32(len(g)), _ptr(g, c_i32p), _ptr(b, c_i32p), _ptr(e, c_i32p),
                                C.c_int32(len(keys)), _ptr(keys, c_u64p), C.c_int32(n_samples), C.byref(par),
                                None if own_arr is None else _ptr(own_arr, c_i32p), C.c_int32(n_threads),
                                _ptr(out, c_i64p))
    if rc != 0:
        raise MemoryError("orc_basefc_summary failed")
    return out


def params(conf):
    return oracle.params(conf)
