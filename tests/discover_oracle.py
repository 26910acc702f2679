"""ctypes front end of tests/discover_oracle.c (orc_snp_discover), the CPU oracle of SNP discovery.  Test
infrastructure only: it is compiled on first use into a temporary directory, together with the baf oracle it
builds on (oracle/xg_oracle.c, included unchanged)."""

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "discover_oracle.c")

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u8p = C.POINTER(C.c_uint8)
c_u64p = C.POINTER(C.c_uint64)


class OrcSites(C.Structure):
    _fields_ = [("n", C.c_int64), ("cap", C.c_int64), ("gid", c_i32p), ("pos", c_i32p), ("ref", c_u8p),
                ("alt", c_u8p), ("tot", c_i64p)]


_lib = None


def load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="xg_discover_oracle_"), "libdiscover_oracle.so")
        base = ["/usr/bin/gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-o", out, SRC]
        if subprocess.run(base[:-3] + ["-fopenmp"] + base[-3:], capture_output=True).returncode != 0:
            subprocess.run(base, check=True, capture_output=True)
        _lib = C.CDLL(out)
        _lib.orc_snp_discover.restype = C.c_int
    return _lib


def _ptr(a, t):
    return a.ctypes.data_as(t)


def orc_snp_discover(host_reads, tg_gid, tg_beg, tg_end, cell_keys, par, min_count, min_maf, n_threads=8):
    """Discovered sites (dict of gid, pos, ref, alt, totals as Context.snp_discover returns them) by brute force
    over every covered target position.  par: oracle.params(conf)."""
    lib = load()
    g, b, e = (np.ascontiguousarray(a, dtype=np.int32) for a in (tg_gid, tg_beg, tg_end))
    keys = np.ascontiguousarray(cell_keys if cell_keys is not None else [], dtype=np.uint64)
    out = OrcSites()
    rc = lib.orc_snp_discover(host_reads.ptr, C.c_int32(len(g)), _ptr(g, c_i32p), _ptr(b, c_i32p), _ptr(e, c_i32p),
                              C.c_int32(len(keys)), _ptr(keys, c_u64p), C.byref(par), C.c_double(float(min_count)),
                              C.c_double(float(min_maf)), C.c_int32(n_threads), C.byref(out))
    if rc != 0:
        raise MemoryError("orc_snp_discover failed")
    n = int(out.n)

    def arr(p, dt, k=1):
        return np.ctypeslib.as_array(p, shape=(n * k,)).astype(dt) if n else np.zeros(0, dt)
    res = {"gid": arr(out.gid, np.int32), "pos": arr(out.pos, np.int32), "ref": arr(out.ref, np.uint8),
           "alt": arr(out.alt, np.uint8), "totals": arr(out.tot, np.int64, 5).reshape(n, 5)}
    lib.orc_sites_free(C.byref(out))
    return res


def params(conf):
    return oracle.params(conf)
