"""A DEFLATE (RFC 1951) writer that makes the choices zlib makes for you: explicit code lengths,
explicit run-length plans for the code lengths, block kinds in any order, codes zlib never writes
(a lone 1-bit distance code, 15-bit codes on the all-ones codeword) and invalid fields one at a
time.  Every stream it writes is checked with zlib (`check`), so the writer is tested against the
reference before any decoder sees its output.

`batches` models how inflate_group<32> (xcltk_b200/csrc/inflate.cuh) cuts a block into batches,
so that a case can assert which switch of the 32-lane write path it reaches."""

import struct
import zlib

LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227,
         258]
LEXT = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
         6145, 8193, 12289, 16385, 24577]
DEXT = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
EOB = 256
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32


def len_sym(n):
    """(symbol, extra value) of a match length; 258 is symbol 285"""
    if n == 258:
        return 285, 0
    k = max(i for i in range(28) if LBASE[i] <= n)
    return 257 + k, n - LBASE[k]


def dist_sym(d):
    k = max(i for i in range(30) if DBASE[i] <= d)
    return k, d - DBASE[k]


def canonical(lens):
    """RFC 1951 3.2.2: symbol -> (code, length) for every symbol of non-zero length"""
    count = [0] * 16
    for l in lens:
        count[l] += 1
    count[0] = 0
    nxt, code = [0] * 16, 0
    for l in range(1, 16):
        code = (code + count[l - 1]) << 1
        nxt[l] = code
    out = {}
    for s, l in enumerate(lens):
        if l:
            out[s] = (nxt[l], l)
            nxt[l] += 1
    return out


def skewed(symbols):
    """lengths 1, 2, ..., L-1, L, L for symbols[0], ..., symbols[L]: a complete code whose two longest
    codes are L bits; the larger of the last two symbols gets the all-ones codeword"""
    L = len(symbols) - 1
    return {s: min(i + 1, L) for i, s in enumerate(symbols)}


def flat(symbols):
    """a complete code over the given symbols with lengths as even as possible"""
    k = len(symbols)
    if k == 1:
        return {symbols[0]: 1}
    d = (k - 1).bit_length()
    short = (1 << d) - k
    return {s: d - 1 if i < short else d for i, s in enumerate(symbols)}


def lens_list(lens, n):
    out = [0] * n
    for s, l in lens.items():
        out[s] = l
    return out


class BitWriter:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, v, n):                   # fields: least significant bit first
        self.acc |= (v & ((1 << n) - 1)) << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, c, l):                   # Huffman codes: most significant bit first
        self.bits(int(format(c, "0%db" % l)[::-1], 2), l)

    def align(self):
        if self.n:
            self.bits(0, 8 - self.n)

    def getvalue(self):
        return bytes(self.out) + (bytes([self.acc]) if self.n else b"")


class Deflate:
    """One raw DEFLATE stream built block by block.  A symbol is a literal (0..255), EOB (256), a match
    (length, distance), or a raw match (length symbol, extra, distance symbol, extra) for fields the
    first form cannot spell.  `payload` is what the stream inflates to (None once a raw field makes it
    undefined); `size` counts the bytes its symbols stand for taken at face value (a match reaching before
    the output included, a symbol without a length left out); `blocks` records per block its kind, output
    offset and symbols; `used` records per coded symbol (alphabet, code length, whether it is the all-ones
    codeword)."""

    def __init__(self):
        self.w = BitWriter()
        self.payload = bytearray()
        self.size = 0
        self.blocks = []
        self.used = set()
        self.end_bits = []                  # bit position (mod 8) where each block's last code ended

    def _header(self, final, kind):
        self.w.bits(1 if final else 0, 1)
        self.w.bits(kind, 2)

    def stored(self, data, final=False):
        self._header(final, 0)
        self.w.align()
        self.w.bits(len(data), 16)
        self.w.bits(len(data) ^ 0xffff, 16)
        for b in data:
            self.w.bits(b, 8)
        self.blocks.append(("stored", len(self.payload), list(data)))
        self.payload += data
        self.size += len(data)
        return self

    def fixed(self, symbols, final=False):
        self._header(final, 1)
        return self._symbols("fixed", symbols, FIXED_LIT, FIXED_DIST)

    def dynamic(self, symbols, lit_lens, dist_lens, final=False, hclen=19, cl_plan=None, cl_lens=None):
        """lit_lens / dist_lens: lists of HLIT / HDIST code lengths (dicts are expanded to 257 / 1 entries
        at least, or to cover their largest symbol); cl_plan: the code-length symbols, each a length 0..15
        or (16 | 17 | 18, repeat); cl_lens: code lengths of the code-length code (default: a flat code over
        the symbols the plan uses)"""
        if isinstance(lit_lens, dict):
            lit_lens = lens_list(lit_lens, max(257, max(lit_lens) + 1))
        if isinstance(dist_lens, dict):
            dist_lens = lens_list(dist_lens, max(1, max(dist_lens) + 1))
        seq = list(lit_lens) + list(dist_lens)
        plan = list(seq) if cl_plan is None else cl_plan
        if cl_lens is None:
            kinds = sorted({p if isinstance(p, int) else p[0] for p in plan})
            if len(kinds) == 1:                 # the code-length code must be complete: add a second symbol
                kinds.append(next(k for k in CL_ORDER[:hclen] if k not in kinds))
            cl_lens = lens_list(flat(kinds), 19)
        self._header(final, 2)
        self.w.bits(len(lit_lens) - 257, 5)
        self.w.bits(len(dist_lens) - 1, 5)
        self.w.bits(hclen - 4, 4)
        for k in range(hclen):
            self.w.bits(cl_lens[CL_ORDER[k]], 3)
        assert all(cl_lens[CL_ORDER[k]] == 0 for k in range(hclen, 19))
        codes = canonical(cl_lens)
        for p in plan:
            s, rep = (p, None) if isinstance(p, int) else p
            self.w.code(*codes[s])
            if s == 16:
                self.w.bits(rep - 3, 2)
            elif s == 17:
                self.w.bits(rep - 3, 3)
            elif s == 18:
                self.w.bits(rep - 11, 7)
        return self._symbols("dynamic", symbols, lit_lens, dist_lens)

    def _symbols(self, kind, symbols, lit_lens, dist_lens):
        lc, dc = canonical(lit_lens), canonical(dist_lens)
        top_l = {l: max(c for c, ll in lc.values() if ll == l) for _, l in lc.values()}
        top_d = {l: max(c for c, ll in dc.values() if ll == l) for _, l in dc.values()}
        start = len(self.payload)

        def put(table, top, alpha, s):
            c, l = table[s]
            self.w.code(c, l)
            self.used.add((alpha, l, c == top[l] and c == (1 << l) - 1))

        for sym in symbols:
            if isinstance(sym, int):
                put(lc, top_l, "lit", sym)
                if sym < 256:
                    self.size += 1
                    if self.payload is not None:
                        self.payload.append(sym)
                continue
            if len(sym) == 2:
                n, d = sym
                (ls, le), (ds, de) = len_sym(n), dist_sym(d)
            else:
                ls, le, ds, de = sym
                n = LBASE[ls - 257] + le if 257 <= ls <= 285 else None
                d = DBASE[ds] + de if ds < 30 else None
            put(lc, top_l, "lit", ls)
            self.w.bits(le, LEXT[ls - 257] if ls <= 285 else 0)
            put(dc, top_d, "dist", ds)
            self.w.bits(de, DEXT[ds] if ds < 30 else 0)
            self.size += n or 0
            if self.payload is None or n is None or d is None or d > len(self.payload):
                self.payload = None
                continue
            for _ in range(n):
                self.payload.append(self.payload[-d])
        self.end_bits.append(self.w.n)
        self.blocks.append((kind, start, list(symbols)))
        return self

    def raw(self):
        return self.w.getvalue()


def member(raw, payload, isize=None):
    """a BGZF member around a raw DEFLATE stream (as synth._bgzf_block writes one)"""
    bsize = len(raw) + 25
    assert bsize <= 65535
    head = struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, bsize)
    return head + raw + struct.pack("<II", zlib.crc32(payload) & 0xffffffff, len(payload) if isize is None else isize)


def check(stream):
    """zlib's reading of the stream must be the payload the writer meant; returns (raw, payload)"""
    raw = stream.raw()
    got = zlib.decompress(raw, -15)
    assert stream.payload is not None and got == bytes(stream.payload)
    return raw, bytes(stream.payload)


def zlib_rejects(raw):
    try:
        d = zlib.decompressobj(-15)
        d.decompress(raw)
        return not d.eof
    except zlib.error:
        return True


def batches(stream, S=32):
    """inflate_group<S>'s batches over the Huffman blocks of a stream: lane 0 queues up to S symbols and an
    EOB ends the batch (an EOB right after S symbols makes a batch of its own).  Per match: its batch
    (block, index), the batch start o, its offset, whether it reads bytes of its own batch (`dep`: the
    ordered loop) and whether the last byte it reads is written in the same 32-byte round as its first
    byte (`same_round`).  Also per batch its symbol count."""
    matches, sizes = [], []
    for bi, (kind, start, symbols) in enumerate(stream.blocks):
        if kind == "stored":
            continue
        o, k, q = start, 0, []

        def flush(o, q, k):
            off = o
            for i, sym in enumerate(q):
                if isinstance(sym, int):
                    off += 1
                    continue
                n, d = sym
                dep = off - d + min(n, d) > o
                last_src = off - d + min(n, d) - 1
                matches.append(dict(block=bi, batch=k, o=o, off=off, len=n, dist=d, first=i == 0,
                                    last=i == len(q) - 1, n=len(q), dep=dep,
                                    same_round=dep and (last_src - o) // 32 == (off - o) // 32))
                off += n
            sizes.append((bi, k, len(q)))
            return off

        for sym in symbols:
            if sym == EOB:
                o = flush(o, q, k)
                q, k = [], k + 1
                break
            q.append(sym)
            if len(q) == S:
                o = flush(o, q, k)
                q, k = [], k + 1
    return matches, sizes
