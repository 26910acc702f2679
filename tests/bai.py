"""A small BAI writer (SAMv1 section 5.2) for tests: the index a BAM's records give, built the way htslib's
hts_idx_push builds it -- reg2bin per record, chunks of consecutive records of a bin, the 16 kb linear index with
its holes filled, the pseudo-bin and n_no_coor -- from the virtual offsets of the records in the file's BGZF
layout.  Works for any BAM (synth.write_bam, xg_write_bam, htslib)."""

import struct
import zlib

from xcltk_b200.synth import reg2bin

PSEUDO_BIN = 37450


def bgzf_blocks(path):
    """[(file offset, inflated bytes)] of every BGZF block."""
    with open(path, "rb") as fp:
        data = fp.read()
    out, off = [], 0
    while off < len(data):
        xlen = struct.unpack_from("<H", data, off + 10)[0]
        bsize, x = None, off + 12
        while x < off + 12 + xlen:
            si1, si2, slen = data[x], data[x + 1], struct.unpack_from("<H", data, x + 2)[0]
            if si1 == 66 and si2 == 67:
                bsize = struct.unpack_from("<H", data, x + 4)[0]
            x += 4 + slen
        total = bsize + 1
        payload = data[off + 12 + xlen:off + total - 8]
        out.append((off, zlib.decompress(payload, -15) if payload else b""))
        off += total
    return out


def bam_records(path):
    """(n_ref, [(tid, pos, end, flag, voff_beg, voff_end)]) in file order; end as bam_endpos."""
    blocks = [(c, u) for c, u in bgzf_blocks(path)]
    stream = b"".join(u for _c, u in blocks)
    starts, at = [], 0
    for c, u in blocks:
        starts.append((at, c, len(u)))
        at += len(u)
    nonempty = [s for s in starts if s[2] > 0]

    def voff(u, as_end):
        # start: the block holding byte u; end: the block holding byte u - 1 (what bgzf_tell gives after a write)
        key = u - 1 if as_end else u
        lo, hi = 0, len(nonempty) - 1
        while lo < hi:
            mid = (lo + hi + 1) // 2
            if nonempty[mid][0] <= key:
                lo = mid
            else:
                hi = mid - 1
        ub, c, _n = nonempty[lo]
        return (c << 16) | (u - ub)

    o = 8 + struct.unpack_from("<i", stream, 4)[0]
    n_ref = struct.unpack_from("<i", stream, o)[0]
    o += 4
    for _ in range(n_ref):
        o += 8 + struct.unpack_from("<i", stream, o)[0]
    recs = []
    while o < len(stream):
        bs = struct.unpack_from("<i", stream, o)[0]
        tid, pos = struct.unpack_from("<ii", stream, o + 4)
        l_name = stream[o + 12]
        n_cig, flag = struct.unpack_from("<HH", stream, o + 16)
        cig = struct.unpack_from("<%dI" % n_cig, stream, o + 36 + l_name)
        rlen = sum(w >> 4 for w in cig if (w & 15) in (0, 2, 3, 7, 8))
        end = pos + (rlen if rlen > 0 and not (flag & 4) else 1)
        recs.append((tid, pos, end, flag, voff(o, False), voff(o + 4 + bs, True)))
        o += 4 + bs
    return n_ref, recs


def build_index(n_ref, recs):
    """[({bin: [(beg, end)]}, [linear offsets], (n_mapped, n_unmapped))] per contig, and n_no_coor."""
    refs = [({}, [], [0, 0], [None, None]) for _ in range(n_ref)]
    n_no_coor = 0
    for tid, pos, end, flag, vb, ve in recs:
        if tid < 0:
            n_no_coor += 1
            continue
        bins, lin, counts, span = refs[tid]
        b = reg2bin(pos, end)
        ch = bins.setdefault(b, [])
        if ch and ch[-1][1] == vb:
            ch[-1] = (ch[-1][0], ve)
        else:
            ch.append((vb, ve))
        for w in range(pos >> 14, ((end - 1) >> 14) + 1):
            while len(lin) <= w:
                lin.append(None)
            if lin[w] is None:
                lin[w] = vb
        counts[1 if flag & 4 else 0] += 1
        span[0] = vb if span[0] is None else span[0]
        span[1] = ve
    out = []
    for bins, lin, counts, span in refs:
        first = next((v for v in lin if v is not None), 0)
        filled, prev = [], None
        for v in lin:                       # holes: the contig's first offset before any entry, else the previous one
            prev = v if v is not None else (prev if prev is not None else first)
            filled.append(prev)
        out.append((bins, filled, tuple(counts), tuple(span)))
    return out, n_no_coor


def write_bai(path, n_ref, recs, pseudo_bin=True, extra_refs=0):
    index, n_no_coor = build_index(n_ref, recs)
    buf = bytearray(b"BAI\1" + struct.pack("<i", n_ref + extra_refs))
    for bins, lin, counts, span in index + [({}, [], (0, 0), (None, None))] * extra_refs:
        items = sorted(bins.items())
        with_pseudo = pseudo_bin and span[0] is not None
        buf += struct.pack("<i", len(items) + (1 if with_pseudo else 0))
        for b, chunks in items:
            buf += struct.pack("<Ii", b, len(chunks))
            for cb, ce in chunks:
                buf += struct.pack("<QQ", cb, ce)
        if with_pseudo:
            buf += struct.pack("<IiQQQQ", PSEUDO_BIN, 2, span[0], span[1], counts[0], counts[1])
        buf += struct.pack("<i", len(lin))
        buf += b"".join(struct.pack("<Q", v) for v in lin)
    buf += struct.pack("<Q", n_no_coor)
    with open(path, "wb") as fp:
        fp.write(bytes(buf))
    return index


def index_bam(bam_path, bai_path=None, **kw):
    """Write <bam>.bai (or bai_path); returns (n_ref, records, index)."""
    n_ref, recs = bam_records(bam_path)
    index = write_bai(bai_path or bam_path + ".bai", n_ref, recs, **kw)
    return n_ref, recs, index


def reg2bins(beg, end):
    """SAMv1 section 5.3: the bins that overlap 0-based [beg, end)."""
    end -= 1
    out = [0]
    for first, shift in ((1, 26), (9, 23), (73, 20), (585, 17), (4681, 14)):
        out += range(first + (beg >> shift), first + (end >> shift) + 1)
    return out


def query_ranges(path, index, intervals, merge_gap, linear=True):
    """The ranges xg_bam_index_ranges documents, computed from an index as build_index returns it: the chunks of the
    reg2bins bins that end after the linear-index offset of the interval's start (linear=False: all of them), merged,
    widened to the end of their last block, merged again across gaps below merge_gap; (virtual offset of the first
    record, file offset after the last block)."""
    import os
    starts = [c for c, _u in bgzf_blocks(path)]
    after = dict(zip(starts, starts[1:] + [os.path.getsize(path)]))
    visit = {}
    for t, b, e in intervals:
        if t < 0 or t >= len(index):
            continue
        b, e = max(0, b), min(e, 1 << 29)
        bins, lin = index[t][0], index[t][1]
        if e <= b or not bins:
            continue
        mo = lin[b >> 14] if linear and (b >> 14) < len(lin) else 0
        for k in reg2bins(b, e):
            if k in bins:
                visit[(t, k)] = min(visit.get((t, k), mo), mo)
    ch = sorted((cb, ce) for (t, k), mo in visit.items() for cb, ce in index[t][0][k] if ce > mo and ce > cb)
    merged = []
    for cb, ce in ch:
        if merged and cb <= merged[-1][1]:
            merged[-1][1] = max(merged[-1][1], ce)
        else:
            merged.append([cb, ce])
    out = []
    for cb, ce in merged:
        hi = after[ce >> 16] if ce & 0xffff else ce >> 16
        if hi <= cb >> 16:
            continue
        if out and (cb >> 16) <= out[-1][1] + merge_gap:
            out[-1][1] = max(out[-1][1], hi)
        else:
            out.append([cb, hi])
    return [tuple(r) for r in out]
