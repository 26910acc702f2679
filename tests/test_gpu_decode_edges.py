"""The device BAM decoder (gpu_decode.cu + inflate.cuh) at its switches.

Inflate: the crafted DEFLATE members of inflate_cases.py (codes zlib never writes, table edges, 32-lane batch
boundaries, invalid fields) through k_inflate, byte for byte against zlib, and BAM blocks re-encoded with those
stream kinds under real records.  Record parse: blocks of 31 / 32 / 33 / 63 / 64 / 65 records (k_extract's 32-link
batches), contig changes and dropped contigs on those links, CIGARs around the 255-op escape, sequence tails,
cell / UMI tags behind every aux type, keys at the 63-bit packing limit, a header that shares its block with records,
empty BGZF blocks and an index range that starts in that shared block.  The reference is the host decoder
(decode.cpp), array for array."""

import gzip
import random
import struct

import numpy as np
import pytest

import bai
import deflate_craft as dc
import inflate_cases as ic
from deflate_craft import EOB, Deflate
from test_decode import limit_keys, packs
from test_gpu_decode import assert_same_batch, full_maps, host_decode

pytestmark = pytest.mark.gpu

VALID = ic.valid_cases()
REJECT = ic.reject_cases()
XG_E_FORMAT = -3


def write_members(path, members):
    from xcltk_b200 import synth
    with open(path, "wb") as fp:
        fp.write(b"".join(members) + synth.BGZF_EOF)


# ---- inflate ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", sorted(VALID))
def test_crafted_stream_inflates_like_zlib(gpu_ctx, tmp_path, name):
    members, payloads = zip(*(ic.member_of(s) for s in VALID[name]))
    p = str(tmp_path / "c.bgzf")
    write_members(p, members)
    assert gpu_ctx.bgzf_inflate(p).tobytes() == b"".join(payloads)


@pytest.mark.parametrize("name", sorted(REJECT))
def test_crafted_invalid_stream_is_a_format_error(gpu_ctx, tmp_path, name):
    from xcltk_b200 import lib
    good = ic.member_of(VALID["batch_32_literals"][0])[0]
    p = str(tmp_path / "r.bgzf")
    write_members(p, [good, ic.member_of(REJECT[name], reject=True)[0], good])
    with pytest.raises(lib.XgError) as ei:
        gpu_ctx.bgzf_inflate(p)
    assert ei.value.code == XG_E_FORMAT
    write_members(p, [good, good])                       # the context is still usable
    assert len(gpu_ctx.bgzf_inflate(p)) == 64


def test_all_crafted_streams_side_by_side(gpu_ctx, tmp_path):
    """every valid member in one file, three times in different orders: many warps decode different stream
    kinds next to each other"""
    pairs = [ic.member_of(s) for name in sorted(VALID) for s in VALID[name]]
    rng = random.Random(1)
    for _ in range(3):
        rng.shuffle(pairs)
        p = str(tmp_path / "all.bgzf")
        write_members(p, [m for m, _ in pairs])
        with gzip.open(p, "rb") as fp:
            exp = fp.read()
        assert exp == b"".join(pl for _, pl in pairs)
        assert gpu_ctx.bgzf_inflate(p).tobytes() == exp


# ---- BAM blocks written with the crafted stream kinds -------------------------------------------------------------

def lz77(data, d1_only=False):
    """greedy LZ77 symbols of `data` (matches of 3..258 within 32 KiB; only distance 1 with d1_only)"""
    out, last, i, n = [], {}, 0, len(data)
    while i < n:
        best, bd = 0, 0
        cands = [i - 1] if d1_only else ([last[data[i:i + 3]]] if data[i:i + 3] in last else [])
        for j in cands:
            if j < 0 or i - j > 32768:
                continue
            k = 0
            while k < 258 and i + k < n and data[j + k] == data[i + k]:
                k += 1
            if k > best:
                best, bd = k, i - j
        if best >= 3:
            out.append((best, bd))
            for k in range(best):
                last[data[i + k:i + k + 3]] = i + k
            i += best
        else:
            out.append(data[i])
            last[data[i:i + 3]] = i
            i += 1
    return out


def _flat_dynamic(s, syms, final=True, d1=False):
    lit, dist = {EOB}, set()
    for x in syms:
        if isinstance(x, int):
            lit.add(x)
        else:
            lit.add(dc.len_sym(x[0])[0])
            dist.add(dc.dist_sym(x[1])[0])
    dl = {0: 1} if d1 else (dc.flat(sorted(dist)) if dist else [0])
    return s.dynamic(list(syms) + [EOB], dc.flat(sorted(lit)), dl, final=final)


# literal/length lengths with a 15-bit code on the all-ones codeword: 255 symbols of 8 bits, a chain of 9 .. 15
LIT15 = {**{s: 8 for s in list(range(7, 255)) + list(range(256, 263))},
         **{1: 9, 2: 10, 3: 11, 4: 12, 5: 13, 6: 14, 0: 15, 255: 15}}


def encode(payload, kind):
    """raw DEFLATE of a block payload with one of the crafted stream kinds (checked against zlib)"""
    s = Deflate()
    if kind == "dyn15":
        s.dynamic(list(payload) + [EOB], LIT15, [0], final=True)
    elif kind == "fixed":
        s.fixed(lz77(payload) + [EOB], final=True)
    elif kind == "stored":
        s.stored(payload, final=True)
    elif kind == "split":
        a, b = len(payload) // 3, 2 * len(payload) // 3
        syms = lz77(payload[:b])
        cut = 0
        for k, x in enumerate(syms):                     # the symbol that reaches byte a
            cut += 1 if isinstance(x, int) else x[0]
            if cut >= a:
                break
        s.fixed(syms[:k + 1] + [EOB])
        _flat_dynamic(s, syms[k + 1:], final=False)
        s.stored(payload[b:], final=True)
    elif kind == "dist1":
        _flat_dynamic(s, lz77(payload, d1_only=True), d1=True)
    return dc.check(s)[0]


KINDS = ["dyn15", "fixed", "stored", "split", "dist1"]


def bam_parts(refs, recs):
    """(header bytes, [record bytes]) of a BAM"""
    from xcltk_b200 import synth
    text = ("@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % r for r in refs)).encode()
    h = bytearray(b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs)))
    for n, l in refs:
        h += struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", l)
    return bytes(h), [synth.pack_record(r) for r in recs]


def htslib_cuts(rb, limit):
    """records per block as bam_write1 flushes: whole records, at most `limit` bytes"""
    cuts, n, size = [], 0, 0
    for r in rb:
        if n and size + len(r) > limit:
            cuts.append(n)
            n, size = 0, 0
        n, size = n + 1, size + len(r)
    return cuts + ([n] if n else [])


def write_bam_blocks(path, header, rb, cuts, kind_of=None, shared=0, empty=(), bad_block=None):
    """a BAM from explicit blocks: the header alone (or with the first `shared` records), then `cuts[i]` records
    per block; `empty`: chunk indexes (0 is the header, len(cuts) + 1 the EOF block) before which an empty BGZF block
    goes; kind_of(i)
    picks block i's stream kind (None: zlib); bad_block: a block index whose stream gets a lone 2-bit distance
    code.  Returns the uncompressed chunks."""
    from xcltk_b200 import synth
    chunks, at = [header + b"".join(rb[:shared])], shared
    for c in cuts:
        chunks.append(b"".join(rb[at:at + c]))
        at += c
    assert at == len(rb)
    with open(path, "wb") as fp:
        for i, ch in enumerate(chunks):
            if i in empty:
                fp.write(synth._bgzf_block(b""))
            if i == bad_block:
                syms = lz77(ch, d1_only=True)
                lits = sorted({x if isinstance(x, int) else dc.len_sym(x[0])[0] for x in syms} | {EOB})
                s = Deflate().dynamic(syms + [EOB], dc.flat(lits), {0: 2}, final=True)
                assert dc.zlib_rejects(s.raw())
                fp.write(dc.member(s.raw(), ch))
            elif kind_of is None or i == 0:
                fp.write(synth._bgzf_block(ch))
            else:
                fp.write(dc.member(encode(ch, kind_of(i)), ch))
        if len(chunks) in empty:
            fp.write(synth._bgzf_block(b""))
        fp.write(synth.BGZF_EOF)
    return chunks


def same_as_host(ctx, p, maps=None, want_seq=True, cell="CB", umi="UB", keyspace=None):
    from xcltk_b200 import lib
    maps = maps or full_maps([p])
    host, ks_h = host_decode([p], maps, cell, umi, want_seq, with_ks=True)
    ks = keyspace if keyspace is not None else lib.KeySpace()
    res = ctx.decode_bams([p], maps, cell, umi, want_seq, ks)
    assert res is not None, ctx.decode_fallback_reason
    assert_same_batch(res[0], res[1], host, ks, ks_h)
    res[0].close()
    return host


@pytest.mark.parametrize("seed", [1, 2])
def test_records_under_every_crafted_stream_kind(gpu_ctx, tmp_path, seed):
    from test_gpu_decode import _random_records
    refs = [("chr1", 10000000), ("chr2", 10000000)]
    header, rb = bam_parts(refs, _random_records(seed, 1200))
    cuts = htslib_cuts(rb, 12000)
    p = str(tmp_path / "k.bam")
    chunks = write_bam_blocks(p, header, rb, cuts, kind_of=lambda i: KINDS[(i + seed) % len(KINDS)])
    assert len(chunks) > 2 * len(KINDS)
    with gzip.open(p, "rb") as fp:
        assert fp.read() == b"".join(chunks)
    host = same_as_host(gpu_ctx, p, want_seq=seed == 1)
    assert host.n > 1000


def test_bam_with_one_rejected_stream_fails_in_both_decoders(gpu_ctx, tmp_path):
    from test_gpu_decode import _random_records
    from xcltk_b200 import lib
    header, rb = bam_parts([("chr1", 10000000), ("chr2", 10000000)], _random_records(4, 1500))
    cuts = htslib_cuts(rb, 12000)
    p = str(tmp_path / "bad.bam")
    write_bam_blocks(p, header, rb, cuts, kind_of=lambda i: KINDS[i % len(KINDS)], bad_block=len(cuts) // 2)
    with pytest.raises(lib.XgError) as ei:
        gpu_ctx.decode_bams([p], full_maps([p]), "CB", "UB", True, lib.KeySpace())
    assert ei.value.code == XG_E_FORMAT
    with pytest.raises(lib.XgError):
        host_decode([p], full_maps([p]), "CB", "UB", True)


# ---- record parse -------------------------------------------------------------------------------------------------

BLOCK_SIZES = [1, 31, 32, 33, 63, 64, 65]
# (block, record of the block) where the contig changes: first records of blocks, links 31 -> 32 and 63 -> 64
CHANGES = [(1, 0), (3, 32), (4, 0), (5, 32), (6, 0), (6, 32), (6, 64)]
DROPPED = {1, 4, 6}              # contigs the caller does not ask for
B_SUBTYPES = "cCsSiIf"


def _cigar(i):
    k = i % 8
    if k == 0:
        return []
    if k == 1:
        return [(0, 20)]                                  # one op, simple: elided
    if k == 2:
        return [(4, 20)]                                  # one op, not simple
    if k == 3:
        return [(0, 1), (1, 1)] * 127                     # 254 ops
    if k == 4:
        return [(0, 1), (1, 1)] * 127 + [(0, 1)]          # 255 ops: the escape
    if k == 5:
        return [(0, 1), (1, 1)] * 128                     # 256 ops
    if k == 6:
        return [(0, 7), (2, 3), (0, 5)]
    return [(3, 200), (0, 9)]


def _tags(i, cb, ub, last_in_block):
    k = i % 11
    if last_in_block:                                     # the CB value is the last byte of the record and block
        return [("UB", "Z", ub), ("CB", "Z", cb)] if i & 1 else [("UB", "Z", ub), ("CB", "A", "A")]
    if k < len(B_SUBTYPES):
        sub = B_SUBTYPES[k]
        vals = [] if i % 3 == 0 else ([0.5 * j for j in range(k + 1)] if sub == "f" else list(range(k + 1)))
        return [("XB", "B", (sub, vals)), ("CB", "Z", cb), ("YB", "B", (sub, [])), ("UB", "Z", ub)]
    if k == 7:
        return [("XH", "H", "0A1B2C"), ("CB", "Z", cb), ("XA", "A", "q"), ("UB", "Z", ub)]
    if k == 8:
        return [("XA", "A", "q"), ("XH", "H", ""), ("UB", "Z", ub), ("CB", "Z", cb)]
    if k == 9:
        return [("CB", "Z", cb), ("UB", "Z", ub)]
    return [("xf", "i", 25), ("CB", "Z", cb)]            # no UB


def parse_records(seed):
    rng = random.Random(seed)
    barcodes = ["".join(rng.choice("ACGT") for _ in range(16)) + "-1" for _ in range(20)]
    recs, tid, pos, i = [], 0, 100, 0
    changes = set(CHANGES)
    for b, n in enumerate(BLOCK_SIZES):
        for j in range(n):
            if (b, j) in changes:
                tid, pos = tid + 1, 100
            pos += rng.randrange(0, 30)
            cig = _cigar(i)
            l_seq = sum(l for op, l in cig if op in (0, 1, 4, 7, 8))
            if i % 5 == 0:
                l_seq = i // 5 % 10                        # 0 .. 9: sequence tails of every length
            seq = "".join(rng.choice("ACGTN") for _ in range(l_seq))
            flag = rng.choice([0, 16, 4, 1024]) if cig else 0
            tags = _tags(i, rng.choice(barcodes), "".join(rng.choice("ACGT") for _ in range(10)), j == n - 1)
            recs.append(("r%d" % i, flag, tid, pos, 30, cig, seq, tags))
            i += 1
    n_ref = tid + 1
    return [("c%d" % t, 1000000) for t in range(n_ref)], recs


@pytest.mark.parametrize("want_seq", [True, False])
def test_record_parse_at_the_32_link_batches(gpu_ctx, tmp_path, want_seq):
    refs, recs = parse_records(5)
    header, rb = bam_parts(refs, recs)
    p = str(tmp_path / "parse.bam")
    write_bam_blocks(p, header, rb, BLOCK_SIZES)
    maps = [np.array([-1 if t in DROPPED else t for t in range(len(refs))], dtype=np.int32)]
    host = same_as_host(gpu_ctx, p, maps, want_seq)
    assert host.n < len(recs) and len(host.runs) == len(refs) - len(DROPPED)
    # the same records with the crafted stream kinds
    write_bam_blocks(p, header, rb, BLOCK_SIZES, kind_of=lambda i: KINDS[i % len(KINDS)])
    same_as_host(gpu_ctx, p, maps, want_seq)


# ---- keys at the 63-bit packing limit -----------------------------------------------------------------------------

@pytest.mark.parametrize("only_packed", [False, True])
@pytest.mark.parametrize("where", ["CB", "UB", "qname"])
def test_keys_at_the_packing_limit(gpu_ctx, tmp_path, where, only_packed):
    """device keys equal the host decoder's and the keyspace's encoding of the same string; a file whose values
    all pack into 63 bits decodes without a keyspace (the device packs every one of them itself)"""
    from xcltk_b200 import lib
    keys = [k for k in limit_keys() if packs(k) or not only_packed]
    recs = []
    for i in range(400):
        s = keys[i % len(keys)]
        other = keys[(i * 7 + 3) % len(keys)]
        name = s if where == "qname" else "q%d" % i
        tags = [("CB", "Z", s), ("UB", "Z", other)] if where == "CB" else [("CB", "Z", other), ("UB", "Z", s)]
        recs.append((name, 0, 0, 100 + i, 30, [(0, 30)], "ACGT" * 7 + "AC", tags))
    p = str(tmp_path / "keys.bam")
    header, rb = bam_parts([("chr1", 100000)], recs)
    write_bam_blocks(p, header, rb, htslib_cuts(rb, 9000))
    ks = lib.KeySpace()
    umi = None if where == "qname" else "UB"
    same_as_host(gpu_ctx, p, want_seq=False, umi=umi, keyspace=ks)
    res = gpu_ctx.decode_bams([p], full_maps([p]), "CB", umi, False, ks)
    got = res[0].download()
    col = 0 if where == "CB" else 1
    for i in range(len(recs)):
        assert int(got.keys[i, col]) == ks.encode(keys[i % len(keys)]), (where, keys[i % len(keys)])
    got.close()
    res[0].close()
    if only_packed:
        res = gpu_ctx.decode_bams([p], full_maps([p]), "CB", umi, False)
        assert res is not None, gpu_ctx.decode_fallback_reason
        assert_same_batch(res[0], res[1], host_decode([p], full_maps([p]), "CB", umi, False))
        res[0].close()


# ---- layout -------------------------------------------------------------------------------------------------------

def layout_records(n=300):
    rng = random.Random(9)
    recs = []
    for i in range(n):
        recs.append(("r%d" % i, 0, i * 3 // n, 100 + 7 * i, 30, [(0, 40)], "ACGT" * 10,
                     [("CB", "Z", rng.choice(["ACGTACGT-1", "TTTTGGGG-1"])), ("UB", "Z", "ACGTAC")]))
    return [("chr1", 100000), ("chr2", 100000), ("chr3", 100000)], recs


def test_header_sharing_its_block_with_records(gpu_ctx, tmp_path):
    refs, recs = layout_records()
    header, rb = bam_parts(refs, recs)
    p = str(tmp_path / "shared.bam")
    for kind_of in (None, lambda i: KINDS[i % len(KINDS)]):
        write_bam_blocks(p, header, rb, [40, 100, 127], kind_of=kind_of, shared=33)
        same_as_host(gpu_ctx, p)


def test_empty_bgzf_blocks_between_blocks(gpu_ctx, tmp_path):
    """ISIZE 0 blocks after the header, between record blocks and before the EOF block"""
    refs, recs = layout_records()
    header, rb = bam_parts(refs, recs)
    p = str(tmp_path / "empty.bam")
    write_bam_blocks(p, header, rb, [100, 100, 100], empty=(1, 2, 3, 4))
    assert sum(1 for _c, u in bai.bgzf_blocks(p) if not u) == 5                # four, and the EOF block
    same_as_host(gpu_ctx, p)
    write_bam_blocks(p, header, rb, [100, 100, 100], empty=(1, 2, 3, 4), kind_of=lambda i: KINDS[i % 5])
    same_as_host(gpu_ctx, p)


def test_index_range_starting_in_the_block_that_ends_the_header(gpu_ctx, tmp_path):
    """walk_start takes the larger of the header's end and the range's skip: a range from the block's start (skip 0,
    inside the header), from its first record (skip = header end) and from a later record"""
    from xcltk_b200 import lib
    refs, recs = layout_records()
    header, rb = bam_parts(refs, recs)
    p = str(tmp_path / "idx.bam")
    write_bam_blocks(p, header, rb, [60, 100, 107], shared=33)
    vb = [r[4] for r in bai.bam_records(p)[1]]
    c0 = vb[0] >> 16
    assert vb[0] & 0xffff == len(header) and vb[5] >> 16 == c0
    size = len(open(p, "rb").read())
    maps = full_maps([p])
    for lo, first in ((c0 << 16, 0), (vb[0], 0), (vb[5], 5)):
        q = str(tmp_path / "exp.bam")
        write_bam_blocks(q, header, rb[first:], [len(rb) - first])
        host = host_decode([q], maps, "CB", "UB", True)
        res = gpu_ctx.decode_bams([p], maps, "CB", "UB", True, lib.KeySpace(), range_lists=[[(lo, size - 28)]])
        if res is None:
            pytest.fail("declined: " + gpu_ctx.decode_fallback_reason)
        assert_same_batch(res[0], res[1], host)
        res[0].close()
