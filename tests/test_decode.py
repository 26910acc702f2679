"""Host decoder (xcltk_b200/csrc/decode.cpp) against an independent pure-Python BAM reader
(oracle/shim/pysam.py) record by record, plus the htslib semantics of SURVEY.md A.3 on
hand-built records and the losslessness of the 64-bit string keys."""

import os
import random
import struct
import sys

import numpy as np
import pytest
from hypothesis import given, settings
from hypothesis import strategies as st

from util import GOLD, ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle", "shim"))
import pysam as shim  # noqa: E402

from xcltk_b200 import lib, synth  # noqa: E402


def decode(paths, cell_tag="CB", umi_tag="UB", want_seq=True, threads=3):
    ks = lib.KeySpace()
    maps = [np.arange(len(lib.bam_references(p)), dtype=np.int32) for p in paths]
    return lib.decode_bams(paths, maps, cell_tag, umi_tag, want_seq, ks, threads), ks


def check_against_shim(path, hr, ks, base=0, cell_tag="CB", umi_tag="UB"):
    af = shim.AlignmentFile(path)
    i = base
    for tid in range(len(af.references)):
        for r in af._recs.get(tid, []):
            pos, end = hr.pos_end[i]
            assert (pos, end) == (r.pos, r.endpos)
            f = int(hr.fmq[i])
            assert (f & 0xffff, (f >> 16) & 0xff) == (r.flag, r.mapq)
            ncw, cig = f >> 24, r._cigar
            if ncw == 0:
                assert len(cig) == 1 and (cig[0] & 15) in (0, 7, 8) and (cig[0] >> 4) == end - pos
            else:
                off = int(hr.cig_off[i])
                if len(cig) == 0:
                    assert hr.cigar[off] == 6
                else:
                    n = int(hr.cigar[off - 1]) if ncw == 255 else ncw
                    assert n == len(cig) and tuple(hr.cigar[off:off + n]) == tuple(cig)
            ck, uk = (int(x) for x in hr.keys[i])
            if cell_tag:
                exp = r.get_tag(cell_tag) if r.has_tag(cell_tag) else None
                assert ks.decode(ck) == exp if isinstance(exp, (str, type(None))) else ck == lib.XG_KEY_NOMATCH
            if umi_tag:
                if not r.has_tag(umi_tag):
                    assert uk == lib.XG_KEY_NONE
                elif isinstance(r.get_tag(umi_tag), str):
                    assert ks.decode(uk) == r.get_tag(umi_tag)
            else:
                assert ks.decode(uk) == r.query_name
            so, qs = int(hr.seq_off[i]), r.query_sequence
            if qs is None:
                assert so == 0xFFFFFFFF
            else:
                nb = (len(qs) + 1) // 2
                assert hr.seq[so:so + (nb + 3) // 4].tobytes()[:nb] == bytes(r._seq_raw)
            i += 1
    return i


def golden_bams():
    out = []
    for case in sorted(os.listdir(GOLD)):
        d = os.path.join(GOLD, case)
        out += [os.path.join(d, f) for f in sorted(os.listdir(d)) if f.endswith(".bam")]
    return out


@pytest.mark.parametrize("path", golden_bams())
def test_decoder_matches_python_reader(path):
    hr, ks = decode([path])
    n = check_against_shim(path, hr, ks)
    assert n == hr.n == hr.n_records_seen
    # tile index: run-aligned, first_pos / max_end consistent
    for rec_beg, n_rec, run, first_pos, max_end in hr.tiles():
        assert 1 <= n_rec <= lib.XG_TILE
        assert first_pos == hr.pos_end[rec_beg, 0]
        assert max_end == hr.pos_end[rec_beg:rec_beg + n_rec, 1].max()
        assert hr.runs[run][2] <= rec_beg and rec_beg + n_rec <= hr.runs[run][3]
    assert np.all(np.diff(hr.cig_off.astype(np.int64)) >= 0)


def test_multi_bam_order_and_runs():
    d = os.path.join(GOLD, "d3_sample_mode")
    paths = [os.path.join(d, "w1.bam"), os.path.join(d, "w2.bam")]
    hr, ks = decode(paths, cell_tag=None, umi_tag=None)
    assert [r[0] for r in hr.runs] == [0, 1]           # BAM-list order = fetch order (B4)
    n = check_against_shim(paths[0], hr, ks, 0, None, None)
    n = check_against_shim(paths[1], hr, ks, n, None, None)
    assert n == hr.n


def _write(tmp_path, recs, refs=(("chr1", 100000), ("chr2", 50000)), name="t.bam"):
    p = str(tmp_path / name)
    synth.write_bam(p, list(refs), recs)
    return p


def test_htslib_semantics_on_handbuilt_records(tmp_path):
    M, I, D, N, S, H, P, EQ, X = range(9)
    recs = [
        ("unmapped_placed", 4, 0, 10, 0, [(M, 20)], "A" * 20, []),            # FUNMAP: endpos = pos + 1
        ("nocigar", 0, 0, 20, 30, [], "", []),                                # no CIGAR, no SEQ
        ("ops", 0, 0, 30, 30, [(S, 3), (EQ, 5), (X, 2), (I, 4), (D, 6), (N, 100), (M, 7), (H, 9)],
         "ACGTNACGTNACGTNACGTNA", [("CB", "Z", "ACGT-1"), ("UB", "A", "Q"), ("XX", "B", ("S", [1, 2, 3]))]),
        ("many", 0, 0, 40, 30, [(M, 1), (I, 1)] * 150, "AC" * 150, [("UB", "i", 7), ("CB", "i", 5)]),
        ("zeroumi", 0, 1, 5, 30, [(M, 10)], "ACGTACGTAC", [("UB", "C", 0), ("CB", "Z", "")]),
    ]
    p = _write(tmp_path, recs)
    hr, ks = decode([p])
    assert hr.n == 5 and len(hr.runs) == 2
    pe = hr.pos_end
    assert tuple(pe[0]) == (10, 11)
    assert tuple(pe[1]) == (20, 21) and int(hr.seq_off[1]) == 0xFFFFFFFF
    assert tuple(pe[2]) == (30, 30 + 5 + 2 + 6 + 100 + 7)
    assert int(hr.fmq[3]) >> 24 == 255 and int(hr.cigar[int(hr.cig_off[3]) - 1]) == 300
    assert hr.max_aln_len == 150
    assert ks.decode(int(hr.keys[2, 0])) == "ACGT-1" and ks.decode(int(hr.keys[2, 1])) == "Q"
    assert int(hr.keys[3, 0]) == lib.XG_KEY_NOMATCH                      # integer CB never matches
    assert int(hr.keys[3, 1]) not in (lib.XG_KEY_NONE, lib.XG_KEY_EMPTY, lib.XG_KEY_NOMATCH)
    assert int(hr.keys[4, 1]) == lib.XG_KEY_EMPTY and int(hr.keys[4, 0]) == lib.XG_KEY_EMPTY
    check_against_shim(p, hr, ks)


def test_contig_filter_and_counts(tmp_path):
    recs = [("a", 0, 0, 5, 30, [(0, 10)], "A" * 10, []), ("b", 0, 1, 5, 30, [(0, 10)], "A" * 10, []),
            ("u", 4, -1, -1, 0, [], "A" * 10, [])]
    p = _write(tmp_path, recs)
    ks = lib.KeySpace()
    hr = lib.decode_bams([p], [np.array([-1, 3], dtype=np.int32)], "CB", "UB", False, ks, 1)
    assert hr.n == 1 and hr.n_records_seen == 3 and hr.runs == [(0, 3, 0, 1)]
    assert not hr.has_seq


def test_errors(tmp_path):
    recs = [("b", 0, 0, 50, 30, [(0, 10)], "A" * 10, []), ("a", 0, 0, 5, 30, [(0, 10)], "A" * 10, [])]
    p = _write(tmp_path, recs)
    with pytest.raises(lib.XgError) as ei:
        decode([p])
    assert ei.value.code == -3 and "sorted" in str(ei.value)
    bad = str(tmp_path / "x.bam")
    with open(bad, "wb") as fp:
        fp.write(b"not a bam file at all")
    with pytest.raises(lib.XgError):
        decode([bad])
    with pytest.raises(lib.XgError):
        lib.bam_references(str(tmp_path / "missing.bam"))


def test_empty_bam(tmp_path):
    p = _write(tmp_path, [])
    hr, ks = decode([p])
    assert hr.n == 0 and hr.runs == [] and hr.n_tiles == 0
    assert lib.bam_references(p) == [("chr1", 100000), ("chr2", 50000)]


def test_large_random_bam_all_threads(tmp_path):
    rng = random.Random(5)
    feats = [("1", 1000, 90000, "g")]
    bcs = synth.make_barcodes(rng, 20)
    refs, recs = synth.gen_10x_records(11, [("1", 100000)], feats, 6000, bcs, chr_prefix="chr")
    p = str(tmp_path / "r.bam")
    synth.write_bam(p, refs, recs, block=3000, align=False)          # many small BGZF blocks, records straddle them
    for thr in (1, 4):
        hr, ks = decode([p], threads=thr)
        assert check_against_shim(p, hr, ks) == 6000


KEY_ALPHABET = st.text(alphabet="ACGTN-0123456789acgtXYZ_.:", min_size=0, max_size=40)


@settings(max_examples=300, deadline=None)
@given(st.lists(KEY_ALPHABET, min_size=1, max_size=30))
def test_keys_are_lossless(strings):
    ks = lib.KeySpace()
    keys = [ks.encode(s) for s in strings]
    for s, k in zip(strings, keys):
        assert ks.decode(k) == s
        assert k not in (lib.XG_KEY_NONE, lib.XG_KEY_NOMATCH)
        assert (k == lib.XG_KEY_EMPTY) == (s == "")
    for a, ka in zip(strings, keys):
        for b, kb in zip(strings, keys):
            assert (a == b) == (ka == kb)


def test_packed_key_examples():
    ks = lib.KeySpace()
    for s in ("ACGTACGTACGTACGT-1", "N" * 21, "ACGTACGTACGT", "A-9"):
        assert ks.encode(s) >> 63 == 0, s          # packed, no interning needed
    assert ks.n_interned() == 0
    assert ks.encode("A" * 22) >> 63 == 1 and ks.encode("read/1") >> 63 == 1
    assert ks.n_interned() == 2


def limit_keys():
    """values at the 63-bit packing limit (3 bits per base or '-', 7 per digit): 20 / 21 / 22 bases, 17 / 18 bases
    + "-1", 8 / 9 / 10 digits, 14 bases + 3 digits (the last digit takes bits 56 -> 63) and neighbours"""
    b = "ACGTN-ACGTACGTACGTACGTAC"
    return [b[:20], b[:21], b[:22], b[:17] + "-1", b[:18] + "-1", "12345678", "123456789", "1234567890",
            "ACGTACGTACGTAC" + "12" + "3", "ACGTACGTACGTAC" + "1234", "ACGTACGTACGTACGTAC7", "ACGTACGTACGTACGTACG7"]


def packs(s):
    return sum(7 if c.isdigit() else 3 for c in s) <= 63


def test_limit_keys_pack_where_expected(tmp_path):
    """63 bits pack, 64 do not (bit 63 marks an interned key); the host decoder gives a record the key the keyspace
    gives its string, as CB, as UB and as query name"""
    ks = lib.KeySpace()
    assert sum(packs(s) for s in limit_keys()) == 7
    for s in limit_keys():
        assert (ks.encode(s) >> 63 == 0) == packs(s), s
    keys = limit_keys()
    recs = [(keys[i], 0, 0, 100 + i, 30, [(0, 10)], "ACGTACGTAC", [("CB", "Z", keys[i]), ("UB", "Z", keys[-1 - i])])
            for i in range(len(keys))]
    p = _write(tmp_path, recs, refs=(("chr1", 100000),))
    for umi_tag, col_of in (("UB", lambda i: keys[-1 - i]), (None, lambda i: keys[i])):
        hr, ks = decode([p], umi_tag=umi_tag)
        assert hr.n == len(keys)
        for i in range(len(keys)):
            assert int(hr.keys[i, 0]) == ks.encode(keys[i]) and int(hr.keys[i, 1]) == ks.encode(col_of(i)), (i, umi_tag)
        hr.close()


BCH869 = os.path.join(GOLD, "bch869_smartseq", "BCH869.output.bam")     # copied from the reference's merge_smartseq/


def test_real_smartseq_bam_and_committed_arrays():
    """The reference's only real BAM: decoder vs the Python reader, and the committed
    tests/golden/bch869_smartseq/reads.npz is exactly what the decoder produces."""
    hr, ks = decode([BCH869], cell_tag="RG", umi_tag=None, threads=4)
    assert check_against_shim(BCH869, hr, ks, 0, "RG", None) == 32764
    z = np.load(os.path.join(GOLD, "bch869_smartseq", "reads.npz"))
    assert np.array_equal(z["pos_end"], hr.pos_end) and np.array_equal(z["fmq"], hr.fmq)
    assert np.array_equal(z["cigar"], hr.cigar) and np.array_equal(z["seq"], hr.seq)
    names = [ks.decode(int(k)) for k in hr.keys[:, 1]]
    umi_names, umi_idx = z["umi_names"], z["umi_idx"]
    assert [str(x) for x in umi_names[umi_idx]] == names


def test_host_decoder_checks_the_gzip_crc(tmp_path):
    """a block whose trailer CRC32 does not match its inflated bytes is rejected (as htslib does)"""
    import struct
    recs = [("r%d" % i, 0, 0, 10 * i, 30, [(0, 20)], "ACGT" * 5, [("CB", "Z", "ACGT-1"), ("UB", "Z", "ACGTAA")])
            for i in range(200)]
    good = _write(tmp_path, recs, name="good.bam")
    raw = bytearray(open(good, "rb").read())
    # second block = first record block: its size from the BC subfield, CRC at the end - 8
    off = 0
    bsize = struct.unpack_from("<H", raw, off + 16)[0] + 1
    off += bsize
    bsize = struct.unpack_from("<H", raw, off + 16)[0] + 1
    raw[off + bsize - 8] ^= 0x01
    bad = str(tmp_path / "badcrc.bam")
    open(bad, "wb").write(bytes(raw))
    hr, _ = decode([good])
    assert hr.n == 200
    with pytest.raises(lib.XgError) as ei:
        decode([bad])
    assert ei.value.code == -3 and "CRC" in str(ei.value)


def _mutated_bam(tmp_path, name, mutate):
    """A valid BAM whose inflated bytes are edited and compressed again (CRCs right): only the record walk can object."""
    import gzip
    from xcltk_b200.synth import _bgzf_block
    recs = [("r%d" % i, 0, 0, 10 * i, 30, [(0, 15), (3, 40), (0, 5)], "ACGT" * 5,
             [("CB", "Z", "ACGT-1"), ("UB", "Z", "ACGTAA"), ("NH", "i", 1)]) for i in range(50)]
    good = _write(tmp_path, recs, name="src_" + name)
    raw = bytearray(gzip.open(good, "rb").read())
    l_text = struct.unpack_from("<i", raw, 4)[0]
    off = 8 + l_text
    n_ref = struct.unpack_from("<i", raw, off)[0]
    off += 4
    for _ in range(n_ref):
        l_name = struct.unpack_from("<i", raw, off)[0]
        off += 4 + l_name + 4
    mutate(raw, off)                      # off = block_size field of the first record
    out = str(tmp_path / name)
    with open(out, "wb") as fp:
        for k in range(0, len(raw), 40000):
            fp.write(_bgzf_block(bytes(raw[k:k + 40000])))
        fp.write(_bgzf_block(b""))
    return out


@pytest.mark.parametrize("field", ["l_seq", "n_cigar", "l_name", "cigar_len", "tag_cut"])
def test_host_decoder_rejects_records_whose_fields_point_outside(tmp_path, field):
    """ADVICE r1: name / CIGAR / sequence lengths that do not fit the record, a reference span past 2^31 and a tag
    value cut off by the record's end must be refused (or, for the tag, read as absent) -- never read past the buffer."""
    import struct as st

    def mutate(raw, off):
        if field == "l_seq":
            st.pack_into("<I", raw, off + 20, 0x3fffffff)
        elif field == "n_cigar":
            st.pack_into("<H", raw, off + 16, 0xffff)
        elif field == "l_name":
            raw[off + 12] = 255
        elif field == "cigar_len":          # pos + reference length of record 0 passes 2^31
            st.pack_into("<i", raw, off + 8, 2147483640)
        elif field == "tag_cut":            # shrink the record so that its last tag's value is cut off; shift the rest
            bs = st.unpack_from("<I", raw, off)[0]
            del raw[off + 4 + bs - 2: off + 4 + bs]
            st.pack_into("<I", raw, off, bs - 2)
    p = _mutated_bam(tmp_path, field + ".bam", mutate)
    if field == "tag_cut":
        hr, ks = decode([p], cell_tag="NH", umi_tag="UB")
        assert hr.n == 50
        assert int(hr.keys[0, 0]) == lib.XG_KEY_NONE          # the cut tag is absent, the others are read
        assert ks.decode(int(hr.keys[0, 1])) == "ACGTAA"
        hr.close()
        return
    with pytest.raises(lib.XgError) as ei:
        decode([p], want_seq=True)
    assert ei.value.code == -3


@pytest.mark.parametrize("want_seq", [True, False])
def test_bam_writer_round_trip(tmp_path, want_seq):
    """xg_write_bam is the decoders' inverse: records -> BAM -> records gives every array back (10x-style reads
    with spliced / clipped / indel CIGARs, absent and empty tags, and the hand-built CIGAR zoo)."""
    src = os.path.join(GOLD, "c1_chr22_10x", "a.bam")
    refs = lib.bam_references(src)
    hr, ks = decode([src], want_seq=want_seq)
    out = str(tmp_path / "rt.bam")
    lib.write_bam(out, hr, refs, ks, "CB", "UB", level=1, n_threads=3)
    assert lib.bam_references(out) == refs
    h2, ks2 = decode([out], want_seq=want_seq)
    assert h2.n == hr.n and h2.n_records_seen == hr.n
    for name in ("pos_end", "fmq", "cig_off", "cigar"):
        assert np.array_equal(getattr(h2, name), getattr(hr, name)), name
    if want_seq:
        assert np.array_equal(h2.seq_off, hr.seq_off) and np.array_equal(h2.seq, hr.seq)
    assert np.array_equal(h2.keys, hr.keys)            # packed keys: the same strings give the same bits
    assert h2.runs == hr.runs and h2.tiles() == hr.tiles()
    assert (h2.max_aln_len, h2.max_span) == (hr.max_aln_len, hr.max_span)
    # the file is in htslib's block layout: whole records per block
    import gzip
    raw = gzip.open(out, "rb").read()
    assert raw[:4] == b"BAM\x01"
    hr.close()
    h2.close()


def test_block_index_and_probe(tmp_path):
    """What the sharded loader reads off a BAM instead of a .bai: block offsets, the block of the first record,
    and the position of the record that starts a block."""
    import gzip
    src = os.path.join(GOLD, "c1_chr22_10x", "a.bam")
    p = str(tmp_path / "aligned.bam")
    synth.reblock_bam(src, p)
    off, first, aligned = lib.bgzf_block_index(p)
    assert aligned and off[0] == 0 and off[-1] == os.path.getsize(p) and np.all(np.diff(off) > 0)
    raw = open(p, "rb").read()
    for o in off[:-1]:
        assert raw[o:o + 4] == b"\x1f\x8b\x08\x04"
    # the records of the file in order; the first record of every block is the record at the block's inflated offset
    hr, _ = decode([p], want_seq=False)
    pos = hr.pos_end[:, 0]
    seen = 0
    for i in range(first, len(off) - 1):
        blk = gzip.decompress(raw[off[i]:off[i + 1]])
        tid, ps = lib.bam_block_probe(p, int(off[i]))
        if len(blk) == 0:
            assert tid == -2
            continue
        assert (tid, ps) == (struct.unpack_from("<i", blk, 4)[0], struct.unpack_from("<i", blk, 8)[0])
        assert ps == pos[seen]                      # whole records per block: counting records gives the same
        n = 0
        q = 0
        while q < len(blk):
            q += 4 + struct.unpack_from("<I", blk, q)[0]
            n += 1
        assert q == len(blk)
        seen += n
    assert seen == hr.n
    # a BAM cut into blocks without regard to records is reported as such
    _off, _first, al2 = lib.bgzf_block_index(src)
    assert not al2
    hr.close()
