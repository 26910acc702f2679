"""Crafted BGZF members for the device DEFLATE decoder (inflate.cuh), each named after the switch it sits
on.  The same files go through the host harness (a one-lane group, test_inflate_crafted_host.py) and
through the GPU (test_gpu_decode_edges.py).  Every valid member passes zlib's self-check when it is
built; every rejection is a well-formed stream with one invalid field, which zlib refuses."""

import random

import deflate_craft as dc
from deflate_craft import EOB, Deflate


def _rand(n, seed):
    rng = random.Random(seed)
    return bytes(rng.getrandbits(8) for _ in range(n))


def _auto(s, symbols, final=True):
    """a dynamic block whose code is flat over the symbols it uses"""
    lit, dist = {EOB}, set()
    for x in symbols:
        if isinstance(x, int):
            lit.add(x)
        else:
            lit.add(dc.len_sym(x[0])[0])
            dist.add(dc.dist_sym(x[1])[0])
    lit = sorted(lit)
    dist = sorted(dist) or None
    return s.dynamic(symbols, dc.flat(lit), dc.flat(dist) if dist else [0], final=final)


def _exercise(lit_order, dist_order):
    """one occurrence of every literal, every length symbol in a match, every distance symbol, behind
    33 000 bytes of stored data so that every distance reaches"""
    lens = [x for x in lit_order if x > 256]
    n = max(len(lens), len(dist_order))
    syms = [x for x in lit_order if x < 256]
    for i in range(n):
        ls, ds = lens[i % len(lens)], dist_order[i % len(dist_order)]
        ln = dc.LBASE[ls - 257] + ((1 << dc.LEXT[ls - 257]) - 1 if i & 1 else 0)
        d = min(32768, dc.DBASE[ds] + ((1 << dc.DEXT[ds]) - 1 if i & 1 else 0))
        syms.append((min(ln, 257 if ls == 284 else 258), d))
    return syms + [EOB]


def _table(L_lit, L_dist):
    head = [97, 0, 256, 257, 264, 265, 284]
    head += [x for x in range(100, 200)][:L_lit - 1 - len(head)]
    lit_order = head + [255, 285]                    # the two longest; 285 on the all-ones codeword
    dhead = [0, 3, 4, 28, 1, 2, 5, 6, 7, 8, 9, 10, 11, 12, 13][:L_dist - 1]
    dist_order = dhead + [27, 29]
    s = Deflate().stored(_rand(33000, L_lit))
    s.dynamic(_exercise(lit_order, dist_order), dc.skewed(lit_order), dc.skewed(dist_order), final=True)
    assert ("lit", L_lit, True) in s.used and ("dist", L_dist, True) in s.used
    assert not any(a == "lit" and l > L_lit or a == "dist" and l > L_dist for a, l, _ in s.used)
    return [s]


def _fixed(symbols, final=True):
    return Deflate().fixed(symbols, final=final)


def _header_runs():
    """HLIT 262 / HDIST 16, every length 4, spelled with 16 x3 / x6, 17 x3 / x10, 18 x11 / x138 and a 16
    that runs from the literal/length lengths into the distance lengths"""
    lit = [4] * 10 + [0] * 246 + [4] * 6
    dist = [4] * 16
    plan = [4, (16, 3), (16, 6), (17, 3), (17, 10), (18, 11), (18, 138), (18, 84), 4, (16, 6), (16, 6), (16, 6),
            (16, 3)]
    syms = list(range(10)) * 30 + [(3 + k % 5, 1 + (k * 17) % 256) for k in range(40)] + [EOB]
    s = Deflate().dynamic(syms, lit, dist, final=True, cl_plan=plan)
    return [s]


def _bit_positions():
    """a stored block behind a fixed block whose EOB ends at bit 0, 1, ..., 7 of its byte"""
    s = Deflate()
    for p in range(8):
        b = (p - s.w.n - 3 - 8 * 5 - 7) % 8           # 5 eight-bit literals, b nine-bit ones, the 7-bit EOB
        s.fixed([65, 66, 67, 68, 69] + [200] * b + [EOB])
        assert s.end_bits[-1] == p
        s.stored(bytes([48 + p]) * (p + 1), final=p == 7)
    return [s]


def _orders():
    import itertools
    out = []
    for k, order in enumerate(itertools.permutations("sfd")):
        s = Deflate()
        for j, kind in enumerate(order):
            final = j == 2
            if kind == "s":
                s.stored(_rand(100 + k, k), final=final)
            elif kind == "f":
                s.fixed([70 + k, 71, 72, (5, 2), (30, 7), EOB], final=final)
            else:
                _auto(s, [80 + k, 81, (4, 1), (9, 3), EOB], final=final)
        out.append(s)
    return out


def _stored_sizes():
    """stored blocks of 0 and 1 bytes and one that fills the member to 65 536 bytes (the BGZF maximum)"""
    s = Deflate().stored(b"")
    s.stored(b"x")
    s.fixed([66] + [(258, 1)] * 21 + [(100, 1), EOB])
    rest = 65536 - len(s.payload)
    s.stored(_rand(rest, 9), final=True)
    assert len(s.payload) == 65536
    return [s]


def _fill(n, seed):
    """a member of exactly n bytes: literals, then runs of (258, 1)"""
    rng = random.Random(seed)
    k = min(n, 1 + rng.randrange(40))
    syms = [rng.randrange(256) for _ in range(k)]
    left = n - k
    while left:
        if left < 3:
            syms.append(rng.randrange(256))
            left -= 1
            continue
        m = min(258, left)
        if 0 < left - m < 3:
            m -= 3
        syms.append((m, 1 + rng.randrange(min(k, 30))))
        left -= m
    return _fixed(syms + [EOB])


def _batch_cases():
    c = {}
    c["batch_32_literals"] = [_fixed(list(range(40, 72)) + [EOB]), _fixed(list(range(40, 104)) + [EOB])]
    c["batch_eob_after_1"] = [_fixed([65, EOB])]
    c["batch_eob_after_31"] = [_fixed(list(range(50, 81)) + [EOB]), _fixed(list(range(50, 83)) + [EOB])]
    # the batch starts at o = 32; its 5th symbol (offset o + 4) copies 3 bytes from d = 7 back: source [o - 3, o)
    pre = list(range(60, 92))
    c["batch_source_ends_at_o"] = [_fixed(pre + [1, 2, 3, 4, (3, 7), 5, EOB])]
    # ... from d = 6 back: source [o - 2, o + 1), o written by the same 32-byte round
    c["batch_source_ends_at_o_plus_1"] = [_fixed(pre + [1, 2, 3, 4, (3, 6), 5, EOB])]
    c["batch_d1_len258_first"] = [_fixed(pre + [(258, 1), 7, 8, EOB])]
    c["batch_d1_len258_last"] = [_fixed(pre + list(range(31)) + [(258, 1), 9, EOB])]
    c["batch_31_dependent_matches"] = [_fixed([77] + [(3 + k % 4, 1 + k % 3) for k in range(31)] + [78, EOB])]
    c["batch_32x258_independent"] = [Deflate().stored(_rand(32768, 3)).fixed([(258, 32768)] * 32 + [EOB], final=True)]
    c["batch_32x258_dependent"] = [_fixed([5] * 32 + [(258, 1)] * 32 + [EOB])]
    return c


def valid_cases():
    """name -> list of Deflate streams, one BGZF member each"""
    c = {}
    c["table_lit10_dist8"] = _table(10, 8)
    c["table_lit11_dist9"] = _table(11, 9)
    c["table_lit15_dist15"] = _table(15, 15)
    c["lengths_distances_extremes"] = [
        Deflate().stored(_rand(32768, 5)).fixed([(3, 1), (10, 4), (11, 5), (257, 32768), (258, 32768), EOB], final=True),
        _fixed([65, 66, 67, (258, 3), EOB]),                                  # distance = output so far: byte 0
        Deflate().stored(_rand(32768, 6)).fixed([(258, 32768), EOB], final=True)]
    c["lone_distance_code_len1"] = [
        Deflate().dynamic([65, (3, 1), EOB], {65: 2, 256: 2, 257: 1}, {0: 1}, final=True)]
    c["literal_only_hdist1"] = [Deflate().dynamic([65, 66, 65, EOB], dc.flat([65, 66, 256]), [0], final=True)]
    c["eob_only_block_between_data"] = [
        Deflate().stored(b"abc").dynamic([EOB], {256: 1}, [0]).fixed([100, (5, 1), EOB], final=True)]
    c["header_runs_16_17_18_and_boundary"] = _header_runs()
    ends_lit, ends_dist = [0, 255, 256, 257, 264, 265, 284, 285], [0, 3, 4, 28, 29]
    c["header_hlit286_hdist30"] = [Deflate().stored(_rand(33000, 8)).dynamic(
        _exercise(ends_lit, ends_dist), dc.lens_list(dc.flat(ends_lit), 286), dc.lens_list(dc.flat(ends_dist), 30),
        final=True)]
    c["block_orders"] = _orders()
    c["stored_0_1_rest_of_64k"] = _stored_sizes()
    c["stored_after_bit_0_to_7"] = _bit_positions()
    c["coff_mod4"] = [_fixed(list(range(65, 65 + n)) + [EOB]) for n in range(1, 9)]
    c.update(_batch_cases())
    c["isize_1_to_33"] = [_fill(n, n) for n in range(1, 34)]
    c["isize_65535_65536"] = [_fill(65535, 1), _fill(65536, 2)]
    return c


# the error inflate_group returns for each rejection: the check the case is named after
REJECT_RC = {
    "lone_distance_code_len2": -12, "lone_litlen_code_len2_eob_only": -11, "oversubscribed_litlen": -11,
    "oversubscribed_distance": -12, "eob_length_0": -10, "repeat_16_first": -8, "repeat_past_hlit_hdist": -9,
    "hlit_287": -5, "hdist_31": -5, "hclen_4_no_eob": -10, "fixed_litlen_286": -14, "fixed_litlen_287": -14,
    "fixed_distance_30": -15, "fixed_distance_31": -15, "distance_past_start": -16,
}


def reject_cases():
    """name -> one Deflate stream with one invalid field"""
    r = {}
    r["lone_distance_code_len2"] = Deflate().dynamic([65, (3, 1), EOB], {65: 2, 256: 2, 257: 1}, {0: 2}, final=True)
    r["lone_litlen_code_len2_eob_only"] = Deflate().stored(b"ab").dynamic([EOB], {256: 2}, [0]).fixed(
        [100, EOB], final=True)
    r["oversubscribed_litlen"] = Deflate().dynamic([65, EOB], {65: 1, 66: 1, 256: 1}, [0], final=True)
    r["oversubscribed_distance"] = Deflate().dynamic([65, (3, 1), EOB], {65: 2, 256: 2, 257: 1},
                                                     {0: 1, 1: 1, 2: 1}, final=True)
    r["eob_length_0"] = Deflate().dynamic([65, 66], {65: 1, 66: 1}, [0], final=True)
    lit = dc.lens_list(dc.flat([65, 66, 256]), 257)
    r["repeat_16_first"] = Deflate().dynamic([65, EOB], lit, [0], final=True, cl_plan=[(16, 3)] + lit[3:] + [0])
    r["repeat_past_hlit_hdist"] = Deflate().dynamic([65, EOB], lit, [0], final=True,
                                                    cl_plan=lit[:250] + [(17, 10)])
    r["hlit_287"] = Deflate().dynamic([65, EOB], dc.lens_list(dc.flat([65, 66, 256]), 287), [0], final=True)
    r["hdist_31"] = Deflate().dynamic([65, EOB], lit, dc.lens_list({0: 1, 1: 1}, 31), final=True)
    r["hclen_4_no_eob"] = Deflate().dynamic([], [0] * 257, [0], final=True, hclen=4,
                                            cl_plan=[(18, 138), (18, 119), 0], cl_lens=dc.lens_list({18: 1, 0: 1}, 19))
    r["fixed_litlen_286"] = _fixed([65, (286, 0, 0, 0), EOB])
    r["fixed_litlen_287"] = _fixed([65, (287, 0, 0, 0), EOB])
    r["fixed_distance_30"] = _fixed([65, 66, 67, (257, 0, 30, 0), EOB])
    r["fixed_distance_31"] = _fixed([65, 66, 67, (257, 0, 31, 0), EOB])
    r["distance_past_start"] = _fixed([65, 66, (3, 3), EOB])
    return r


def member_of(s, reject=False):
    """(member bytes, payload) of one stream; a valid stream is checked against zlib first"""
    if reject:
        # ISIZE is the size the stream gives taken at face value, so that the invalid field is the only one (the
        # bytes a match would read before the output are unknown: zeros stand for them in the CRC); a member of
        # ISIZE 0 is never inflated, so a stream of no output carries 4 bytes
        raw = s.raw()
        assert dc.zlib_rejects(raw)
        payload = bytes(s.payload) if s.payload is not None else bytes(s.size)
        if not payload:
            payload = b"AAAA"
        return dc.member(raw, payload), payload
    raw, payload = dc.check(s)
    return dc.member(raw, payload), payload
