"""Crafted DEFLATE streams (inflate_cases.py: codes zlib never writes, table edges, header encodings,
block sequences, 32-lane batch boundaries, invalid fields) through the device decoder's inflate logic
compiled for the host with a one-lane group (tests/inflate_host_harness.cpp), against zlib.  The
batch model's coverage is asserted here; the GPU run (test_gpu_decode_edges.py) confirms the
32-lane write paths on the same files."""

import os
import subprocess
import zlib

import pytest

import deflate_craft as dc
import inflate_cases as ic
from util import ROOT

from xcltk_b200 import synth

VALID = ic.valid_cases()
REJECT = ic.reject_cases()


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("inflate") / "harness")
    src = os.path.join(ROOT, "tests", "inflate_host_harness.cpp")
    subprocess.check_call(["g++", "-O1", "-o", exe, src, "-lz"])
    return exe


def run(exe, members, tmp_path):
    p = str(tmp_path / "crafted.bgzf")
    with open(p, "wb") as fp:
        fp.write(b"".join(members) + synth.BGZF_EOF)
    out = subprocess.run([exe, p, "-r"], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    rcs = [int(x.split("rc ")[1]) for x in out if " rc " in x]
    n_blocks, n_bad = (int(x) for x in out[-1].replace(" blocks,", "").replace(" bad", "").split())
    return rcs, n_blocks, n_bad, "\n".join(out)


def test_writer_agrees_with_zlib_on_the_two_lone_distance_codes():
    """the stream of the divergence: lone distance code of length 1 is legal (AAAA), of length 2 not"""
    good = dc.Deflate().dynamic([65, (3, 1), dc.EOB], {65: 2, 256: 2, 257: 1}, {0: 1}, final=True)
    assert zlib.decompress(good.raw(), -15) == b"AAAA" == bytes(good.payload)
    bad = dc.Deflate().dynamic([65, (3, 1), dc.EOB], {65: 2, 256: 2, 257: 1}, {0: 2}, final=True)
    with pytest.raises(zlib.error, match="invalid distances set"):
        zlib.decompress(bad.raw(), -15)


@pytest.mark.parametrize("name", sorted(VALID))
def test_crafted_valid_stream_inflates_like_zlib(harness, tmp_path, name):
    members, payloads = zip(*(ic.member_of(s) for s in VALID[name]))
    rcs, n_blocks, n_bad, out = run(harness, members, tmp_path)
    assert n_blocks == len(members) + 1 and n_bad == 0, out
    assert rcs == [len(p) for p in payloads] + [0], out


@pytest.mark.parametrize("name", sorted(REJECT))
def test_crafted_invalid_stream_is_refused(harness, tmp_path, name):
    """refused by the check the case is named after (its own error code), with ISIZE the size of the stream's
    output taken at face value, so that no other check can refuse it"""
    member, payload = ic.member_of(REJECT[name], reject=True)
    if REJECT[name].size:
        assert len(payload) == REJECT[name].size
    rcs, n_blocks, n_bad, out = run(harness, [member], tmp_path)
    assert n_blocks == 2 and rcs[0] == ic.REJECT_RC[name], out


def test_all_valid_cases_in_one_file(harness, tmp_path):
    members = [ic.member_of(s)[0] for name in sorted(VALID) for s in VALID[name]]
    rcs, n_blocks, n_bad, out = run(harness, members, tmp_path)
    assert n_blocks == len(members) + 1 and n_bad == 0, out


# ---- what the cases reach (the batch model of inflate_group<32> and the codes the writer emitted) ----

def _matches(name):
    out = []
    for s in VALID[name]:
        out += dc.batches(s)[0]
    return out


def _sizes(name):
    out = []
    for s in VALID[name]:
        out += [n for _, _, n in dc.batches(s)[1]]
    return out


def test_model_batch_sizes():
    assert 32 in _sizes("batch_32_literals")
    assert _sizes("batch_32_literals")[:2] == [32, 0]                   # EOB right after 32 symbols: a batch of its own
    assert _sizes("batch_eob_after_1") == [1]
    assert 31 in _sizes("batch_eob_after_31") and 1 in _sizes("batch_eob_after_31")


def test_model_dependence_switch():
    m = [x for x in _matches("batch_source_ends_at_o") if x["dist"] == 7]
    assert len(m) == 1 and m[0]["off"] > m[0]["o"] and m[0]["off"] - 7 + 3 == m[0]["o"] and not m[0]["dep"]
    m = [x for x in _matches("batch_source_ends_at_o_plus_1") if x["dist"] == 6]
    assert len(m) == 1 and m[0]["off"] - 6 + 3 == m[0]["o"] + 1 and m[0]["dep"] and m[0]["same_round"]


def test_model_d1_len258_first_and_last():
    m = [x for x in _matches("batch_d1_len258_first") if (x["len"], x["dist"]) == (258, 1)]
    assert len(m) == 1 and m[0]["first"] and m[0]["o"] > 0 and not m[0]["dep"]
    m = [x for x in _matches("batch_d1_len258_last") if (x["len"], x["dist"]) == (258, 1)]
    assert len(m) == 1 and m[0]["last"] and m[0]["n"] == 32 and m[0]["dep"]


def test_model_dependent_run_and_full_batches_of_258():
    m = _matches("batch_31_dependent_matches")
    assert sum(x["dep"] for x in m if x["batch"] == 0) == 31
    for name, dep in (("batch_32x258_independent", 0), ("batch_32x258_dependent", 31)):
        m = [x for x in _matches(name) if x["len"] == 258 and x["n"] == 32]
        assert len(m) == 32 and sum(x["dep"] for x in m) == dep
        assert sum(x["len"] for x in m) == 8256                          # 258 rounds of 32 bytes


def test_model_codes_at_the_table_edges():
    for name, L_lit, L_dist in (("table_lit10_dist8", 10, 8), ("table_lit11_dist9", 11, 9),
                                ("table_lit15_dist15", 15, 15)):
        used = VALID[name][0].used
        assert ("lit", L_lit, True) in used and ("dist", L_dist, True) in used, name
        assert max(l for a, l, _ in used if a == "lit") == L_lit
        assert max(l for a, l, _ in used if a == "dist") == L_dist


def test_model_alphabet_ends_and_length_distance_extremes():
    for name in ("table_lit10_dist8", "header_hlit286_hdist30"):
        blk = VALID[name][0].blocks[-1]
        lits = {x for x in blk[2] if isinstance(x, int)}
        mt = [x for x in blk[2] if not isinstance(x, int)]
        lsyms = {dc.len_sym(n)[0] for n, _ in mt}
        dsyms = {dc.dist_sym(d)[0] for _, d in mt}
        assert {0, 255, 256} <= lits and {257, 264, 265, 284, 285} <= lsyms and {0, 3, 4, 28, 29} <= dsyms, name
    mt = _matches("lengths_distances_extremes")
    assert {3, 10, 11, 257, 258} <= {x["len"] for x in mt} and {1, 4, 5, 32768} <= {x["dist"] for x in mt}
    assert any(x["dist"] == x["off"] for x in mt)                        # reads byte 0


def test_case_layouts():
    s = VALID["stored_after_bit_0_to_7"][0]
    assert sorted(s.end_bits) == list(range(8))
    stored = [len(b[2]) for b in VALID["stored_0_1_rest_of_64k"][0].blocks if b[0] == "stored"]
    assert stored[:2] == [0, 1] and len(VALID["stored_0_1_rest_of_64k"][0].payload) == 65536
    kinds = [tuple(b[0][0] for b in s.blocks) for s in VALID["block_orders"]]
    assert len(set(kinds)) == 6
    # member payload offsets mod 4 (BitReader::init), output offsets mod 16 (crc32_warp's head and body)
    coff, co = set(), 0
    for s in VALID["coff_mod4"]:
        coff.add((co + 18) % 4)
        co += len(ic.member_of(s)[0])
    assert coff == {0, 1, 2, 3}
    uoff, u = set(), 0
    for s in VALID["isize_1_to_33"]:
        uoff.add(u % 16)
        u += len(s.payload)
    assert uoff == set(range(16))
    assert [len(s.payload) for s in VALID["isize_1_to_33"]] == list(range(1, 34))
    assert [len(s.payload) for s in VALID["isize_65535_65536"]] == [65535, 65536]
