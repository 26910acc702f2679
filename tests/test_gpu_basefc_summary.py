"""basefc's read-assignment summary (`--summary`, xg_basefc_summary) on the GPU against the CPU oracle
(tests/summary_oracle.c): the golden runs through fc_wrapper -- whose other outputs must stay the reference's bytes --
the edges of the contract one fate at a time, a synthetic library of millions of reads, and the same table with and
without a .bai, from either decoder, split over emulated GPUs and on repeated calls."""

import logging
import os

import numpy as np
import pytest

import oracle_backend
import summary_oracle
from recsets import D, M, N, build, cell_keys, umi_keys
from util import GOLD, RDR_FILES, golden_runs, read, resolve
from xcltk_b200 import engine, lib
from xcltk_b200.lib import XG_KEY_EMPTY, XG_KEY_NONE

pytestmark = pytest.mark.gpu
logging.disable(logging.CRITICAL)
FATES = summary_oracle.FATES


class Conf(object):
    min_mapq, min_len, min_include = 20, 10, 1
    incl_flag, excl_flag, no_orphan = 0, 772, True
    barcodes, umi = True, True

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return self.barcodes

    def use_umi(self):
        return self.umi


def read_summary(path):
    """(cell names, (n, 7) table) of a summary.tsv, checking its header and totals."""
    lines = open(path).read().split("\n")
    assert lines[0] == "\t".join(("cell", "total") + FATES) and lines[-1] == ""
    rows = [ln.split("\t") for ln in lines[1:-1]]
    t = np.array([[int(x) for x in r[2:]] for r in rows], dtype=np.int64).reshape(-1, 7)
    assert [int(r[1]) for r in rows] == t.sum(axis=1).tolist()
    return [r[0] for r in rows], t


def spy_count_features(monkeypatch):
    from xcltk_b200.rdr.fc import main as rdr_main
    seen = []
    real = rdr_main.count_features
    monkeypatch.setattr(rdr_main, "count_features", lambda conf, batch=None: seen.append(conf) or real(conf, batch))
    return seen


def oracle_table(conf):
    """The oracle's table for a run's configuration (as prepare_config left it)."""
    chroms = list(dict.fromkeys(r.chrom for r in conf.reg_list))
    host, ks, gid_of = oracle_backend.decode_host(conf.sam_fn_list, chroms, conf.cell_tag, conf.umi_tag, False)
    gid, beg, end = oracle_backend.feature_arrays(conf.reg_list, gid_of)
    keys = np.array([ks.encode(b) for b in conf.barcodes], dtype=np.uint64) if conf.use_barcodes() else None
    t = summary_oracle.summary(host, gid, beg, end, keys, len(conf.samples), summary_oracle.params(conf))
    host.close()
    return t


def use_npz_reads(monkeypatch, r):
    """The case whose BAM cannot travel feeds its decoded records to the same upload path (test_golden_gpu)."""
    if not r["reads_npz"]:
        return
    from npz_reads import load_npz_reads

    def load_reads(sam_fn_list, chroms, cell_tag, umi_tag, want_seq, n_threads=0, device=0, mapped=False,
                   host_only=False):
        ctx = engine.get_context(device)
        host, ks, gid_of = load_npz_reads(sam_fn_list[0], list(chroms))
        stats = {"n_reads": host.n, "n_records_seen": host.n, "max_aln_len": host.max_aln_len,
                 "max_span": host.max_span, "bytes": host.nbytes()}
        return engine.ReadBatch(ctx, ctx.upload(host), ks, gid_of, stats)
    monkeypatch.setattr(engine, "load_reads", load_reads)


# ---------------------------------------------------------------------------------------------------------- goldens
GOLDEN = [(c, r) for c, r in golden_runs("basefc") if c in ("d1_basefc_mini", "c1_chr22_10x", "bch869_smartseq")]


@pytest.mark.parametrize("case,run", GOLDEN)
def test_golden_summary_equals_oracle_and_outputs_keep_their_bytes(case, run, tmp_path, gpu_ctx, monkeypatch):
    from xcltk_b200.rdr.fc.main import fc_wrapper
    r = resolve(case, run)
    use_npz_reads(monkeypatch, r)
    seen = spy_count_features(monkeypatch)
    out = str(tmp_path / "out")
    ret = fc_wrapper(",".join(r["sam"]), r["barcodes"], r["features"], out, summary=True, **r["kwargs"])
    assert ret == int(read(r["expected"] + "/RETCODE")) == 0
    for f in RDR_FILES:
        assert read(os.path.join(r["expected"], f)) == read(os.path.join(out, f)), f
    assert sorted(os.listdir(out)) == sorted(RDR_FILES + ["summary.tsv"])
    names, got = read_summary(os.path.join(out, "summary.tsv"))
    assert names == open(os.path.join(out, "barcodes.tsv")).read().split("\n")[:-1] + ["__no_cell"]
    want = oracle_table(seen[0])
    assert got.tolist() == want.tolist()
    assert got.sum() > 0
    if not seen[0].use_barcodes():
        assert got[-1].sum() == 0


# ---------------------------------------------------------------------------------------------------------- edges
A, B, U = cell_keys(3)
CELLS = np.array([A, B], dtype=np.uint64)


def device_table(ctx, reads, feats, conf, n_cols=2, own=None):
    params = engine.make_params(conf, reads.max_aln_len, with_include=True)
    d = ctx.upload(reads)
    try:
        return ctx.basefc_summary(d, *feats, CELLS if conf.barcodes else None, n_cols, params, own)
    finally:
        d.close()


def check(ctx, reads, feats, conf, want, n_cols=2, own=None):
    """Device table == oracle table == `want` ({(row, fate name): count}, everything else 0)."""
    got = device_table(ctx, reads, feats, conf, n_cols, own)
    orc = summary_oracle.summary(reads, *feats, CELLS if conf.barcodes else None, n_cols,
                                 summary_oracle.params(conf), own=own)
    exp = np.zeros((n_cols + 1, 7), dtype=np.int64)
    for (row, fate), v in want.items():
        exp[row, FATES.index(fate)] = v
    assert orc.tolist() == exp.tolist()
    assert got.tolist() == exp.tolist()


def feats(*iv):
    return tuple(np.array(x, dtype=np.int32) for x in zip(*iv))


def batch(recs, runs=None):
    """recs: (pos, end or CIGAR, cell, umi, flag, mapq)."""
    uk = umi_keys(len(recs))
    ops = [r[1] if isinstance(r[1], list) else None for r in recs]
    end = [r[1] if isinstance(r[1], int) else 0 for r in recs]
    umi = [int(uk[k]) if r[3] is None else r[3] for k, r in enumerate(recs)]
    return build([r[0] for r in recs], [r[2] for r in recs], np.array(umi, dtype=np.uint64),
                 runs or [(0, 0, 0, len(recs))], end=end, ops=ops, flag=[r[4] for r in recs],
                 mapq=[r[5] for r in recs])


def test_record_ending_at_feature_beg_is_out_of_range(gpu_ctx):
    f = feats((0, 100, 200))
    check(gpu_ctx, batch([(50, 100, A, None, 0, 60), (200, 260, A, None, 0, 60)]), f, Conf(), {})
    check(gpu_ctx, batch([(50, 101, A, None, 0, 60)]), f, Conf(), {(0, "one_feature"): 1})


def test_overlap_through_n_gap_or_deletion_only_is_not_included(gpu_ctx):
    f = feats((0, 100, 110))
    recs = [(90, [(M, 10), (N, 30), (M, 10)], A, None, 0, 60), (95, [(M, 5), (D, 20), (M, 10)], B, None, 0, 60)]
    check(gpu_ctx, batch(recs), f, Conf(), {(0, "not_included"): 1, (1, "not_included"): 1})


def test_nested_and_duplicated_features_are_multi_feature(gpu_ctx):
    f = feats((0, 100, 300), (0, 150, 200), (0, 150, 200))
    recs = [(110, 140, A, None, 0, 60), (160, 190, A, None, 0, 60), (170, 230, B, None, 0, 60)]
    check(gpu_ctx, batch(recs), f, Conf(min_include=0.9),
          {(0, "one_feature"): 1, (0, "multi_feature"): 1, (1, "one_feature"): 1})


def test_feature_on_a_contig_the_bam_lacks_counts_nothing(gpu_ctx):
    f = feats((1, 100, 200), (7, 0, 1000), (-1, 0, 0), (0, 1000, 1100))
    check(gpu_ctx, batch([(120, 180, A, None, 0, 60), (1050, 1080, B, None, 0, 60)]), f, Conf(),
          {(1, "one_feature"): 1})


def test_missing_and_empty_umi_are_no_umi(gpu_ctx):
    f = feats((0, 100, 200))
    recs = [(120, 150, A, XG_KEY_NONE, 0, 60), (120, 150, A, XG_KEY_EMPTY, 0, 60)]
    check(gpu_ctx, batch(recs), f, Conf(), {(0, "no_umi"): 2})
    check(gpu_ctx, batch(recs), f, Conf(umi=False), {(0, "one_feature"): 2})


def test_unlisted_barcode_with_low_mapq_is_no_cell_mapq(gpu_ctx):
    f = feats((0, 100, 200))
    recs = [(120, 150, U, None, 0, 5), (121, 150, XG_KEY_NONE, None, 1024, 60), (122, 150, A, None, 4, 60)]
    check(gpu_ctx, batch(recs), f, Conf(), {(2, "mapq"): 1, (2, "one_feature"): 1, (0, "flag"): 1})
    check(gpu_ctx, batch(recs), f, Conf(incl_flag=16), {(2, "mapq"): 1, (2, "flag"): 1, (0, "flag"): 1})


def test_min_len_and_include_on_both_sides_of_their_thresholds(gpu_ctx):
    f = feats((0, 100, 200))
    short = [(150, 159, A, None, 0, 60), (150, 160, B, None, 0, 60)]            # 9 / 10 aligned bases
    check(gpu_ctx, batch(short), f, Conf(), {(0, "short"): 1, (1, "one_feature"): 1})
    frac = [(180, 220, A, None, 0, 60), (181, 221, B, None, 0, 60)]             # 20 / 40 and 19 / 40 inside
    check(gpu_ctx, batch(frac), f, Conf(min_include=0.5), {(0, "one_feature"): 1, (1, "not_included"): 1})
    check(gpu_ctx, batch(frac), f, Conf(min_include=20), {(0, "one_feature"): 1, (1, "not_included"): 1})


def test_contigs_without_features_and_sample_mode(gpu_ctx):
    f = feats((1, 100, 200))
    recs = [(120, 150, A, None, 0, 60), (130, 150, A, None, 0, 60), (120, 150, B, None, 0, 60)]
    runs = [(0, 0, 0, 2), (1, 1, 2, 3)]                                         # BAM 0 on contig 0, BAM 1 on 1
    check(gpu_ctx, batch(recs, runs), f, Conf(barcodes=False), {(1, "one_feature"): 1})


def test_records_over_several_tiles(gpu_ctx):
    rng = np.random.default_rng(3)
    n = 5 * lib.XG_TILE + 17
    pos = np.sort(rng.integers(0, 200000, n))
    end = pos + rng.integers(5, 120, n)
    cells = np.array([A, B, U, XG_KEY_NONE], dtype=np.uint64)[rng.integers(0, 4, n)]
    umi = umi_keys(n)
    umi[rng.random(n) < 0.05] = XG_KEY_NONE
    reads = build(pos, cells, umi, [(0, 0, 0, n)], end=end, flag=rng.choice([0, 4, 1, 3, 16], n),
                  mapq=rng.integers(0, 60, n))
    beg = np.sort(rng.integers(0, 200000, 300))
    f = (np.zeros(300, np.int32), beg.astype(np.int32), (beg + rng.integers(1, 3000, 300)).astype(np.int32))
    for conf in (Conf(), Conf(min_include=0.6, no_orphan=False), Conf(barcodes=False, umi=False, min_len=30)):
        n_cols = 2 if conf.barcodes else 1
        got = device_table(gpu_ctx, reads, f, conf, n_cols)
        want = summary_oracle.summary(reads, *f, CELLS if conf.barcodes else None, n_cols, summary_oracle.params(conf))
        assert got.tolist() == want.tolist()
        assert got[:, 5:].sum() > 0 and got[:n_cols, :4].sum() > 0
    own = (0, int(pos[n // 3]), 0, int(pos[2 * n // 3]))
    part = device_table(gpu_ctx, reads, f, Conf(), 2, own)
    assert part.tolist() == summary_oracle.summary(reads, *f, CELLS, 2, summary_oracle.params(Conf()), own=own).tolist()


# ---------------------------------------------------------------------------------------------------------- scale
def test_synthetic_library_against_oracle(gpu_ctx):
    """2.5M synthetic 10x reads on chr21 / chr22, 4 000 genes and seeded nested intervals, 5 000 cells."""
    from xcltk_b200 import workload
    w = workload.make_basefc_workload(gpu_ctx, 2500000, 5000, n_features=4000, seed=21, chroms={"21", "22"})
    host = w.dreads.download()
    try:
        for conf in (Conf(min_len=30, min_include=0.9), Conf(min_mapq=0, min_len=1, min_include=30, no_orphan=False)):
            params = engine.make_params(conf, host.max_aln_len, with_include=True)
            got = gpu_ctx.basefc_summary(w.dreads, w.gid, w.beg, w.end, w.cell_keys, 5000, params)
            want = summary_oracle.summary(host, w.gid, w.beg, w.end, w.cell_keys, 5000, summary_oracle.params(conf))
            assert got.tolist() == want.tolist()
            assert got[:, 6].sum() > 0 and got[-1].sum() > 0 and got.sum() > 1000000
    finally:
        host.close()
        w.dreads.close()


# ---------------------------------------------------------------------------------------------------------- invariance
@pytest.mark.parametrize("mode", ["device", "device_bai", "host", "host_bai", "shards2", "shards3", "twice"])
def test_summary_is_the_same_however_the_library_is_read(mode, tmp_path, gpu_ctx, monkeypatch):
    """c1_chr22_10x in htslib's block layout: with and without a .bai, from the device or the host decoder, split
    over 2 or 3 emulated GPUs, and on two consecutive calls -- one table, the oracle's."""
    import bai
    from xcltk_b200 import synth
    from xcltk_b200.rdr.fc.main import fc_wrapper
    r = resolve("c1_chr22_10x", "rdr_defaults")
    bam = str(tmp_path / "a.bam")
    synth.reblock_bam(r["sam"][0], bam)
    if mode.endswith("_bai"):
        bai.index_bam(bam)
    if mode.startswith("host"):
        monkeypatch.setenv("XCLTK_B200_DEVICE_DECODE", "0")
    sharded = []
    if mode.startswith("shards"):
        monkeypatch.setenv("XCLTK_B200_GPUS", mode[-1])
        monkeypatch.setenv("XCLTK_B200_EMULATE_SHARDS", "1")
        real = engine.load_reads_sharded
        monkeypatch.setattr(engine, "load_reads_sharded", lambda *a, **kw: sharded.append(real(*a, **kw)) or sharded[-1])
    seen = spy_count_features(monkeypatch)
    outs = [str(tmp_path / ("out%d" % k)) for k in range(2 if mode == "twice" else 1)]
    for out in outs:
        assert fc_wrapper(bam, r["barcodes"], r["features"], out, summary=True, **r["kwargs"]) == 0
        for f in RDR_FILES:
            assert read(os.path.join(r["expected"], f)) == read(os.path.join(out, f)), f
    if mode.startswith("shards"):
        assert sharded and sharded[0] is not None and len(sharded[0].stats["cuts"]) == int(mode[-1]) + 1
    tables = [read_summary(os.path.join(o, "summary.tsv"))[1] for o in outs]
    want = oracle_table(seen[0])
    for t in tables:
        assert t.tolist() == want.tolist()


def test_shard_cut_inside_a_run_of_equal_starts(tmp_path, gpu_ctx, monkeypatch):
    """A library split in two where the cut falls inside a run of 30 000 records that all start at one position and
    fill many BGZF blocks, and the second shard's only feature lies on the next contig (no halo reaches back to the
    cut): records with the cut's own key also end the block before the one the cut was read from, and the second
    shard must decode them.  The sharded table equals the unsharded one and the oracle's."""
    from xcltk_b200.rdr.fc.main import fc_wrapper
    ks = lib.KeySpace()
    rng = np.random.default_rng(11)

    def word(v, n):
        return "".join("ACGT"[(int(v) >> (2 * k)) & 3] for k in range(n))
    bcs = [word(c, 16) + "-1" for c in range(1, 41)]
    P, n_lead, n_run, n_tail = 1000000, 2000, 30000, 2000
    pos = np.concatenate([np.sort(rng.integers(10000, P - 1000, n_lead)), np.full(n_run, P),
                          np.sort(rng.integers(500000, 600000, n_tail))])
    n, n0 = len(pos), n_lead + n_run
    cell = np.array([ks.encode(bcs[c]) for c in rng.integers(0, 40, n)], dtype=np.uint64)
    umi = np.array([ks.encode(word(i, 12)) for i in range(n)], dtype=np.uint64)
    reads = build(pos, cell, umi, [(0, 0, 0, n0), (0, 1, n0, n)], ops=[(M, 60)], mapq=rng.integers(0, 61, n))
    bam = str(tmp_path / "run.bam")
    lib.write_bam(bam, reads, [("chr1", 2000000), ("chr2", 2000000)], ks, "CB", "UB", level=1, n_threads=4)
    bc, ft = str(tmp_path / "bc.tsv"), str(tmp_path / "ft.tsv")
    open(bc, "w").write("".join(b + "\n" for b in bcs[:30]))
    open(ft, "w").write("chr1\t20001\t300000\tlead\nchr1\t%d\t%d\tat_run\nchr2\t550001\t560000\ttail\n" % (P - 9, P + 100))
    one = str(tmp_path / "one")
    seen = spy_count_features(monkeypatch)
    assert fc_wrapper(bam, bc, ft, one, summary=True) == 0
    monkeypatch.setenv("XCLTK_B200_GPUS", "2")
    monkeypatch.setenv("XCLTK_B200_EMULATE_SHARDS", "1")
    sharded = []
    real = engine.load_reads_sharded
    monkeypatch.setattr(engine, "load_reads_sharded", lambda *a, **kw: sharded.append(real(*a, **kw)) or sharded[-1])
    two = str(tmp_path / "two")
    assert fc_wrapper(bam, bc, ft, two, summary=True) == 0
    st = sharded[0].stats
    assert st["cuts"][1] == (0, P) and [len(s) for s in sharded[0].shards] == [2, 1]
    off, _first, _aligned = lib.bgzf_block_index(bam)
    k = int(np.searchsorted(off, st["byte_ranges"][1][0][0]))
    # shard 1 starts before the run; the run fills several blocks before the cut's one (the old start, the last block
    # that began at or before the cut, would have dropped all but the run's last block)
    assert lib.bam_block_probe(bam, int(off[k]))[1] < P
    assert lib.bam_block_probe(bam, int(off[k + 1])) == lib.bam_block_probe(bam, int(off[k + 2])) == (0, P)
    for f in RDR_FILES + ["summary.tsv"]:
        assert read(os.path.join(one, f)) == read(os.path.join(two, f)), f
    t = read_summary(os.path.join(two, "summary.tsv"))[1]
    assert t.tolist() == oracle_table(seen[0]).tolist() and t.sum() > n_run
