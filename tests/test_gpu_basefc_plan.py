"""The epoch plan of basefc, computed on the device (k_plan_*): every switch of its rules against the CPU oracle,
entry by entry -- features that live one, two or three and more epochs (rotating arenas vs the long region, arena
reuse after e - 2), features without candidates, contigs and runs without features, features spanning many runs
(sample mode), all / some / none of the segments big, every feature a set (the zero lists), the streaming call, and
calls back to back on different feature sets and batches (the plan's summary resizes the pool)."""

import numpy as np
import pytest

from recsets import build, cell_keys, umi_keys
from xcltk_b200 import engine

pytestmark = pytest.mark.gpu

N_CELLS = 40


class Conf(object):
    min_mapq, min_len, min_include = 20, 30, 0.5
    incl_flag, excl_flag, no_orphan = 0, 772, False

    def __init__(self, barcodes=True):
        self.barcodes = barcodes

    def use_barcodes(self):
        return self.barcodes

    def use_umi(self):
        return True


def make_case(seed, n_runs, reads_per_run, span, n_feats, barcodes=True):
    """n_runs runs of reads on contig 0, each over [0, span), and one run on contig 1, which has no features; features
    on contig 0 of widths from 500 b to span / 4, some past the last read (no candidates), and a few on contig 2,
    which has no reads.  Run k is BAM k (sample mode: column k); the contig-1 run belongs to BAM 0."""
    rng = np.random.RandomState(seed)
    ck = cell_keys(N_CELLS, salt=seed)
    umis = umi_keys(4 * N_CELLS, salt=seed)             # a small pool: many (cell, UMI) duplicates
    pos, cell, umi, runs = [], [], [], []
    n = 0
    specs = [(0, 0, reads_per_run), (0, 1, reads_per_run // 4)] + [(b, 0, reads_per_run) for b in range(1, n_runs)]
    for bam, g, k in specs:
        p = np.sort(rng.randint(0, span, k))
        pos.append(p)
        cell.append(rng.randint(0, N_CELLS, k))
        umi.append(umis[rng.randint(0, len(umis), k)])
        runs.append((bam, g, n, n + k))
        n += k
    pos = np.concatenate(pos)
    mapq = np.where(rng.rand(n) < 0.05, 0, 60).astype(np.uint32)      # candidates that never count
    reads = build(pos, ck[np.concatenate(cell)], np.concatenate(umi), runs, end=pos + 60, mapq=mapq)
    beg = rng.randint(0, span, n_feats)
    width = np.exp(rng.uniform(np.log(500), np.log(span / 4), n_feats)).astype(np.int64)
    gid = np.zeros(n_feats, np.int32)
    n_empty = n_feats // 10
    beg[:n_empty] = span + 1000 + 5000 * np.arange(n_empty)          # past every read of the contig
    gid[n_empty:n_empty + 3] = 2
    perm = rng.permutation(n_feats)                                   # features in no particular order
    beg, width, gid = beg[perm], width[perm], gid[perm]
    n_cols = N_CELLS if barcodes else n_runs
    return reads, gid, beg.astype(np.int32), (beg + width).astype(np.int32), (ck if barcodes else None), n_cols


@pytest.fixture(scope="module")
def case():
    return make_case(1, 1, 90000, 3000000, 300)


@pytest.fixture(scope="module")
def sample_case():
    return make_case(2, 24, 3000, 2000000, 150, barcodes=False)


def check(ctx, c, monkeypatch, env, host=False, barcodes=True):
    """basefc of case c under the environment env == oracle.basefc; returns the call's timing()."""
    from oracle import oracle
    reads, gid, beg, end, ck, n_cols = c
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    conf = Conf(barcodes)
    p = engine.make_params(conf, reads.max_aln_len, True)
    d = ctx.upload(reads)
    try:
        if host:
            h = d.download()
            try:
                got = [np.asarray(x) for x in ctx.basefc_host(h, gid, beg, end, ck, n_cols, p)[:3]]
            finally:
                h.close()
        else:
            got = [np.asarray(x) for x in ctx.basefc(d, gid, beg, end, ck, n_cols, p)[:3]]
        t = ctx.timing()
    finally:
        d.close()
    exp = oracle.basefc(reads, gid, beg, end, ck, n_cols, oracle.params(conf), 8)
    assert len(exp[2]) > 500
    for a, b in zip(got, exp):
        assert np.array_equal(a, b), env
    for k in env:
        monkeypatch.delenv(k)
    return t


@pytest.mark.parametrize("tiles", ["1", "2", "3", "97"])
def test_feature_lifetimes_across_epochs(gpu_ctx, case, monkeypatch, tiles):
    t = check(gpu_ctx, case, monkeypatch, {"XG_EPOCH_TILES": tiles})
    assert t[5] >= 100 // int(tiles) and t[6] > 0 and t[7] > 0


@pytest.mark.parametrize("tiles", ["1", "3"])
def test_sample_mode_features_span_runs(gpu_ctx, sample_case, monkeypatch, tiles):
    check(gpu_ctx, sample_case, monkeypatch, {"XG_EPOCH_TILES": tiles}, barcodes=False)


@pytest.mark.parametrize("big", ["0", "300", str(1 << 40)])
@pytest.mark.parametrize("tiles", ["2", "97"])
def test_all_some_or_no_big_segments(gpu_ctx, case, monkeypatch, big, tiles):
    t = check(gpu_ctx, case, monkeypatch, {"XG_SEG_BIG": big, "XG_EPOCH_TILES": tiles})
    assert t[14] > 0 and t[15] == 0


@pytest.mark.parametrize("tiles", ["1", "3", "97"])
def test_every_feature_a_set(gpu_ctx, case, monkeypatch, tiles):
    t = check(gpu_ctx, case, monkeypatch, {"XG_SEG_MAX": "0", "XG_EPOCH_TILES": tiles})
    assert t[14] == 0 and t[15] > 0


def test_sets_and_segments_mixed(gpu_ctx, case, monkeypatch):
    t = check(gpu_ctx, case, monkeypatch, {"XG_SEG_MAX": "200", "XG_SEG_BIG": "100", "XG_EPOCH_TILES": "2"})
    assert t[14] > 0 and t[15] > 0


@pytest.mark.parametrize("tiles", ["1", "2", "5"])
def test_streaming_call(gpu_ctx, case, monkeypatch, tiles):
    check(gpu_ctx, case, monkeypatch, {"XG_EPOCH_TILES_HOST": tiles}, host=True)


def test_calls_back_to_back_resize_the_plan(gpu_ctx, case, sample_case, monkeypatch):
    small = make_case(3, 1, 8000, 500000, 40)
    large = make_case(4, 1, 150000, 4000000, 900)
    pools = []
    for c, env, bc in ((small, {}, True), (large, {"XG_EPOCH_TILES": "3"}, True), (small, {"XG_EPOCH_TILES": "1"}, True),
                       (sample_case, {}, False), (large, {"XG_SEG_MAX": "0"}, True), (case, {}, True)):
        pools.append(check(gpu_ctx, c, monkeypatch, env, barcodes=bc)[6])
    assert pools[1] > pools[0]
