"""Seeking with the BAM index on the device decoder: a multi-range decode equals the host decode of a BAM made of the
same blocks, array for array; and fc_wrapper / afc_wrapper / pileup_wrapper write the same bytes with and without a
.bai next to the BAM while reading only the ranges' share of the file."""

import os
import random
import shutil

import pytest

import bai
from test_gpu_decode import assert_same_batch, full_maps, host_decode, tenx_bam

pytestmark = pytest.mark.gpu


def cut_bam(src, ranges, dst):
    """The header blocks of `src`, then the records of `ranges` (virtual offset of the first record, file offset after
    the last block), then the EOF block: a BAM holding exactly the records those ranges decode.  A range that starts
    inside a block gets that block's tail as a block of its own."""
    from xcltk_b200 import lib, synth
    off, first, aligned = lib.bgzf_block_index(src)
    assert aligned
    inflated = dict(bai.bgzf_blocks(src))
    with open(src, "rb") as fp:
        data = fp.read()
    with open(dst, "wb") as fp:
        fp.write(data[:off[first]])
        for lo, hi in ranges:
            c, skip = max(lo >> 16, int(off[first])), lo & 0xffff
            if skip:
                fp.write(synth._bgzf_block(inflated[c][skip:]))
                c = int(off[list(off).index(c) + 1])
            fp.write(data[c:hi])
        fp.write(synth.BGZF_EOF)


def random_ranges(path, n, seed):
    """n ascending, disjoint ranges behind the header, each starting at a random record of its first block (the last
    block before EOF included at random)"""
    from xcltk_b200 import lib
    off, first, _ = lib.bgzf_block_index(path)
    starts = {}
    for _t, _p, _e, _f, vb, _ve in bai.bam_records(path)[1]:
        starts.setdefault(vb >> 16, []).append(vb)
    n_data = len(off) - 2 - first                              # data blocks (the EOF block left out)
    rng = random.Random(seed)
    cuts = sorted(rng.sample(range(n_data + 1), min(2 * n, n_data + 1 - (n_data + 1) % 2)))
    return [(rng.choice(starts[int(off[first + a])]), int(off[first + b])) for a, b in zip(cuts[::2], cuts[1::2])
            if b > a]


def check_ranges(ctx, paths, range_lists, tmp_path, maps=None, want_seq=True):
    maps = maps or full_maps(paths)
    cuts = []
    for k, (p, rl) in enumerate(zip(paths, range_lists)):
        q = str(tmp_path / ("cut%d.bam" % k))
        cut_bam(p, rl if rl is not None else [(lib_first(p) << 16, os.path.getsize(p) - 28)], q)
        cuts.append(q)
    host = host_decode(cuts, maps, "CB", "UB", want_seq)
    dev, seen = ctx.decode_bams(paths, maps, "CB", "UB", want_seq, range_lists=range_lists)
    assert_same_batch(dev, seen, host)
    br = dev.bytes_read
    dev.close()
    return host, br


def lib_first(p):
    from xcltk_b200 import lib
    off, first, _ = lib.bgzf_block_index(p)
    return int(off[first])


@pytest.mark.parametrize("n_ranges", [1, 2, 40])
@pytest.mark.parametrize("small", [False, True])
def test_multi_range_decode_equals_host_decode_of_the_same_blocks(gpu_ctx, tmp_path, monkeypatch, n_ranges, small):
    """ranges cut runs and contigs; with small staging chunks and windows they also cross chunks and windows"""
    if small:
        monkeypatch.setenv("XG_STAGE_BYTES", str(132 << 10))
        monkeypatch.setenv("XG_DECODE_WINDOW", str(300000))
    p = tenx_bam(tmp_path, 40000, 21, level=1)
    rl = random_ranges(p, n_ranges, 3 + n_ranges)
    assert len(rl) == n_ranges and any(lo & 0xffff for lo, _hi in rl)       # ranges start inside blocks too
    host, br = check_ranges(gpu_ctx, [p], [rl], tmp_path)
    assert len(host.runs) >= 1 and host.n > 0
    header = min(os.path.getsize(p), 64 << 10)
    assert br <= sum(hi - (lo >> 16) for lo, hi in rl) + header
    if small and n_ranges == 40:
        assert gpu_ctx.timing()[5] >= 3                         # windows


def test_two_bams_and_empty_and_whole_lists(gpu_ctx, tmp_path):
    p = tenx_bam(tmp_path, 30000, 22, "a.bam", level=1)
    q = tenx_bam(tmp_path, 12000, 23, "b.bam", level=6)
    maps = full_maps([p, q])
    maps[1][1] = -1
    check_ranges(gpu_ctx, [p, q], [random_ranges(p, 5, 1), random_ranges(q, 3, 2)], tmp_path, maps)
    check_ranges(gpu_ctx, [p, q], [None, random_ranges(q, 7, 4)], tmp_path, maps)      # whole file + ranges
    check_ranges(gpu_ctx, [p, q], [random_ranges(p, 1, 5), []], tmp_path, maps)          # nothing of the second BAM
    from xcltk_b200 import lib
    off, first, _ = lib.bgzf_block_index(p)
    # a first range from the file's start (header inflated in the stream), then another
    check_ranges(gpu_ctx, [p], [[(0, int(off[first + 5])), (int(off[first + 9]) << 16, int(off[first + 12]))]],
                 tmp_path)
    # every data block as one range each: the same batch as the whole file
    each = [(int(off[i]) << 16, int(off[i + 1])) for i in range(first, len(off) - 1)]
    dev, seen = gpu_ctx.decode_bams([p], full_maps([p]), "CB", "UB", True, range_lists=[each])
    assert_same_batch(dev, seen, host_decode([p], full_maps([p]), "CB", "UB", True))
    dev.close()


def test_cross_block_bam_is_still_declined(gpu_ctx, tmp_path):
    """records cross blocks: a range that starts at any block -- most of them inside a record -- or at a record is
    declined, and the caller decodes the whole file on the host"""
    from xcltk_b200 import lib
    p = tenx_bam(tmp_path, 8000, 24, align=False)
    off, _first, _ = lib.bgzf_block_index(p)
    maps = full_maps([p])

    def decode(lo, hi):
        return gpu_ctx.decode_bams([p], maps, "CB", "UB", True, range_lists=[[(lo, hi)]])
    for i in range(1, len(off) - 2):
        assert decode(int(off[i]) << 16, int(off[-1])) is None
        assert decode(int(off[i]) << 16, int(off[i + 1])) is None
    for _t, _p, _e, _f, vb, _ve in bai.bam_records(p)[1][::97]:
        if (vb >> 16) < off[-3]:                               # the last data block's records cross no boundary
            assert decode(vb, int(off[-1])) is None
    assert gpu_ctx.decode_bams([p], maps, "CB", "UB", True) is None


def test_ranges_that_do_not_fit_the_file_are_an_argument_error(gpu_ctx, tmp_path):
    from xcltk_b200 import lib
    p = tenx_bam(tmp_path, 3000, 25)
    size = os.path.getsize(p)
    f = lib_first(p) << 16
    for rl in ([(100 << 16, 50)], [(f, size + 1)], [(f, size - 28), (f, size - 28)]):
        with pytest.raises(lib.XgError):
            gpu_ctx.decode_bams([p], full_maps([p]), "CB", "UB", True, range_lists=[rl])
    assert gpu_ctx.decode_bams([p], full_maps([p]), "CB", "UB", True) is not None      # still usable


# ---- end to end: the same bytes with and without the index ------------------------------------------------------

CONTIGS = [("1", 2600000), ("2", 1800000), ("3", 1500000), ("7", 900000), ("22", 1200000)]


@pytest.fixture(scope="module")
def library(tmp_path_factory):
    from xcltk_b200 import synth
    d = tmp_path_factory.mktemp("seek")
    rng = random.Random(41)
    feats = synth.synth_features(rng, [(c, l - 20000) for c, l in CONTIGS], 400, mean_len=15000)
    for c, l in CONTIGS:                                        # features at contig starts and ends
        feats += [(c, 1, 4000, "s" + c), (c, l - 16000, l - 6200, "e" + c)]
    barcodes = synth.make_barcodes(rng, 60)
    snps = synth.gen_snps(42, feats, 3000)
    out = {"dir": str(d), "feats": feats, "snps": snps}
    bams = []
    for k, n in enumerate((150000, 30000, 30000)):
        refs, recs = synth.gen_10x_records(50 + k, CONTIGS, feats, n, barcodes, snps=snps, chr_prefix="chr")
        p = str(d / ("lib%d.bam" % k))
        synth.write_bam(p, refs, recs, level=1)
        bams.append(p)
    out["bams"] = bams
    out["barcodes"] = str(d / "barcodes.tsv")
    synth.write_lines(out["barcodes"], barcodes)
    out["snp_tsv"] = str(d / "snps.tsv")
    synth.write_snp_tsv(out["snp_tsv"], snps, chr_prefix="chr")
    return out


def _subset(lib_, case):
    rng = random.Random(7)
    feats = lib_["feats"]
    if case == "one_contig":
        return [f for f in feats if f[0] == "3"]
    if case == "subset_1pct":
        return sorted(rng.sample(feats, max(3, len(feats) // 100)), key=lambda f: (int(f[0]), f[1]))
    if case == "edges":
        return [f for f in feats if f[3][0] in "se"]
    if case == "absent":
        return [f for f in feats if f[0] == "7"] + [("9", 1000, 50000, "x1"), ("X", 5, 900, "x2")]
    return feats


def _run_twice(tmp_path, monkeypatch, bams, run, index=(True,)):
    """run(out_dir) without any .bai and with .bai files next to bams[i] where index[i]; returns both directories'
    bytes and the compressed bytes each run's decode read."""
    from xcltk_b200 import engine
    os.makedirs(str(tmp_path), exist_ok=True)
    read = []
    real = engine.load_reads

    def spy(*a, **kw):
        b = real(*a, **kw)
        read.append(b.stats.get("bytes_read"))
        return b
    monkeypatch.setattr(engine, "load_reads", spy)
    res = []
    for with_index in (False, True):
        for k, p in enumerate(bams):
            if os.path.exists(p + ".bai"):
                os.remove(p + ".bai")
            if with_index and index[k % len(index)]:
                bai.index_bam(p)
        out = str(tmp_path / ("idx" if with_index else "whole"))
        assert run(out) == 0
        res.append({f: open(os.path.join(out, f), "rb").read() for f in sorted(os.listdir(out))})
    for p in bams:
        if os.path.exists(p + ".bai"):
            os.remove(p + ".bai")
    assert res[0] == res[1]
    assert len(read) == 2 and None not in read
    return res[0], read


@pytest.mark.parametrize("case", ["one_contig", "subset_1pct", "edges", "absent", "all"])
def test_fc_and_afc_same_bytes_with_and_without_index(library, tmp_path, monkeypatch, case):
    from xcltk_b200 import synth
    from xcltk_b200.baf.fc.main import afc_wrapper
    from xcltk_b200.rdr.fc.main import fc_wrapper
    bam = library["bams"][0]
    feats = _subset(library, case)
    ft = str(tmp_path / "features.tsv")
    synth.write_features(ft, [("chr" + c, s, e, n) for c, s, e, n in feats])
    size = os.path.getsize(bam)
    files, read = _run_twice(tmp_path / "fc", monkeypatch, [bam],
                             lambda out: fc_wrapper(bam, library["barcodes"], ft, out, ncores=4))
    assert files["matrix.mtx"].count(b"\n") > 20 or case == "absent"
    if case == "all":
        assert read[1] >= 0.9 * read[0]
    else:
        assert read[1] < 0.6 * read[0] and read[0] >= size
    files, read = _run_twice(tmp_path / "afc", monkeypatch, [bam],
                             lambda out: afc_wrapper(bam, library["barcodes"], ft, library["snp_tsv"], out, ncores=4,
                                                     output_all_reg=True))
    if case != "all":
        assert read[1] < 0.6 * read[0]


def test_afc_with_cellsnp_dir_and_local_phasing(library, tmp_path, monkeypatch):
    from xcltk_b200 import synth
    from xcltk_b200.baf.fc.main import afc_wrapper
    from xcltk_b200.baf.pileup import pileup_wrapper
    bam = library["bams"][0]
    feats = [f for f in library["feats"] if f[0] in ("2", "22")]
    ft = str(tmp_path / "features.tsv")
    synth.write_features(ft, [("chr" + c, s, e, n) for c, s, e, n in feats])
    csd = str(tmp_path / "cellsnp")
    assert pileup_wrapper(bam, library["barcodes"], library["snp_tsv"], csd, ncores=4) == 0
    files, read = _run_twice(tmp_path, monkeypatch, [bam],
                             lambda out: afc_wrapper(bam, library["barcodes"], ft, library["snp_tsv"], out,
                                                     cellsnp_dir=csd, ncores=4, output_all_reg=True))
    assert files["xcltk.DP.mtx"].count(b"\n") > 20
    assert read[1] < 0.8 * read[0]


def test_pileup_with_candidates_and_discovery(library, tmp_path, monkeypatch):
    from xcltk_b200.baf.pileup import pileup_wrapper
    bam = library["bams"][0]
    snp22 = str(tmp_path / "snps22.tsv")
    with open(library["snp_tsv"]) as fp:
        lines = fp.read().splitlines()
    open(snp22, "w").write("\n".join([lines[0]] + [x for x in lines[1:] if x.startswith("chr22\t")]) + "\n")
    files, read = _run_twice(tmp_path / "cand", monkeypatch, [bam],
                             lambda out: pileup_wrapper(bam, library["barcodes"], snp22, out, ncores=4))
    assert files["cellSNP.tag.DP.mtx"].count(b"\n") > 20 and read[1] < 0.4 * read[0]
    for chrom in ("22", "22,3,1"):
        files, read = _run_twice(tmp_path / chrom.replace(",", "_"), monkeypatch, [bam],
                                 lambda out: pileup_wrapper(bam, library["barcodes"], None, out, ncores=4, chrom=chrom,
                                                            min_count=3, min_maf=0.1))
        assert files["cellSNP.tag.DP.mtx"].count(b"\n") > 20
        if chrom == "22":
            assert read[1] < 0.4 * read[0]


def test_sample_mode_three_bams_one_indexed(library, tmp_path, monkeypatch):
    from xcltk_b200 import synth
    from xcltk_b200.rdr.fc.main import fc_wrapper
    bams = library["bams"]
    feats = [f for f in library["feats"] if f[0] == "1"][:30]
    ft = str(tmp_path / "features.tsv")
    synth.write_features(ft, [("chr" + c, s, e, n) for c, s, e, n in feats])
    files, read = _run_twice(tmp_path, monkeypatch, bams,
                             lambda out: fc_wrapper(",".join(bams), None, ft, out, sample_ids="A,B,C", cell_tag=None,
                                                    ncores=4), index=(False, True, False))
    assert files["matrix.mtx"].count(b"\n") > 20
    assert read[1] < read[0]


def test_bch869_goldens_through_the_seek_path(tmp_path, monkeypatch, gpu_ctx):
    """the reference's htslib-written BAM with a test-written .bai: its golden runs give the same bytes"""
    from util import BAF_FILES, GOLD, RDR_FILES, compare_dirs, golden_runs, read, resolve
    from xcltk_b200 import engine
    bam = str(tmp_path / "BCH869.output.bam")
    shutil.copy(os.path.join(GOLD, "bch869_smartseq", "BCH869.output.bam"), bam)
    bai.index_bam(bam)
    seen = []
    real = engine.load_reads

    def spy(*a, **kw):
        b = real(*a, **kw)
        seen.append(b.stats)
        return b
    monkeypatch.setattr(engine, "load_reads", spy)
    for run in [r for c, r in golden_runs() if c == "bch869_smartseq"]:
        r = resolve("bch869_smartseq", run)
        out = str(tmp_path / run)
        if r["kind"] == "basefc":
            from xcltk_b200.rdr.fc.main import fc_wrapper
            ret = fc_wrapper(bam, r["barcodes"], r["features"], out, **r["kwargs"])
            files = RDR_FILES
        else:
            from xcltk_b200.baf.fc.main import afc_wrapper
            ret = afc_wrapper(bam, r["barcodes"], r["features"], r["snps"], out, **r["kwargs"])
            files = BAF_FILES
        assert ret == int(read(r["expected"] + "/RETCODE")) == 0
        compare_dirs(r["expected"], out, files)
    assert seen and all(s.get("range_lists") is not None for s in seen)
