"""Host side of `xcltk pileup`: the candidate-site loader, the cellSNP directory writer and the command line."""

import gzip
import os

import numpy as np
import pytest
import scipy.io

from xcltk_b200.baf import pileup
from xcltk_b200.utils import csp_io

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

SITES = [  # (CHROM, POS, REF, ALT): kept?
    ("chr1", "100", "a", "g", True),        # lowercase
    ("1", "200", "N", "C", True),           # REF N
    ("chr1", "300", "T", "n", True),        # ALT n
    ("1", "400", "A", "C,G", False),        # multi-allelic
    ("1", "500", "AT", "A", False),         # deletion
    ("1", "600", "C", "CTT", False),        # insertion
    ("Chr2", "700", "G", "R", False),       # IUPAC ALT
    ("2", "800", "G", ".", False),          # no ALT
    ("chr1", "100", "A", "G", True),        # duplicate site
    ("X", "1", "c", "c", True),             # REF == ALT
]
KEPT = [s for s in SITES if s[4]]


def check_sites(snp_set):
    got = [(s.chrom_text, s.chrom, s.pos, s.ref, s.alt, s.ref_idx, s.alt_idx, s.index) for s in snp_set.snps]
    exp = [(c, c[3:] if c.lower().startswith("chr") else c, int(p), r.upper(), a.upper(), 0, 1, k)
           for k, (c, p, r, a, _) in enumerate(KEPT)]
    assert got == exp
    assert [s.pos for s in snp_set.fetch("chr1", 100, 101)] == [100, 100]      # both duplicates, 'chr' stripped


def test_vcf_sites_without_genotype(tmp_path, capsys):
    fn = str(tmp_path / "sites.vcf")
    with open(fn, "w") as fp:
        fp.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\n")
        for c, p, r, a, _ in SITES:
            fp.write("%s\t%s\t.\t%s\t%s\n" % (c, p, r, a))
        fp.write("1\t900\t.\tA\n")                                            # too few columns
    check_sites(pileup.load_sites(fn))
    err = capsys.readouterr().err
    assert err.count("invalid ALT base") == 4 and err.count("invalid REF base") == 1 and "too few columns" in err


def test_vcf_sites_ignore_genotype_columns(tmp_path):
    fn = str(tmp_path / "sites.vcf.gz")
    with gzip.open(fn, "wt") as fp:
        fp.write("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\n")
        for (c, p, r, a, _), gt in zip(SITES, ["0|1", "1/1", "0/0", "./.", "1|0", "0|0", "0|1", "1|1", "0/1", "."]):
            fp.write("%s\t%s\t.\t%s\t%s\t.\tPASS\t.\tGT\t%s\n" % (c, p, r, a, gt))
    check_sites(pileup.load_sites(fn))


def test_tsv_sites_use_four_columns(tmp_path):
    fn = str(tmp_path / "sites.tsv")
    with open(fn, "w") as fp:
        fp.write("chrom\tpos\tref\talt\tref_hap\talt_hap\n")
        for k, (c, p, r, a, _) in enumerate(SITES):
            fp.write("%s\t%s\t%s\t%s" % (c, p, r, a) + ("\t1\t1\n" if k % 2 else "\n"))
    check_sites(pileup.load_sites(fn))


def test_phased_loaders_are_unchanged(tmp_path):
    """Without `sites` the readers still need and honour a phased genotype."""
    from xcltk_b200.baf.fc.utils import load_snp_from_tsv
    fn = str(tmp_path / "snps.tsv")
    with open(fn, "w") as fp:
        fp.write("chrom\tpos\tref\talt\tref_hap\talt_hap\nchr1\t5\tA\tG\t1\t0\n1\t6\tA\tG\n1\t7\tA\tG\t1\t1\n")
    s = load_snp_from_tsv(fn)
    assert [(x.pos, x.ref_idx, x.alt_idx) for x in s.snps] == [(5, 1, 0)]
    assert not hasattr(s.snps[0], "chrom_text")


# ------------------------------------------------------------------------------------------ writer
def triples(rows, cols, vals, n_rows, n_cols):
    return (np.asarray(rows, np.int32), np.asarray(cols, np.int32), np.asarray(vals, np.int32), (n_rows, n_cols))


class Site(object):
    def __init__(self, chrom_text, pos, ref, alt):
        self.chrom_text, self.chrom, self.pos, self.ref, self.alt = chrom_text, chrom_text[3:], pos, ref, alt


SNPS = [Site("chr1", 10, "A", "G"), Site("chr1", 20, "C", "T"), Site("chr2", 5, "G", "G"), Site("chr2", 9, "N", "A")]
SAMPLES = ["AAAC-1", "AAAG-1", "CCCT-1"]


def write(tmp_path, name, ad, dp, oth, keep):
    out = tmp_path / name
    out.mkdir()
    pileup.write_cellsnp_dir(str(out), SAMPLES, SNPS, ad, dp, oth, np.array(keep, np.uint8))
    return str(out)


def written(tmp_path, name):
    ad = triples([0, 2, 2, 3], [1, 0, 2, 0], [2, 1, 7, 1], 4, 3)
    dp = triples([0, 0, 2, 2, 3], [0, 1, 0, 2, 0], [1, 3, 1, 7, 1], 4, 3)
    oth = triples([1, 3], [2, 1], [4, 1], 4, 3)
    return write(tmp_path, name, ad, dp, oth, [1, 1, 1, 1])


def test_writer_all_kept(tmp_path):
    out = written(tmp_path, "a")
    with open(os.path.join(out, "cellSNP.samples.tsv")) as fp:
        assert fp.read() == "AAAC-1\nAAAG-1\nCCCT-1\n"
    raw = open(os.path.join(out, "cellSNP.base.vcf.gz"), "rb").read()
    assert raw[:4] == b"\x1f\x8b\x08\x00" and raw[4:8] == b"\0\0\0\0"           # no file name, mtime 0
    assert gzip.decompress(raw).decode() == (
        "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
        "chr1\t10\t.\tA\tG\t.\tPASS\tAD=2;DP=4;OTH=0\n"
        "chr1\t20\t.\tC\tT\t.\tPASS\tAD=0;DP=0;OTH=4\n"
        "chr2\t5\t.\tG\tG\t.\tPASS\tAD=8;DP=8;OTH=0\n"
        "chr2\t9\t.\tN\tA\t.\tPASS\tAD=1;DP=1;OTH=1\n")
    with open(os.path.join(out, "cellSNP.tag.DP.mtx")) as fp:
        lines = fp.read().split("\n")
    assert lines[0].startswith("%%MatrixMarket matrix coordinate integer general")
    assert lines[1] == "%%" and lines[2] == "4\t3\t5"
    assert lines[3:] == ["1\t1\t1", "1\t2\t3", "3\t1\t1", "3\t3\t7", "4\t1\t1", ""]
    d = csp_io.load_data(out)
    assert list(d.cells) == SAMPLES and list(d.chrom) == ["chr1", "chr1", "chr2", "chr2"]
    assert list(d.pos) == [10, 20, 5, 9]
    assert (d.AD.toarray() == np.array([[0, 0, 1, 1], [2, 0, 0, 0], [0, 0, 7, 0]])).all()
    assert (d.DP.toarray() == np.array([[1, 0, 1, 1], [3, 0, 0, 0], [0, 0, 7, 0]])).all()
    oth = scipy.io.mmread(os.path.join(out, "cellSNP.tag.OTH.mtx"))
    assert (np.asarray(oth.todense()) == np.array([[0, 0, 0], [0, 0, 4], [0, 0, 0], [0, 1, 0]])).all()
    again = written(tmp_path, "b")
    for f in os.listdir(out):
        assert open(os.path.join(out, f), "rb").read() == open(os.path.join(again, f), "rb").read(), f


def test_writer_drops_filtered_rows(tmp_path):
    """SNPs 1 and 3 removed by the filter (their rows would be empty): rows renumber over the kept SNPs."""
    ad = triples([0, 2, 2], [1, 0, 2], [2, 1, 7], 4, 3)
    dp = triples([0, 0, 2, 2], [0, 1, 0, 2], [1, 3, 1, 7], 4, 3)
    oth = triples([], [], [], 4, 3)
    out2 = write(tmp_path, "filtered", ad, dp, oth, [1, 0, 1, 0])
    with open(os.path.join(out2, "cellSNP.tag.AD.mtx")) as fp:
        assert fp.read().split("\n")[2:] == ["2\t3\t3", "1\t2\t2", "2\t1\t1", "2\t3\t7", ""]
    assert gzip.decompress(open(os.path.join(out2, "cellSNP.base.vcf.gz"), "rb").read()).decode().split("\n")[2:] == [
        "chr1\t10\t.\tA\tG\t.\tPASS\tAD=2;DP=4;OTH=0", "chr2\t5\t.\tG\tG\t.\tPASS\tAD=8;DP=8;OTH=0", ""]
    d = csp_io.load_data(str(out2))
    assert d.shape == (3, 2) and list(d.pos) == [10, 5]
    with open(os.path.join(out2, "cellSNP.tag.OTH.mtx")) as fp:
        assert fp.read().split("\n")[2:] == ["2\t3\t0", ""]


# ------------------------------------------------------------------------------------------ command line
def test_usage_for_two_or_fewer_args(capsys):
    for argv in (["xcltk", "pileup"], ["xcltk"]):
        with pytest.raises(SystemExit) as e:
            pileup.pileup_main(argv)
        assert e.value.code == 0
    out = capsys.readouterr().out
    assert "Usage:   xcltk pileup <options>" in out and "--snpvcf FILE" in out and "--minMAF FLOAT" in out


def test_help_lists_the_command(capsys):
    from xcltk_b200 import xcltk
    with pytest.raises(SystemExit) as e:
        xcltk.main(["xcltk", "--help"])
    assert e.value.code == 0
    out = capsys.readouterr().out
    head, tail = out.split("-- BAF calculation")
    assert "pileup" in tail.split("-- Others")[0] and "pileup" not in head


def test_parse_options():
    from xcltk_b200.baf.fc.config import Config
    conf = Config()
    argv = ["xcltk", "pileup", "-s", "a.bam", "-b", "bc.tsv", "-P", "s.vcf", "-O", "out", "-p", "4", "--cellTAG", "RG",
            "--UMItag", "None", "-D", "2", "--minCOUNT", "3", "--minMAF", "0.25", "--inclFLAG", "2", "--exclFLAG", "4",
            "--minLEN", "20", "--minMAPQ", "7.5", "--countORPHAN"]
    assert pileup.parse_args(argv, conf) is None
    assert (conf.sam_fn, conf.barcode_fn, conf.snp_fn, conf.out_dir, conf.nproc) == ("a.bam", "bc.tsv", "s.vcf", "out", 4)
    assert (conf.cell_tag, conf.umi_tag, conf.debug) == ("RG", "None", 2)
    assert (conf.min_count, conf.min_maf, conf.incl_flag, conf.excl_flag) == (3, 0.25, 2, 4)
    assert (conf.min_len, conf.min_mapq, conf.no_orphan) == (20, 7.5, False)
    conf = Config()
    assert pileup.parse_args(["xcltk", "pileup", "-S", "l.txt", "-I", "a,b", "--snpvcf", "x.tsv",
                              "--outdir", "o", "-i", "ids.txt"], conf) is None
    assert (conf.sam_list_fn, conf.sample_id_str, conf.snp_fn, conf.out_dir, conf.sample_id_fn) == \
        ("l.txt", "a,b", "x.tsv", "o", "ids.txt")
    assert pileup.parse_args(["xcltk", "pileup", "--help"], Config()) == "--help"


def test_input_errors_return_minus_one(tmp_path):
    bam = os.path.join(GOLD, "c1_chr22_10x", "a.bam")
    bc = os.path.join(GOLD, "c1_chr22_10x", "barcodes.tsv")
    out = str(tmp_path / "o")
    assert pileup.pileup_wrapper(bam, bc, str(tmp_path / "missing.vcf"), out) == -1
    assert pileup.pileup_wrapper(bam, bc, None, out) == -1
    assert pileup.pileup_wrapper(bam, None, os.path.join(GOLD, "c1_chr22_10x", "snps.tsv"), out) == -1  # CB, no barcodes
    empty = str(tmp_path / "empty.vcf")
    with open(empty, "w") as fp:
        fp.write("#CHROM\tPOS\tID\tREF\tALT\n1\t5\t.\tAT\tA\n")
    assert pileup.pileup_wrapper(bam, bc, empty, out) == -1
