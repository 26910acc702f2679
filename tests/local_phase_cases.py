"""Inputs of the local-phasing tests and the two ways of running them: the host reference (reg_local_phasing region by
region in list order, as afc_core runs it on cellsnp-lite counts) and the device (local_phasing_device, in waves)."""

import os
import warnings

import numpy as np

from util import GOLD

C1 = os.path.join(GOLD, "c1_chr22_10x")
C2 = os.path.join(GOLD, "c2_local_phasing")


class Case(object):
    """pos / ref0: per SNP; AD / DP: cells x SNPs (the cells that take part); regions: SNP id lists, list order."""

    def __init__(self, pos, ref0, AD, DP, regions, name="case"):
        self.pos = np.asarray(pos, dtype=np.int64)
        self.ref0 = np.asarray(ref0, dtype=np.int64)
        self.AD = np.asarray(AD, dtype=np.int64)
        self.DP = np.asarray(DP, dtype=np.int64)
        self.regions = [list(r) for r in regions]
        self.name = name

    def snps(self):
        from xcltk_b200.baf.fc.gfeature import SNP
        out = []
        for i, (p, r) in enumerate(zip(self.pos, self.ref0)):
            s = SNP("1", int(p), "A", "G", int(r), 1 - int(r))
            s.index = i
            out.append(s)
        return out

    def regs(self, snps):
        from xcltk_b200.baf.fc.gfeature import BlockRegion
        return [BlockRegion("1", int(self.pos[r[0]]) if r else 1, int(self.pos[r[-1]]) + 1 if r else 2, "r%d" % k,
                            [snps[i] for i in r]) for k, r in enumerate(self.regions)]

    def csr(self):
        from xcltk_b200.baf.fc.phasing import csr_from_coo
        n_cells = self.DP.shape[0]
        r, c = np.nonzero(self.DP.T)
        ar, ac = np.nonzero(self.AD.T)
        return csr_from_coo(len(self.pos), (ar, ac, self.AD.T[ar, ac]), (r, c, self.DP.T[r, c]),
                            np.ones(n_cells, dtype=bool))


def _result(regs, snps, flips):
    return {"lists": [[s.index for s in reg.snp_list] for reg in regs],
            "flips": [None if f is None else [int(x) for x in f] for f in flips],
            "ref_idx": [s.ref_idx for s in snps], "alt_idx": [s.alt_idx for s in snps],
            "gt": [sorted(s.gt.items()) for s in snps],
            "counters": (len(regs), sum(f is None for f in flips), sum(len(r.snp_list) for r in regs),
                         int(sum(np.sum(f) for f in flips if f is not None)))}


def host_run(case):
    from xcltk_b200.baf.fc.phasing import reg_local_phasing
    snps = case.snps()
    regs = case.regs(snps)
    flips = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for reg in regs:
            ids = sorted(s.index for s in reg.snp_list)      # the cellsnp path's columns: SNP file order
            _reg, f = reg_local_phasing(reg, case.AD[:, ids], case.DP[:, ids])
            flips.append(f)
    return _result(regs, snps, flips)


def device_run(ctx, case):
    from xcltk_b200.baf.fc.phasing import local_phasing_device
    snps = case.snps()
    regs = case.regs(snps)
    flips, timing = local_phasing_device(ctx, regs, snps, case.csr(), case.DP.shape[0])
    out = _result(regs, snps, flips)
    out["timing"] = timing
    return out


def imbalanced(seed, n_snp, n_cell, dens, spacing, n_regions=1, overlap=0, p_hi=0.85):
    """Seeded SNP x cell counts with allele-imbalanced cells (BAF p or 1 - p per cell and haplotype) and a random
    reference phasing; regions of n_snp // n_regions consecutive SNPs, each sharing `overlap` SNPs with the next."""
    rng = np.random.default_rng(seed)
    DP = (rng.random((n_cell, n_snp)) < dens) * rng.integers(1, 4, (n_cell, n_snp))
    hap = rng.random(n_snp) < 0.5
    p = np.where(rng.random(n_cell) < 0.5, p_hi, 1 - p_hi)[:, None]
    p = np.where(hap[None, :], 1 - p, p)
    AD = rng.binomial(DP, p)
    pos = 1000 + np.cumsum(rng.integers(max(1, spacing // 2), spacing * 3 // 2 + 1, n_snp))
    ref0 = (rng.random(n_snp) < 0.5).astype(np.int64)
    step = n_snp // n_regions
    regions = [list(range(max(0, k * step - overlap), min(n_snp, (k + 1) * step))) for k in range(n_regions)]
    return Case(pos, ref0, AD, DP, regions, "imbalanced%d" % seed)


def small_seeded(seed):
    """The small inputs of the seed search in test_gpu_local_phase (one region, 2..6 SNPs, 3..11 cells)."""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(2, 7))
    c = int(rng.integers(3, 12))
    spacing = int(rng.choice([300, 30000, 700000]))
    DP = (rng.random((c, n)) < 0.6) * rng.integers(1, 4, (c, n))
    hap = rng.random(n) < 0.5
    p = np.where(rng.random(c) < 0.5, 0.85, 0.15)[:, None]
    p = np.where(hap[None, :], 1 - p, p)
    AD = rng.binomial(DP, p)
    return Case(1000 + np.arange(n) * spacing, np.zeros(n, np.int64), AD, DP, [list(range(n))], "small%d" % seed)


def golden_c2(with_ref_cells):
    """The 65 long regions of the C2 golden inputs (c1_chr22_10x regions and SNPs, the cellsnp-lite directory of
    c2_local_phasing), as afc_core selects them; AD / DP = the cellsnp matrices over the SNP file's SNPs, minus the
    reference cells when asked.  Returns (Case, [cols of the cellsnp path per region], cellsnp data, the cellsnp
    column of every SNP)."""
    return cellsnp_case(os.path.join(C1, "features.tsv"), os.path.join(C1, "snps.tsv"), os.path.join(C2, "cellsnp"),
                        os.path.join(C2, "ref_cells.tsv") if with_ref_cells else None,
                        "c2" + ("_ref_cells" if with_ref_cells else ""))


def cellsnp_case(features, snp_fn, csp_dir, ref_cell_fn=None, name="cellsnp"):
    """The long regions of `features` with the counts of a cellsnp-lite directory, as afc_core selects them."""
    from xcltk_b200.baf.fc.config import Config
    from xcltk_b200.baf.fc.phasing import is_long_region
    from xcltk_b200.baf.fc.utils import load_region_from_txt, load_snp_from_tsv
    from xcltk_b200.utils.csp_io import load_data
    from xcltk_b200.utils.grange import format_chrom
    conf = Config()
    regs = load_region_from_txt(features)
    ss = load_snp_from_tsv(snp_fn)
    data = load_data(csp_dir)
    if ref_cell_fn:
        ref = np.atleast_1d(np.genfromtxt(ref_cell_fn, dtype="str", delimiter="\t"))
        data = data.subset_cells(~np.isin(data.cells.astype(str), ref))
    chrom = np.array([format_chrom(c) for c in data.chrom], dtype=object)
    at = {(format_chrom(c), int(p)): k for k, (c, p) in enumerate(zip(data.chrom, data.pos))}
    snps = ss.snps
    col_of = np.array([at[(s.chrom, s.pos)] for s in snps])
    AD = data.AD.toarray()[:, col_of]
    DP = data.DP.toarray()[:, col_of]
    regions, cols, names = [], [], []
    for reg in regs:
        sl = ss.fetch(reg.chrom, reg.start, reg.end)
        if not sl:
            continue
        reg.snp_list = sl
        if not is_long_region(conf, reg):
            continue
        regions.append([s.index for s in sl])
        names.append(reg.name)
        cols.append(np.nonzero((chrom == reg.chrom) & (data.pos >= reg.start) & (data.pos < reg.end))[0])
    case = Case([s.pos for s in snps], [s.ref_idx for s in snps], AD, DP, regions, name)
    case.names = names
    return case, cols, data, col_of
