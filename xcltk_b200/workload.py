"""Synthetic workloads of the shapes BASELINE.json names (SURVEY.md section 8(d) C1-C5).

Features: the hg38 gene table the reference ships (data/anno, first four columns, kept as
xcltk_b200/data/hg38_genes_4col.tsv.gz) optionally extended with seeded nested /
overlapping intervals; reads: generated directly in HBM by xg_synth_reads, spread
uniformly over the union of the feature spans (coordinate sorted by construction).
"""

import gzip
import os
import random

import numpy as np

from . import engine, lib

HERE = os.path.dirname(os.path.abspath(__file__))
GENES = os.path.join(HERE, "data", "hg38_genes_4col.tsv.gz")

HG38_CHROMS = [str(i) for i in range(1, 23)] + ["X", "Y"]
HG38_LEN = dict(zip(HG38_CHROMS, (
    248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636,
    138394717, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345,
    83257441, 80373285, 58617616, 64444167, 46709983, 50818468, 156040895, 57227415)))


def load_genes(chroms=None):
    """[(chrom, start1, end1_incl, name)] in file order."""
    out = []
    with gzip.open(GENES, "rt") as fp:
        for line in fp:
            c, s, e, n = line.rstrip("\n").split("\t")
            if chroms is None or c in chroms:
                out.append((c, int(s), int(e), n))
    return out


def extend_features(feats, n_total, seed=11):
    """Add seeded nested / overlapping intervals until n_total features (config 3: ~60k)."""
    rng = random.Random(seed)
    out = list(feats)
    k = 0
    while len(out) < n_total:
        c, s, e, _ = feats[rng.randrange(len(feats))]
        L = e - s + 1
        a = s + rng.randrange(max(1, L))
        ln = max(8, int(rng.expovariate(1.0 / max(200.0, L / 3.0))))
        b = min(HG38_LEN.get(c, e + ln), a + ln)
        out.append((c, max(1, a - rng.randrange(500)), b, "syn%d" % k))
        k += 1
    return out


def bin_features(bin_kb=1000):
    """Fixed-size genomic bins (config 5: 1 Mb bins -> 3 102 rows for hg38;
    xcltk/utils/gregion.py:200-227 get_fixsize_regions)."""
    out = []
    step = bin_kb * 1000
    for c in HG38_CHROMS:
        L = HG38_LEN[c]
        for k, s in enumerate(range(1, L + 1, step)):
            out.append((c, s, min(L, s + step - 1), "%s_bin%d" % (c, k)))
    return out


def merged_spans(feats, gid_of):
    """Union of the feature spans per contig: sorted, disjoint [beg0, end0) with gid."""
    by = {}
    for c, s, e, _ in feats:
        if c in gid_of and e >= s and s >= 1:
            by.setdefault(gid_of[c], []).append((s - 1, e))
    sg, sb, se = [], [], []
    for g in sorted(by):
        iv = sorted(by[g])
        cb, ce = iv[0]
        for b, e in iv[1:]:
            if b <= ce:
                ce = max(ce, e)
            else:
                sg.append(g), sb.append(cb), se.append(ce)
                cb, ce = b, e
        sg.append(g), sb.append(cb), se.append(ce)
    return np.array(sg, np.int32), np.array(sb, np.int32), np.array(se, np.int32)


class Conf(object):
    """The reference's default filters (rdr/fc/config.py:98-111, baf/fc/config.py:149-164)."""
    min_mapq, min_len, min_include = 20, 30, 0.9
    incl_flag, excl_flag, no_orphan = 0, 772, True
    cell_tag, umi_tag = "CB", "UB"

    def use_barcodes(self):
        return True

    def use_umi(self):
        return True


class Workload(object):
    pass


def feature_arrays(feats, gid_of):
    gid = np.array([gid_of.get(f[0], -1) for f in feats], dtype=np.int32)
    beg = np.array([f[1] - 1 for f in feats], dtype=np.int32)
    end = np.array([f[2] for f in feats], dtype=np.int32)
    return gid, beg, end


HALO_BP = 6000        # longest reference span of a synthetic read (91 bases + a 5 000 bp intron), rounded up


def genomic_chunk(ctx, n_total, seed, sg, sb, se, gid, beg, end, part):
    """One of `world` contiguous genomic chunks of a synthetic library, balanced by reads (the north star's
    multi-GPU split; the reference cuts its feature list into contiguous chunks the same way,
    rdr/fc/main.py:191-212).  Returns (feature indices of the chunk, first read, number of reads): the
    features whose start lies in the chunk, and every read that can overlap one of them (halo included).
    Reads are spread uniformly over the concatenated spans, so equal span length = equal reads."""
    rank, world = part
    lens = (se - sb).astype(np.int64)
    pre = np.concatenate([[0], np.cumsum(lens)])
    total = int(pre[-1])
    # coordinate of every feature start in the concatenated span space (starts lie inside spans)
    key_span = sg.astype(np.int64) << 32 | sb.astype(np.int64)
    key_feat = gid.astype(np.int64) << 32 | beg.astype(np.int64)
    si = np.clip(np.searchsorted(key_span, key_feat, side="right") - 1, 0, len(sg) - 1)
    u = pre[si] + np.clip(beg.astype(np.int64) - sb[si], 0, lens[si])
    valid = (gid >= 0) & (end > beg)
    lo_u, hi_u = total * rank // world, total * (rank + 1) // world
    mine = np.nonzero(valid & (u >= lo_u) & (u < hi_u))[0]
    if rank == world - 1:          # features that can never be fetched travel with the last chunk (empty rows)
        mine = np.concatenate([mine, np.nonzero(~valid)[0]])
        mine.sort()
    ok = mine[valid[mine]]
    if len(ok) == 0:
        return mine, 0, 0
    order = np.lexsort((beg[ok], gid[ok]))
    first = ok[order[0]]
    last_key = np.max(gid[ok].astype(np.int64) << 32 | end[ok].astype(np.int64))
    g0, p0 = int(gid[first]), max(0, int(beg[first]) - HALO_BP)
    g1, p1 = int(last_key >> 32), int(last_key & 0xFFFFFFFF)
    i0 = lib.synth_read_index(n_total, sg, sb, se, g0, p0, seed=seed)
    i1 = lib.synth_read_index(n_total, sg, sb, se, g1, p1, seed=seed)
    return mine, i0, max(0, i1 - i0)


def make_basefc_workload(ctx, n_reads, n_cells, n_features=33472, seed=7, chroms=None, bins_kb=None, part=None):
    """Config 1 (chr22 only: chroms={'22'}), config 3 (n_features ~ 60k) or config 5 (bins).
    part = (rank, world): only that genomic chunk of the library -- its features (w.feat_index gives their
    rows in the whole matrix) and the reads that can overlap them."""
    w = Workload()
    if bins_kb:
        feats = [f for f in bin_features(bins_kb) if chroms is None or f[0] in chroms]
    else:
        genes = load_genes(chroms)
        feats = genes if n_features <= len(genes) else extend_features(genes, n_features, seed + 4)
        feats = feats[:n_features] if n_features < len(feats) else feats
    names = [c for c in HG38_CHROMS if chroms is None or c in chroms]
    gid_of = {c: i for i, c in enumerate(names)}
    w.feats, w.gid_of = feats, gid_of
    w.gid, w.beg, w.end = feature_arrays(feats, gid_of)
    sg, sb, se = merged_spans(feats, gid_of)
    w.spans = (sg, sb, se)
    w.n_rows_total = len(w.gid)
    if part is None:
        w.feat_index = np.arange(len(w.gid))
        w.dreads, w.cell_keys = ctx.synth_reads(n_reads, n_cells, sg, sb, se, seed=seed, want_seq=False)
        w.n_reads = n_reads
    else:
        idx, i0, n_loc = genomic_chunk(ctx, n_reads, seed, sg, sb, se, w.gid, w.beg, w.end, part)
        w.feat_index, w.first_read = idx, i0
        w.gid, w.beg, w.end = w.gid[idx], w.beg[idx], w.end[idx]
        w.dreads, w.cell_keys = ctx.synth_reads(max(1, n_loc), n_cells, sg, sb, se, seed=seed, want_seq=False,
                                                first_read=i0, total_reads=n_reads)
        w.n_reads = n_loc
    w.n_cells = n_cells
    w.params = engine.make_params(Conf(), 91, with_include=True)
    return w


def make_baf_workload(ctx, n_reads, n_cells, n_snps=200000, seed=7, chroms=None, part=None, snp_seed=None,
                      ref_error=None):
    """Config 2: chr1-22 reads, 5k cells, 200k phased het SNPs inside gene spans.
    ref_error not None: the bases away from the SNPs follow a pseudo-reference with this error rate (SNP discovery).
    part = (rank, world): the regions of that genomic chunk (w.feat_index: their rows in the whole matrices),
    the whole SNP table, and the reads that can overlap the chunk's regions."""
    w = Workload()
    auto = [c for c in HG38_CHROMS[:22] if chroms is None or c in chroms]
    genes = load_genes(set(auto))
    gid_of = {c: i for i, c in enumerate(auto)}
    w.feats, w.gid_of = genes, gid_of
    w.gid, w.beg, w.end = feature_arrays(genes, gid_of)
    sg, sb, se = merged_spans(genes, gid_of)
    rng = np.random.RandomState(seed + 1 if snp_seed is None else snp_seed)     # snp_seed: one SNP set for many batches
    # SNP positions uniform over the merged gene spans
    lens = (se - sb).astype(np.int64)
    cum = np.concatenate([[0], np.cumsum(lens)])
    u = np.sort(rng.randint(0, cum[-1], size=int(n_snps * 1.02)))
    u = np.unique(u)[:n_snps]
    si = np.searchsorted(cum, u, side="right") - 1
    w.snp_gid = sg[si].astype(np.int32)
    w.snp_pos = (sb[si] + (u - cum[si])).astype(np.int32)          # 0-based
    w.snp_ref = rng.randint(0, 4, size=len(u)).astype(np.uint8)
    w.snp_alt = ((w.snp_ref + rng.randint(1, 4, size=len(u))) % 4).astype(np.uint8)
    w.snp_ref_hap = rng.randint(0, 2, size=len(u)).astype(np.uint8)
    w.n_rows_total = len(w.gid)
    snps = (w.snp_gid, w.snp_pos, w.snp_ref, w.snp_alt, w.snp_ref_hap)
    if part is None:
        w.feat_index = np.arange(len(w.gid))
        w.dreads, w.cell_keys = ctx.synth_reads(n_reads, n_cells, sg, sb, se, seed=seed, want_seq=True, snps=snps,
                                                ref_error=ref_error)
        w.n_reads = n_reads
    else:
        idx, i0, n_loc = genomic_chunk(ctx, n_reads, seed, sg, sb, se, w.gid, w.beg, w.end, part)
        w.feat_index, w.first_read = idx, i0
        w.gid, w.beg, w.end = w.gid[idx], w.beg[idx], w.end[idx]
        w.dreads, w.cell_keys = ctx.synth_reads(max(1, n_loc), n_cells, sg, sb, se, seed=seed, want_seq=True,
                                                snps=snps, first_read=i0, total_reads=n_reads, ref_error=ref_error)
        w.n_reads = n_loc
    w.n_cells = n_cells
    w.contigs = auto
    w.params = engine.make_params(Conf(), 91, with_include=False)
    # region -> SNP lists (start0 <= pos0 < end0), hap table
    order = np.lexsort((w.snp_pos, w.snp_gid))
    sg_sorted, sp_sorted = w.snp_gid[order], w.snp_pos[order]
    key = sg_sorted.astype(np.int64) << 32 | sp_sorted.astype(np.int64)
    lo = np.searchsorted(key, w.gid.astype(np.int64) << 32 | w.beg.astype(np.int64))
    hi = np.searchsorted(key, w.gid.astype(np.int64) << 32 | w.end.astype(np.int64))
    hi = np.maximum(hi, lo)
    w.reg_ptr = np.concatenate([[0], np.cumsum(hi - lo)]).astype(np.int64)
    w.reg_snp = np.concatenate([order[a:b] for a, b in zip(lo, hi)] + [np.zeros(0, np.int64)]).astype(np.int32)
    hap = np.full((len(u), 8), 2, dtype=np.uint8)
    idx = np.arange(len(u))
    hap[idx, w.snp_ref] = w.snp_ref_hap
    hap[idx, w.snp_alt] = 1 - w.snp_ref_hap
    w.hap_of = hap
    return w
