"""baf feature-level allele counting on B200 (AD / DP / OTH matrices at phased het SNPs).

Same entry points, arguments, return codes and output files as the reference
(xcltk/baf/fc/main.py: afc_wrapper :32, afc_core :81, afc_run :262, prepare_config :298);
the per-SNP pysam pileup of fc_features / fc_fet1 / plp_snp (xcltk/baf/fc/core.py:42-247) is
replaced by: decode BAMs (with sequences) -> HBM -> xg_baf_pileup -> SNP filter (host, exact
float compare) -> xg_baf_count -> MTX / TSV text.
"""

import os
import sys
import time
from logging import debug, error, info
from logging import warning as warn

import numpy as np

from ... import engine
from ...utils.zfile import zopen
from ...utils.csp_io import load_data as csp_load_data
from ...utils.grange import format_chrom
from .config import Config
from .phasing import reg_local_phasing
from .utils import load_region_from_txt, load_snp_from_tsv, load_snp_from_vcf

BASES = "ACGTN"
BASE_IDX = {"A": 0, "C": 1, "G": 2, "T": 3, "N": 4}      # MCount.base_idx, baf/fc/mcount.py:178


def afc_wrapper(sam_fn, barcode_fn, region_fn, phased_snp_fn, out_dir, sam_list_fn=None,
                sample_ids=None, sample_id_fn=None, debug_level=0, ncores=1, cellsnp_dir=None,
                ref_cell_fn=None, cell_tag="CB", umi_tag="UB", min_count=1, min_maf=0,
                output_all_reg=False, no_dup_hap=True, min_mapq=20, min_len=30, incl_flag=0,
                excl_flag=None, no_orphan=True):
    """Python API, signature of baf/fc/main.py:32-47."""
    conf = Config()
    conf.sam_fn, conf.sam_list_fn = sam_fn, sam_list_fn
    conf.barcode_fn, conf.region_fn, conf.snp_fn = barcode_fn, region_fn, phased_snp_fn
    conf.sample_id_str, conf.sample_id_fn = sample_ids, sample_id_fn
    conf.out_dir, conf.debug = out_dir, debug_level
    conf.cellsnp_dir, conf.ref_cell_fn = cellsnp_dir, ref_cell_fn
    conf.cell_tag, conf.umi_tag = cell_tag, umi_tag
    conf.nproc = ncores
    conf.min_count, conf.min_maf = min_count, min_maf
    conf.output_all_reg, conf.no_dup_hap = output_all_reg, no_dup_hap
    conf.min_mapq, conf.min_len = min_mapq, min_len
    conf.incl_flag = incl_flag
    conf.excl_flag = -1 if excl_flag is None else excl_flag
    conf.no_orphan = no_orphan
    return afc_run(conf)


def prepare_samples(conf):
    """BAM list and columns (baf/fc/main.py:298-357): conf.sam_fn_list, conf.barcodes (sorted) or conf.sample_ids,
    conf.samples; then the output directory.  0 if ok, -1 otherwise."""
    if conf.sam_fn:
        if conf.sam_list_fn:
            error("should not specify 'sam_fn' and 'sam_list_fn' together.")
            return -1
        conf.sam_fn_list = conf.sam_fn.split(",")
    else:
        if not conf.sam_list_fn:
            error("one of 'sam_fn' and 'sam_list_fn' should be specified.")
            return -1
        with open(conf.sam_list_fn, "r") as fp:
            conf.sam_fn_list = [x.rstrip() for x in fp.readlines()]
    for fn in conf.sam_fn_list:
        if not os.path.isfile(fn):
            error("sam file '%s' does not exist." % fn)
            return -1

    if conf.barcode_fn:
        conf.sample_ids = None
        if conf.sample_id_str or conf.sample_id_fn:
            error("should not specify barcodes and sample IDs together.")
            return -1
        if not os.path.isfile(conf.barcode_fn):
            error("barcode file '%s' does not exist." % conf.barcode_fn)
            return -1
        with zopen(conf.barcode_fn, "rt") as fp:
            conf.barcodes = sorted(x.strip() for x in fp)
        if len(set(conf.barcodes)) != len(conf.barcodes):
            error("duplicate barcodes!")
            return -1
    else:
        conf.barcodes = None
        if conf.sample_id_str and conf.sample_id_fn:
            error("should not specify 'sample_id_str' and 'sample_fn' together.")
            return -1
        elif conf.sample_id_str:
            conf.sample_ids = conf.sample_id_str.split(",")
        elif conf.sample_id_fn:
            with zopen(conf.sample_id_fn, "rt") as fp:
                conf.sample_ids = [x.strip() for x in fp]
        else:
            warn("use default sample IDs ...")
            conf.sample_ids = ["Sample%d" % i for i in range(len(conf.sam_fn_list))]
        if len(conf.sample_ids) != len(conf.sam_fn_list):
            error("numbers of sam files and sample IDs are different.")
            return -1
    conf.samples = conf.barcodes if conf.barcodes else conf.sample_ids

    if not conf.out_dir:
        error("out dir needed!")
        return -1
    if not os.path.isdir(conf.out_dir):
        os.mkdir(conf.out_dir)
    return 0


def prepare_tags(conf):
    """Cell / UMI tags ('None' / 'Auto') and the default exclude flag (baf/fc/main.py:467-495).  0 if ok, -1
    otherwise."""
    if conf.cell_tag and conf.cell_tag.upper() == "NONE":
        conf.cell_tag = None
    if (not conf.cell_tag) != (not conf.barcodes):
        error("should not specify cell_tag or barcodes alone.")
        return -1
    if conf.umi_tag:
        if conf.umi_tag.upper() == "AUTO":
            conf.umi_tag = None if conf.barcodes is None else conf.defaults.UMI_TAG_BC
        elif conf.umi_tag.upper() == "NONE":
            conf.umi_tag = None
    if conf.excl_flag < 0:
        conf.excl_flag = conf.defaults.EXCL_FLAG_UMI if conf.use_umi() else conf.defaults.EXCL_FLAG_XUMI
    return 0


def prepare_config(conf):
    """Validate options, load regions / SNPs; 0 if ok, -1 otherwise (baf/fc/main.py:298-495)."""
    if prepare_samples(conf) < 0:
        return -1
    pre = os.path.join(conf.out_dir, conf.out_prefix)
    conf.out_region_fn, conf.out_sample_fn = pre + "region.tsv", pre + "samples.tsv"
    conf.out_ad_fn, conf.out_dp_fn, conf.out_oth_fn = pre + "AD.mtx", pre + "DP.mtx", pre + "OTH.mtx"

    if not conf.region_fn:
        error("region file needed!")
        return -1
    if not os.path.isfile(conf.region_fn):
        error("region file '%s' does not exist." % conf.region_fn)
        return -1
    conf.reg_list = load_region_from_txt(conf.region_fn, verbose=True)
    if not conf.reg_list:
        error("failed to load region file.")
        return -1
    info("count %d regions in %d single cells." % (len(conf.reg_list), len(conf.samples)))

    if not conf.snp_fn:
        error("SNP file needed!")
        return -1
    if not os.path.isfile(conf.snp_fn):
        error("snp file '%s' does not exist." % conf.snp_fn)
        return -1
    if conf.snp_fn.endswith((".vcf", ".vcf.gz", ".vcf.bgz")):
        conf.snp_set = load_snp_from_vcf(conf.snp_fn, verbose=True)
    else:
        conf.snp_set = load_snp_from_tsv(conf.snp_fn, verbose=True)
    if not conf.snp_set or conf.snp_set.get_n() <= 0:
        error("failed to load snp file.")
        return -1
    info("%d SNPs loaded." % conf.snp_set.get_n())

    # cellsnp-lite counts for the local-phasing pre-step (baf/fc/main.py:419-463; always given by `xcltk baf`,
    # baf/pipeline.py:352).  The reference's assertions are kept as assertions.
    if conf.cellsnp_dir is not None:
        assert os.path.exists(conf.cellsnp_dir)
        snp_data = csp_load_data(conf.cellsnp_dir)
        info("cellsnp SNP adata shape = %s." % str(snp_data.shape))
        assert len(conf.samples) == snp_data.shape[0]
        known = set(snp_data.cells.tolist())
        for cell in conf.samples:
            assert cell in known
        if snp_data.shape[1] != conf.snp_set.get_n():
            warn("n_snp: snp_adata=%d; snp_set=%d!" % (snp_data.shape[1], conf.snp_set.get_n()))
            assert snp_data.shape[1] >= conf.snp_set.get_n()
        idx_lst = []                       # SNPs that are still in the phased set
        for i in range(snp_data.shape[1]):
            if conf.snp_set.fetch(snp_data.chrom[i], int(snp_data.pos[i]), int(snp_data.pos[i]) + 1):
                idx_lst.append(i)
            elif conf.debug > 0:
                warn("SNP '%s:%d' was filtered before!" % (snp_data.chrom[i], snp_data.pos[i]))
        if len(idx_lst) < snp_data.shape[1]:
            snp_data = snp_data.subset_snps(idx_lst)
            info("SNP adata shape after subset: %s." % str(snp_data.shape))
        conf.snp_adata = snp_data
    if conf.ref_cell_fn is not None:
        assert os.path.exists(conf.ref_cell_fn)
        conf.ref_cells = np.atleast_1d(np.genfromtxt(conf.ref_cell_fn, dtype="str", delimiter="\t"))
        assert len(conf.ref_cells) <= len(conf.samples)
        for cell in conf.ref_cells:
            assert cell in conf.samples

    if prepare_tags(conf) < 0:
        return -1
    with open(conf.out_sample_fn, "w") as fp:
        fp.write("".join(smp + "\n" for smp in conf.samples))
    return 0


def snp_filter(conf, snps, totals):
    """plp_snp's SNP filter (baf/fc/core.py:238-246) from the five bucket totals: skip a SNP iff
    `snp_cnt < min_count` or `min(ref_cnt, alt_cnt) < snp_cnt * min_maf`.  Vectorised with the
    reference's own arithmetic: the counts are < 2^53, so int64 -> float64 is exact and
    `int < int * float` / `int < float` give what Python's mixed comparisons give."""
    n = len(snps)
    if n == 0:
        return np.zeros(0, dtype=np.uint8)
    t = np.asarray(totals, dtype=np.int64).reshape(n, 5)
    snp_cnt = t[:, 0] + t[:, 1] + t[:, 2] + t[:, 3] + t[:, 4]
    ref_i = np.fromiter((BASE_IDX[s.ref] for s in snps), dtype=np.int64, count=n)
    alt_i = np.fromiter((BASE_IDX[s.alt] for s in snps), dtype=np.int64, count=n)
    ar = np.arange(n)
    minor = np.minimum(t[ar, ref_i], t[ar, alt_i])
    skip = (snp_cnt < conf.min_count) | (minor < snp_cnt * conf.min_maf)
    return (~skip).astype(np.uint8)


def hap_table(snps):
    """hap_of[8*i + code]: region haplotype (0 / 1) of base code at SNP i, 2 = other allele
    (SNP.get_region_allele_index, gfeature.py:38-39; codes 0..4 = A,C,G,T,N, 5 = any other)."""
    hap = np.full((len(snps), 8), 2, dtype=np.uint8)
    for i, snp in enumerate(snps):
        for code, base in enumerate(BASES):
            h = snp.get_region_allele_index(base)
            if h in (0, 1):
                hap[i, code] = h
    return hap


def snp_arrays(conf, batch, snps):
    """Device arguments of a list of SNPs on one batch: contig ids, 0-based positions (fetch(chrom, pos-1, pos); a
    SNP that can never be fetched gets gid -1), the barcode keys and the read filters."""
    gid = np.array([batch.gid_of.get(s.chrom, -1) for s in snps], dtype=np.int32)
    pos0 = np.array([s.pos - 1 for s in snps], dtype=np.int64)
    bad = (pos0 < 0) | (pos0 >= 2147483647)
    gid[bad] = -1
    pos0[bad] = 0
    cell_keys = None
    if conf.use_barcodes():
        cell_keys = np.array([batch.keyspace.encode(b) for b in conf.barcodes], dtype=np.uint64)
    params = engine.make_params(conf, batch.stats["max_aln_len"], with_include=False)
    return gid, pos0.astype(np.int32), cell_keys, params


def allele_indices(snps):
    """MCount.base_idx of every SNP's REF and ALT (baf/fc/mcount.py:178)."""
    n = len(snps)
    return (np.fromiter((BASE_IDX[s.ref] for s in snps), dtype=np.uint8, count=n),
            np.fromiter((BASE_IDX[s.alt] for s in snps), dtype=np.uint8, count=n))


def _count_shard(conf, batch, regs, snps):
    """Pileup + count of `regs` (whose snp_list entries index `snps`) on one device."""
    local = {}                                   # SNPs of this shard, renumbered
    reg_ptr = np.zeros(len(regs) + 1, dtype=np.int64)
    reg_snp = []
    for r, reg in enumerate(regs):
        for s in (reg.snp_list or ()):
            reg_snp.append(local.setdefault(s.index, len(local)))
        reg_ptr[r + 1] = len(reg_snp)
    sub = [None] * len(local)
    for gi, li in local.items():
        sub[li] = snps[gi]
    gid, pos0, cell_keys, params = snp_arrays(conf, batch, sub)
    # pileup -> plp_snp's filter (on the device, IEEE double as Python evaluates it; `snp_filter` above is the same
    # test on the host, kept for the tests) -> region count, one library call
    ref_i, alt_i = allele_indices(sub)
    ctx = batch.ctx
    out = ctx.baf_fc(batch.dreads, gid, pos0, cell_keys, len(conf.samples), params, ref_i, alt_i,
                     conf.min_count, conf.min_maf, reg_ptr, np.array(reg_snp, dtype=np.int32), hap_table(sub),
                     conf.no_dup_hap)
    return out, [ctx.timing()], None


def shard_units(conf, chroms, unit_chrom, unit_beg, unit_end, run, batch=None):
    """Device work on independent units (regions, single SNPs, genomic windows) with one read batch per GPU.
    unit_chrom / unit_beg / unit_end: contig (None: never fetched) and 0-based [beg, end) of every unit; run(batch,
    idx) works on the units `idx` of one batch.  With several GPUs the units are cut into contiguous genomic chunks,
    no collective.  Returns ([(idx, run(batch, idx), or None for a chunk without reads or units)], sharded)."""
    from ... import parallel
    n_unit = len(unit_beg)
    n_dev = parallel.n_devices(getattr(conf, "n_gpus", None))
    own = batch is None
    if own:
        threads = engine.n_decode_threads(conf.nproc)
        if n_dev > 1:
            batch = engine.load_reads_sharded(conf.sam_fn_list, chroms, conf.cell_tag, conf.umi_tag, True,
                                              parallel.device_list(n_dev), unit_chrom, unit_beg, unit_end)
            if batch is None:
                batch = engine.load_reads_multi(conf.sam_fn_list, chroms, conf.cell_tag, conf.umi_tag, True,
                                                threads, devices=parallel.device_list(n_dev))
        else:
            batch = engine.load_reads(conf.sam_fn_list, engine.Request(chroms, unit_chrom, unit_beg, unit_end),
                                      conf.cell_tag, conf.umi_tag, True, threads, mapped=True)
    try:
        if isinstance(batch, (engine.ShardedBatch, engine.MultiBatch)):
            if isinstance(batch, engine.ShardedBatch):
                shards = batch.shards
            else:
                gid = np.array([batch.gid_of.get(c, -1) if c is not None else -1 for c in unit_chrom], dtype=np.int32)
                load, total = parallel.reads_before(gid, np.asarray(unit_beg, dtype=np.int64), batch.runs,
                                                    batch.pos_of_run)
                shards = parallel.partition(gid, np.asarray(unit_beg, dtype=np.int64), load, total,
                                            len(batch.batches))

            def one(k):
                b = batch.batches[k]
                if b is None or len(shards[k]) == 0:
                    return None
                return run(b, shards[k])
            res = list(zip(shards, parallel.run_on_devices(len(shards), one))), True
        else:
            idx = np.arange(n_unit, dtype=np.int64)
            res = [(idx, run(batch, idx))], False
        conf.last_stats = dict(batch.stats)
    finally:
        if own:
            batch.close()
    return res


def count_units(conf, chroms, unit_chrom, unit_beg, unit_end, count, batch=None):
    """Device counting of independent units (regions, or single SNPs) with one read batch per GPU (shard_units).
    count(batch, idx) -> ((ad, dp, oth), timings, per_unit) counts the units `idx` on one batch, the rows of its
    matrices indexing idx, per_unit an array over idx or None.  Returns the three (row, col, val, shape) tuples in
    unit order and the [(idx, per_unit)] of the shards."""
    from ... import parallel
    n_unit = len(unit_beg)
    shape = (n_unit, len(conf.samples))
    res, sharded = shard_units(conf, chroms, unit_chrom, unit_beg, unit_end, count, batch)
    if not sharded:
        idx, (out, conf.last_timing, pu) = res[0]
        return out, ([] if pu is None else [(idx, pu)])
    z = np.zeros(0, np.int32)
    shards = [idx for idx, _ in res]
    parts = [p if p is not None else (((z, z, z, shape),) * 3, [[0.0] * 16, [0.0] * 16], None) for _, p in res]
    out = []
    for w in range(3):
        r, c, v = parallel.merge_coo([[np.array(x) for x in p[0][w][:3]] for p in parts], shards, n_unit)
        out.append((r, c, v, shape))
    conf.last_timing = parts[0][1]
    per_unit = [(idx, p[2]) for idx, p in zip(shards, parts) if p[2] is not None]
    return tuple(out), per_unit


def count_regions(conf, regs, batch=None):
    """Device counting; returns three (row, col, val, shape) tuples (AD, DP, OTH), rows index
    `regs`.  With several GPUs the regions are cut into contiguous genomic chunks (their SNPs
    follow them; a SNP shared by regions of two chunks is piled up on both), no collective."""
    snps = conf.snp_set.snps
    chroms = list(dict.fromkeys([s.chrom for s in snps]))
    out, _ = count_units(conf, chroms, [r.chrom if r.snp_list else None for r in regs], [r.start - 1 for r in regs],
                         [r.end - 1 for r in regs], lambda b, idx: _count_shard(conf, b, [regs[i] for i in idx], snps),
                         batch)
    return out


def afc_core(conf):
    if prepare_config(conf) < 0:
        raise ValueError("errcode -2")
    info("program configuration:")
    conf.show(fp=sys.stderr, prefix="\t")

    # SNPs of each region: start <= pos < end, sorted by pos (baf/fc/main.py:88-104)
    with_snps = []
    for reg in conf.reg_list:
        snp_list = conf.snp_set.fetch(reg.chrom, reg.start, reg.end)
        if snp_list:
            reg.snp_list = snp_list
            with_snps.append(reg)
        elif conf.debug > 2:
            debug("region '%s': no SNP fetched." % reg.name)
    info("#regions: total=%d; with_snps=%d." % (len(conf.reg_list), len(with_snps)))
    if not conf.output_all_reg:
        conf.reg_list = with_snps
    # local phasing inside long regions (baf/fc/main.py:107-149): host numpy EM on the cellsnp-lite counts; it
    # may drop unexpressed SNPs from a region's list and swap the haplotype indices of (shared) SNP objects.
    # The device gets the lists and haplotype tables as they are afterwards.
    n_rlp = n_rlp_failed = n_slp = n_slp_flipped = 0
    if conf.use_local_phasing():
        data = conf.snp_adata
        if conf.ref_cells is not None:
            data = data.subset_cells(~np.isin(data.cells.astype(str), np.asarray(conf.ref_cells, dtype=str)))
        chrom = np.array([format_chrom(c) for c in data.chrom], dtype=object)
        for reg in conf.reg_list:
            if reg.end - reg.start < conf.rlp_min_len:
                continue
            if reg.snp_list is None or len(reg.snp_list) < max(1, conf.rlp_min_n_snps):
                continue
            if reg.snp_list[-1].pos - reg.snp_list[0].pos + 1 < conf.rlp_min_gap:
                continue
            if conf.debug > 2:
                debug("region '%s': do local phasing ..." % reg.name)
            cols = np.nonzero((chrom == reg.chrom) & (data.pos >= reg.start) & (data.pos < reg.end))[0]
            reg, flip = reg_local_phasing(reg, data.AD[:, cols].toarray(), data.DP[:, cols].toarray())
            if flip is None:
                n_rlp_failed += 1
                if conf.debug > 1:
                    debug("region '%s': local phasing failed." % reg.name)
            else:
                if conf.debug > 1:
                    debug("region '%s': #SNPs - total=%d; flipped=%d" % (reg.name, len(reg.snp_list), np.sum(flip)))
                n_slp_flipped += np.sum(flip)
            n_slp += len(reg.snp_list)
            n_rlp += 1
        conf.snp_adata = conf.ref_cells = None
    info("#regions: total=%d; local_phasing=%d; local_phasing_failed=%d." % (len(conf.reg_list), n_rlp, n_rlp_failed))
    info("#SNPs: local_phasing=%d; local_phasing_flipped=%d." % (n_slp, n_slp_flipped))

    regs = conf.reg_list
    if len(regs) == 0:
        # the reference divides by the worker count min(nproc, 0) here (main.py:152-158)
        raise ZeroDivisionError("integer division or modulo by zero")

    (ad, dp, oth) = count_regions(conf, regs)

    # emit (baf/fc/core.py:70-122): a region with SNPs gets a row iff it has a DP or OTH
    # entry, or output_all_reg; SNP-less regions only with output_all_reg.
    n_reg = len(regs)
    has = np.zeros(n_reg, dtype=bool)
    has[np.asarray(dp[0])] = True
    has[np.asarray(oth[0])] = True
    emitted = np.ones(n_reg, dtype=bool) if conf.output_all_reg else has
    with open(conf.out_region_fn, "w") as fp:
        fp.write("".join("%s\t%d\t%d\t%s\n" % (r.chrom, r.start, r.end - 1, r.name)
                         for r, e in zip(regs, emitted) if e))
    for fn, (row, col, val, _shape) in ((conf.out_ad_fn, ad), (conf.out_dp_fn, dp), (conf.out_oth_fn, oth)):
        engine.write_mtx(fn, n_reg, row, col, val, emitted, len(conf.samples), engine.n_decode_threads(conf.nproc))


def afc_run(conf, core=afc_core):
    """Runs `core(conf)` with the reference's logging (baf/fc/main.py:262-295); 0, or -1 on ValueError."""
    ret = -1
    cmdline = None
    start_time = time.time()
    info("start time: %s." % time.strftime("%Y-%m-%d %H:%M:%S", time.localtime(start_time)))
    if conf.argv is not None:
        cmdline = " ".join(conf.argv)
        info("CMD: %s" % cmdline)
    try:
        ret = core(conf)
    except ValueError as e:
        error(str(e))
        error("Running program failed.")
        error("Quiting ...")
        ret = -1
    else:
        info("All Done!")
        ret = 0
    finally:
        if conf.argv is not None:
            info("CMD: %s" % cmdline)
        end_time = time.time()
        info("end time: %s" % time.strftime("%Y-%m-%d %H:%M:%S", time.localtime(end_time)))
        info("time spent: %.2fs" % (end_time - start_time, ))
    return ret
