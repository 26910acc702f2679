"""`xcltk basefc` on B200: per-feature, per-cell read / UMI counting (RDR total depth).

Same entry points, options, return codes and output files as the reference
(xcltk/rdr/fc/main.py: fc_main :61, fc_wrapper :142, fc_core :185, fc_run :270,
prepare_config :305); the per-feature pysam loop of fc_features (xcltk/rdr/fc/core.py:69-178)
is replaced by: decode BAMs -> records in HBM -> xg_basefc (CUDA) -> MTX / TSV text.
"""

import getopt
import os
import sys
import time
from logging import error, info
from logging import warning as warn

import numpy as np

from ... import engine, lib
from ...config import APP, VERSION
from ...utils.grange import Region
from ...utils.xlog import init_logging
from ...utils.zfile import zopen
from .config import Config

COMMAND = "basefc"


def usage(fp=sys.stdout, conf=None):
    d = conf
    rows = [
        "",
        "Version: %s" % VERSION,
        "Usage:   %s %s <options>" % (APP, COMMAND),
        "",
        "Options:",
        "  -s, --sam FILE         Comma separated indexed sam/bam/cram file.",
        "  -S, --samList FILE     A list file containing bam files, each per line.",
        "  -b, --barcode FILE     A plain file listing all effective cell barcode.",
        "  -R, --region FILE      A TSV file listing target regions. The first 4 columns shoud be:",
        "                         chrom, start, end (both 1-based and inclusive), name.",
        "  -i, --sampleList FILE  A list file containing sample IDs, each per line.",
        "  -I, --sampleIDs STR    Comma separated sample IDs.",
        "  -O, --outdir DIR       Output directory for sparse matrices.",
        "  -h, --help             Print this message and exit.",
        "",
        "Optional arguments:",
        "  -p, --ncores INT       Number of processes [%d]" % d.NPROC,
        "      --cellTAG STR      Tag for cell barcodes, set to None when using sample IDs [%s]" % d.CELL_TAG,
        "      --UMItag STR       Tag for UMI, set to None when reads only [%s]" % d.UMI_TAG,
        "  -D, --debug INT        Used by developer for debugging [%d]" % d.DEBUG,
        "",
        "Read filtering:",
        "  --inclFLAG INT          Required flags: skip reads with all mask bits unset [%d]" % d.INCL_FLAG,
        "  --exclFLAG INT          Filter flags: skip reads with any mask bits set [%d" % d.EXCL_FLAG_UMI,
        "                          (when use UMI) or %d (otherwise)]" % d.EXCL_FLAG_XUMI,
        "  --minLEN INT            Minimum mapped length for read filtering [%d]" % d.MIN_LEN,
        "  --minMAPQ INT           Minimum MAPQ for read filtering [%d]" % d.MIN_MAPQ,
        "  --minINCLUDE FLOAT|INT  Minimum fraction or length of included part within specific feature [%f]"
        % d.MIN_INCLUDE,
        "  --countORPHAN           If use, do not skip anomalous read pairs.",
        "",
        "B200 notes: input must be coordinate-sorted BAM (a .bai is used when present; SAM/CRAM are not decoded);",
        "  -p sets the host BGZF/BAM decode threads; counting runs on the GPU (no CPU fallback).",
        "",
    ]
    fp.write("\n".join(rows) + "\n")


_LONG = ["sam=", "samList=", "barcode=", "region=", "sampleList=", "sampleIDs=", "outdir=", "help",
         "ncores=", "cellTAG=", "UMItag=", "debug=", "inclFLAG=", "exclFLAG=", "minLEN=", "minMAPQ=",
         "minINCLUDE=", "countORPHAN"]


def fc_main(argv, conf=None):
    """Command-line interface; returns 0 on success, -1 otherwise (rdr/fc/main.py:61-139)."""
    if conf is None:
        conf = Config()
    if len(argv) <= 2:
        usage(sys.stdout, conf.defaults)
        sys.exit(0)
    conf.argv = argv.copy()
    init_logging(stream=sys.stderr)
    opts, _args = getopt.getopt(argv[2:], "-s:-S:-b:-R:-i:-I:-O:-h-p:-D:", _LONG)
    setters = {
        "-s": ("sam_fn", str), "--sam": ("sam_fn", str),
        "-S": ("sam_list_fn", str), "--samlist": ("sam_list_fn", str),
        "-b": ("barcode_fn", str), "--barcode": ("barcode_fn", str),
        "-R": ("region_fn", str), "--region": ("region_fn", str),
        "-i": ("sample_id_fn", str), "--samplelist": ("sample_id_fn", str),
        "-I": ("sample_id_str", str), "--sampleids": ("sample_id_str", str),
        "-O": ("out_dir", str), "--outdir": ("out_dir", str),
        "-p": ("nproc", int), "--ncores": ("nproc", int),
        "--celltag": ("cell_tag", str), "--umitag": ("umi_tag", str),
        "-D": ("debug", int), "--debug": ("debug", int),
        "--inclflag": ("incl_flag", int), "--exclflag": ("excl_flag", int),
        "--minlen": ("min_len", int), "--minmapq": ("min_mapq", float),
        "--mininclude": ("min_include", lambda v: float(v) if "." in v else int(v)),
    }
    for op, val in opts:
        if len(op) > 2:
            op = op.lower()          # long options are case-insensitive (main.py:107-108)
        if op in ("-h", "--help"):
            usage(sys.stdout, conf.defaults)
            sys.exit(0)
        elif op == "--countorphan":
            conf.no_orphan = False
        elif op in setters:
            attr, conv = setters[op]
            setattr(conf, attr, conv(val))
        else:
            error("invalid option: '%s'." % op)
            return -1
    return fc_run(conf)


def fc_wrapper(sam_fn, barcode_fn, region_fn, out_dir, sam_list_fn=None, sample_ids=None,
               sample_id_fn=None, debug_level=0, ncores=1, cell_tag="CB", umi_tag="UB",
               output_all_reg=True, min_mapq=20, min_len=30, min_include=0.9, incl_flag=0,
               excl_flag=None, no_orphan=True):
    """Python API, signature of rdr/fc/main.py:142-156.  As in the reference, a caller-supplied
    `excl_flag` is ignored (main.py:177-178 only handles None): the default applies."""
    conf = Config()
    conf.sam_fn, conf.sam_list_fn = sam_fn, sam_list_fn
    conf.barcode_fn, conf.region_fn = barcode_fn, region_fn
    conf.sample_id_str, conf.sample_id_fn = sample_ids, sample_id_fn
    conf.out_dir, conf.debug = out_dir, debug_level
    conf.cell_tag, conf.umi_tag = cell_tag, umi_tag
    conf.nproc, conf.output_all_reg = ncores, output_all_reg
    conf.min_mapq, conf.min_len, conf.min_include = min_mapq, min_len, min_include
    conf.incl_flag, conf.no_orphan = incl_flag, no_orphan
    if excl_flag is None:
        conf.excl_flag = -1
    return fc_run(conf)


def load_region_from_txt(fn, sep="\t", verbose=False):
    """Header-less TSV: chrom, start, end (1-based inclusive), name (rdr/fc/utils.py:10-45).
    Returns a list of Region (end exclusive) or None when a line has < 4 columns."""
    func = "load_region_from_txt"
    if verbose:
        sys.stderr.write("[I::%s] start to load regions from file '%s' ...\n" % (func, fn))
    regs = []
    with zopen(fn, "rt") as fp:
        for nl, line in enumerate(fp, 1):
            parts = line.rstrip().split(sep)
            if len(parts) < 4:
                if verbose:
                    sys.stderr.write("[E::%s] too few columns of line %d.\n" % (func, nl))
                return None
            regs.append(Region(parts[0], int(parts[1]), int(parts[2]) + 1, parts[3]))
    return regs


def prepare_config(conf):
    """Validate options and derive the run configuration; 0 if ok, -1 otherwise.
    Checks, their order and the messages follow rdr/fc/main.py:305-431."""
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
            conf.barcodes = sorted(x.strip() for x in fp)      # columns = sorted barcodes
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
    conf.out_region_fn = os.path.join(conf.out_dir, conf.out_prefix + "features.tsv")
    conf.out_sample_fn = os.path.join(conf.out_dir, conf.out_prefix + "barcodes.tsv")
    conf.out_mtx_fn = os.path.join(conf.out_dir, conf.out_prefix + "matrix.mtx")

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

    with open(conf.out_sample_fn, "w") as fp:
        fp.write("".join(smp + "\n" for smp in conf.samples))

    if conf.excl_flag < 0:
        conf.excl_flag = conf.defaults.EXCL_FLAG_UMI if conf.use_umi() else conf.defaults.EXCL_FLAG_XUMI
    return 0


def feature_arrays(regs, gid_of):
    """0-based half-open [start-1, end) of every Region; gid -1 where fetch() would raise or
    be empty (unknown contig, start <= 0; utils/sam.py:105-118)."""
    gid = np.array([gid_of.get(r.chrom, -1) for r in regs], dtype=np.int32)
    beg = np.array([r.start - 1 for r in regs], dtype=np.int64)       # fetch(chrom, start-1, end)
    end = np.array([r.end - 1 for r in regs], dtype=np.int64)
    bad = (beg < 0) | (end <= beg) | (end > 2147483647)
    gid[bad] = -1
    beg[bad] = 0
    end[bad] = 0
    return gid, beg.astype(np.int32), end.astype(np.int32)


def count_features(conf, batch=None):
    """Device counting for conf.reg_list; returns (row, col, val) 0-based, sorted by (row, col).
    Replaces the pool of fc_features workers (rdr/fc/main.py:213-235, rdr/fc/core.py:69-148).
    With several GPUs (conf.n_gpus / $XCLTK_B200_GPUS) the features are cut into contiguous
    genomic chunks balanced by reads, one per GPU; rows are merged on the host (no collective)."""
    from ... import parallel
    regs = conf.reg_list
    n_dev = parallel.n_devices(getattr(conf, "n_gpus", None))
    own = batch is None
    if own:
        chroms = list(dict.fromkeys(r.chrom for r in regs))
        threads = engine.n_decode_threads(conf.nproc)
        if n_dev > 1:
            # one library cut into genomic chunks: every GPU decodes only the blocks of its chunk (+ halo) ...
            batch = engine.load_reads_sharded(conf.sam_fn_list, chroms, conf.cell_tag, conf.umi_tag, False,
                                              parallel.device_list(n_dev), [r.chrom for r in regs],
                                              [r.start - 1 for r in regs], [r.end - 1 for r in regs])
            if batch is None:      # ... or, when the files cannot be split, every GPU gets the whole batch
                batch = engine.load_reads_multi(conf.sam_fn_list, chroms, conf.cell_tag, conf.umi_tag, False,
                                                threads, devices=parallel.device_list(n_dev))
        else:
            req = engine.Request(chroms, [r.chrom for r in regs], [r.start - 1 for r in regs], [r.end - 1 for r in regs])
            batch = engine.load_reads(conf.sam_fn_list, req, conf.cell_tag, conf.umi_tag, False, threads, host_only=True)
    try:
        gid, beg, end = feature_arrays(regs, batch.gid_of)
        cell_keys = None
        if conf.use_barcodes():
            cell_keys = np.array([batch.keyspace.encode(b) for b in conf.barcodes], dtype=np.uint64)
        if isinstance(batch, engine.ShardedBatch):
            shards = batch.shards
            empty = (np.zeros(0, np.int32),) * 3

            def one(k):
                b, sh = batch.batches[k], shards[k]
                if b is None or len(sh) == 0:
                    return empty + (None,)
                params = engine.make_params(conf, b.stats["max_aln_len"], with_include=True)
                r, c, v, _ = b.ctx.basefc(b.dreads, gid[sh], beg[sh], end[sh], cell_keys, len(conf.samples), params)
                return np.array(r), np.array(c), np.array(v), b.ctx.timing()
            parts = parallel.run_on_devices(len(shards), one)
            row, col, val = parallel.merge_coo([p[:3] for p in parts], shards, len(regs))
            conf.last_timing = next((p[3] for p in parts if p[3] is not None), [0.0] * 16)
            conf.shard_sizes = [len(s) for s in shards]
        elif isinstance(batch, engine.MultiBatch):
            load, total = parallel.reads_before(gid, beg, batch.runs, batch.pos_of_run)
            shards = parallel.partition(gid, beg, load, total, len(batch.batches))

            def one(k):
                b, sh = batch.batches[k], shards[k]
                params = engine.make_params(conf, b.stats["max_aln_len"], with_include=True)
                r, c, v, _ = b.ctx.basefc(b.dreads, gid[sh], beg[sh], end[sh], cell_keys, len(conf.samples), params)
                return np.array(r), np.array(c), np.array(v), b.ctx.timing()
            parts = parallel.run_on_devices(len(shards), one)
            row, col, val = parallel.merge_coo([p[:3] for p in parts], shards, len(regs))
            conf.last_timing = parts[0][3]
            conf.shard_sizes = [len(s) for s in shards]
        else:
            params = engine.make_params(conf, batch.stats["max_aln_len"], with_include=True)
            # fc_core: rows as completed, packed -- 16 bits per entry for the UMI counts of barcoded data (small numbers),
            # column | count in 32 bits for read counts per sample
            seg = ("tiny" if conf.use_barcodes() and conf.use_umi() else "narrow") if getattr(conf, "row_segments", False) else False
            if batch.dreads is None:       # pinned host batch: H2D streamed under the kernels
                res = batch.ctx.basefc_host(batch.host, gid, beg, end, cell_keys, len(conf.samples), params,
                                            segments=seg)
            else:
                res = batch.ctx.basefc(batch.dreads, gid, beg, end, cell_keys, len(conf.samples), params,
                                       segments=seg)
            conf.last_timing = batch.ctx.timing()
            if seg:
                conf.last_stats = dict(batch.stats)
                conf.last_ctx = batch.ctx            # its staging area still holds the rows (device-side MTX text)
                return res
            row, col, val, _shape = res
        conf.last_stats = dict(batch.stats)
    finally:
        if own:
            batch.close()
    return row, col, val


def fc_core(conf):
    if prepare_config(conf) < 0:
        raise ValueError("errcode -2")
    info("program configuration:")
    conf.show(fp=sys.stderr, prefix="\t")

    regs = conf.reg_list
    conf.row_segments = True         # one GPU: rows in completion order, copied out under the kernels
    res = count_features(conf)

    # emit (rdr/fc/core.py:96-124): a feature gets an output row iff it has a non-zero
    # count or output_all_reg; rows are numbered over the emitted features, input order.
    n_reg = len(regs)
    if isinstance(res, lib.RowSegments):
        has = res.row_cnt > 0
    else:
        row, col, val = res
        row = np.asarray(row)        # CSR result: rows are expanded on the host
        has = np.zeros(n_reg, dtype=bool)
        has[row] = True
    emitted = np.ones(n_reg, dtype=bool) if conf.output_all_reg else has
    with open(conf.out_region_fn, "w") as fp:
        fp.write("".join("%s\t%d\t%d\t%s\n" % (r.chrom, r.start, r.end - 1, r.get_id())
                         for r, e in zip(regs, emitted) if e))
    if isinstance(res, lib.RowSegments):
        out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
        ctx = getattr(conf, "last_ctx", None)
        if ctx is not None and os.environ.get("XCLTK_B200_DEVICE_MTX", "1") not in ("0", "", "no", "false"):
            # merge_mtx on the device: the rows are still in the context's staging area
            ctx.basefc_write_mtx(conf.out_mtx_fn, out_row, int(np.count_nonzero(emitted)),
                                 engine.n_decode_threads(conf.nproc))
        else:
            lib.write_mtx_rows(conf.out_mtx_fn, res, out_row, int(np.count_nonzero(emitted)),
                               engine.n_decode_threads(conf.nproc))
    else:
        engine.write_mtx(conf.out_mtx_fn, n_reg, row, col, val, emitted, len(conf.samples),
                         engine.n_decode_threads(conf.nproc))
    info("[GPU] %d reads counted in %.2f ms of kernels." % (
        conf.last_stats["n_reads"], conf.last_timing[0]))


def fc_run(conf):
    ret = -1
    cmdline = None
    start_time = time.time()
    info("start time: %s." % time.strftime("%Y-%m-%d %H:%M:%S", time.localtime(start_time)))
    if conf.argv is not None:
        cmdline = " ".join(conf.argv)
        info("CMD: %s" % cmdline)
    try:
        ret = fc_core(conf)
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
