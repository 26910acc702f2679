"""Host-side plumbing shared by basefc and baf: BAM decode -> HBM, parameter packing, output.

Replaces the process pool of the reference (`multiprocessing.Pool` over feature chunks,
xcltk/rdr/fc/main.py:191-235, xcltk/baf/fc/main.py:156-211): one context per GPU, the decoded
read batch is uploaded once and every feature / SNP is evaluated against it on the device.
"""

import logging
import math
import os

import numpy as np

from . import lib
from .utils.sam import build_tid_maps

INT32_MAX = 2147483647


def min_mapq_int(min_mapq):
    """`read.mapq < conf.min_mapq` with a possibly float threshold (rdr/fc/main.py:126,
    core.py:47): for integer mapq, mapq < x  <=>  mapq < ceil(x)."""
    return int(math.ceil(min_mapq))


def include_threshold(min_include, max_aln_len):
    """Integer form of the include test (rdr/fc/core.py:160-165).

    Fraction mode iff 0 < min_include < 1: keep iff not (m / float(n) < min_include); the
    table gives, for every aligned length n, the smallest m that is kept, found with the
    reference's own float expression (m / float(n) is monotone in m, so bisection is exact).
    Otherwise length mode: keep iff not (m < min_include)  <=>  m >= ceil(min_include).
    Returns (table or None, min_len)."""
    if 0 < min_include < 1:
        tab = np.empty(max(1, max_aln_len) + 1, dtype=np.int32)
        tab[0] = INT32_MAX            # n == 0: the reference's frac is None (never reached with min_len >= 1)
        for n in range(1, len(tab)):
            lo, hi = 0, n + 1         # smallest m in [0, n+1) with not (m/float(n) < f); n+1 = none
            while lo < hi:
                mid = (lo + hi) // 2
                if mid / float(n) < min_include:
                    lo = mid + 1
                else:
                    hi = mid
            tab[n] = lo if lo <= n else INT32_MAX
        return tab, 0
    return None, int(math.ceil(min_include))


class ReadBatch(object):
    """Decoded reads of all BAMs resident on one GPU + what is needed to address them."""

    def __init__(self, ctx, dreads, keyspace, gid_of, stats):
        self.ctx, self.dreads, self.keyspace, self.gid_of, self.stats = ctx, dreads, keyspace, gid_of, stats

    def close(self):
        if self.dreads is not None:
            self.dreads.close()
            self.dreads = None
        host = getattr(self, "host", None)
        if host is not None:             # zero-copy batch: the pinned records were still in use
            host.close()
            self.host = None


_contexts = {}


def get_context(device=0):
    """One xg_ctx per device, created on first use.  Raises XgError without a GPU: the
    counting paths have no CPU fallback."""
    ctx = _contexts.get(device)
    if ctx is None:
        ctx = lib.Context(device)
        _contexts[device] = ctx
    return ctx


def device_decode_enabled():
    """The device decoder (BGZF inflate + BAM parse on the GPU) is tried first unless
    $XCLTK_B200_DEVICE_DECODE is 0; files it declines go through the host decoder."""
    return os.environ.get("XCLTK_B200_DEVICE_DECODE", "1") not in ("0", "", "no", "false")


def _device_decode(ctx, sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, keyspace=None, range_lists=None):
    """(dreads, stats) or None."""
    if not device_decode_enabled():
        return None
    res = ctx.decode_bams(sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, keyspace, range_lists=range_lists)
    if res is None:
        logging.getLogger(__name__).info("device decoder declined (%s); decoding on the host.",
                                         getattr(ctx, "decode_fallback_reason", "?"))
        return None
    dreads, seen = res
    i = dreads.info()
    return dreads, {"n_reads": i["n_reads"], "n_records_seen": seen, "max_aln_len": i["max_aln_len"],
                    "max_span": i["max_span"], "bytes": i["bytes"], "decoder": "device",
                    "bytes_read": getattr(dreads, "bytes_read", None), "range_lists": range_lists}


def index_ranges(sam_fn_list, gid_of, tid_maps, units):
    """Per BAM, the BGZF block ranges its .bai gives for the units (contig as in gid_of, or None; 0-based [beg, end)),
    or None to read the file whole: no index, or one that cannot be trusted (one warning).  A read that overlaps a
    unit lies in the index chunks of the unit's interval, so the ranges hold every read the counting can use."""
    unit_chrom, unit_beg, unit_end = units
    gid = np.array([gid_of.get(c, -1) if c is not None else -1 for c in unit_chrom], dtype=np.int64)
    beg = np.asarray(unit_beg, dtype=np.int64)
    end = np.asarray(unit_end, dtype=np.int64)
    out = []
    for fn, tmap in zip(sam_fn_list, tid_maps):
        tid_of_gid = np.full(len(gid_of) + 1, -1, dtype=np.int32)
        for t, g in enumerate(tmap):
            if g >= 0:
                tid_of_gid[g] = t
        idx = None
        try:
            idx = lib.BamIndex.open(fn)
            out.append(idx.ranges(tid_of_gid[gid], beg, end) if idx is not None else None)
        except lib.XgError as ex:
            logging.getLogger(__name__).warning("%s; reading '%s' whole.", ex, fn)
            out.append(None)
        finally:
            if idx is not None:
                idx.close()
    return out


class Request(list):
    """The distinct contigs a call counts on -- what the loaders take as `chroms` -- with the call's units: contig
    (or None: never fetched) and 0-based [beg, end) of every feature / region / SNP / window.  Being a list, it goes
    wherever a contig list goes; load_reads takes the units from it to seek with the BAM index."""

    def __init__(self, chroms, unit_chrom, unit_beg, unit_end):
        list.__init__(self, chroms)
        self.units = (unit_chrom, unit_beg, unit_end)


def load_reads(sam_fn_list, chroms, cell_tag, umi_tag, want_seq, n_threads=0, device=0, mapped=False,
               host_only=False):
    """Bring every BAM's reads to `device` as one batch.

    The device decoder is tried first (the compressed files cross PCIe, the batch is built in
    HBM); when it declines -- records crossing BGZF blocks, keys that need the intern table --
    the BAMs are decoded on the host (multi-threaded) and uploaded.
    chroms: distinct (already 'chr'-stripped) contig names the features / SNPs use; reads on
    other contigs can never be fetched by the reference and are dropped at decode time.
    When `chroms` is a Request, the device decoder reads only the blocks that the .bai of a BAM gives for its
    units (index_ranges); a BAM without a usable index is read whole.  The batch may then hold fewer reads and a
    smaller max_aln_len / max_span; every read that overlaps a unit is in it, in file order.
    Host decoder only -- mapped: keep the records in pinned host memory and copy only pos/end
    (baf pileup); host_only: no upload at all, the caller streams the batch with
    Context.basefc_host."""
    ctx = get_context(device)
    ks = lib.KeySpace()
    bam_refs = [lib.bam_references(fn) for fn in sam_fn_list]
    gid_of, tid_maps = build_tid_maps(bam_refs, list(chroms))
    range_lists = None
    units = getattr(chroms, "units", None)
    if units is not None and device_decode_enabled():
        range_lists = index_ranges(sam_fn_list, gid_of, tid_maps, units)
        if all(r is None for r in range_lists):
            range_lists = None
    dev = _device_decode(ctx, sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, ks, range_lists)
    if dev is not None:
        return ReadBatch(ctx, dev[0], ks, gid_of, dev[1])
    host = lib.decode_bams(sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, ks, n_threads)
    stats = {"n_reads": host.n, "n_records_seen": host.n_records_seen, "max_aln_len": host.max_aln_len,
             "max_span": host.max_span, "bytes": host.nbytes()}
    if mapped or host_only:
        batch = ReadBatch(ctx, None if host_only else ctx.map_reads(host), ks, gid_of, stats)
        batch.host = host
        return batch
    dreads = ctx.upload(host)
    host.close()
    return ReadBatch(ctx, dreads, ks, gid_of, stats)


class MultiBatch(object):
    """The decoded batch resident on several GPUs (one full copy each; the genomic sharding
    happens on the feature side, see parallel.py) + the tile starts used to balance shards."""

    def __init__(self, batches, runs, tile_pos):
        self.batches, self.runs, self._tile_pos = batches, runs, tile_pos
        b0 = batches[0]
        self.keyspace, self.gid_of, self.stats = b0.keyspace, b0.gid_of, b0.stats

    def pos_of_run(self, r):
        """(sorted start positions sampled once per tile, reads per sample) of run r."""
        return self._tile_pos[r], float(lib.XG_TILE)

    def close(self):
        for b in self.batches:
            b.close()


def _tile_pos(runs, tiles):
    tile_pos = {}
    for rec_beg, n_rec, run, first_pos, max_end in tiles:
        tile_pos.setdefault(run, []).append(first_pos)
    tile_pos = {r: np.asarray(v, dtype=np.int64) for r, v in tile_pos.items()}
    for r in range(len(runs)):
        tile_pos.setdefault(r, np.zeros(0, dtype=np.int64))
    return tile_pos


def load_reads_multi(sam_fn_list, chroms, cell_tag, umi_tag, want_seq, n_threads=0, devices=(0,)):
    """The batch on every device in `devices`: each GPU decodes the files itself (device
    decoder, one host thread per GPU), else they are decoded once on the host and uploaded."""
    from . import parallel
    ctxs = [get_context(d) for d in devices]
    ks = lib.KeySpace()
    bam_refs = [lib.bam_references(fn) for fn in sam_fn_list]
    gid_of, tid_maps = build_tid_maps(bam_refs, list(chroms))
    devs = parallel.run_on_devices(len(ctxs), lambda k: _device_decode(ctxs[k], sam_fn_list, tid_maps, cell_tag,
                                                                       umi_tag, want_seq, ks))
    if all(d is not None for d in devs):
        runs, tiles = devs[0][0].index()
        return MultiBatch([ReadBatch(c, d[0], ks, gid_of, d[1]) for c, d in zip(ctxs, devs)], runs, _tile_pos(runs, tiles))
    for d in devs:
        if d is not None:
            d[0].close()
    host = lib.decode_bams(sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, ks, n_threads)
    stats = {"n_reads": host.n, "n_records_seen": host.n_records_seen, "max_aln_len": host.max_aln_len,
             "max_span": host.max_span, "bytes": host.nbytes()}
    runs = list(host.runs)
    tile_pos = _tile_pos(runs, host.tiles())
    try:
        dreads = parallel.run_on_devices(len(ctxs), lambda k: ctxs[k].upload(host))
    finally:
        host.close()
    return MultiBatch([ReadBatch(c, d, ks, gid_of, stats) for c, d in zip(ctxs, dreads)], runs, tile_pos)


class ShardedBatch(object):
    """One library cut into contiguous genomic chunks, one per GPU: batches[k] holds only the records of chunk k
    (+ halo), shards[k] the indices of the units (features / regions) counted there."""

    def __init__(self, batches, shards, keyspace, gid_of, stats):
        self.batches, self.shards = batches, shards
        self.keyspace, self.gid_of, self.stats = keyspace, gid_of, stats

    def close(self):
        for b in self.batches:
            if b is not None:
                b.close()


_INF_KEY = (1 << 40, 0)


def load_reads_sharded(sam_fn_list, chroms, cell_tag, umi_tag, want_seq, devices, unit_chrom, unit_beg, unit_end,
                       span=1 << 20):
    """The north star's multi-GPU split for real files: the BAM is cut at BGZF block boundaries into len(devices)
    contiguous byte ranges; a unit (feature / region; 0-based [beg, end)) belongs to the chunk its start falls
    into; every GPU inflates and parses only the blocks that can hold reads overlapping its units -- its own
    range, extended by a halo of `span` bp to the left and to the end of its last unit to the right -- with the
    device decoder.  What pysam's fetch gets from the .bai index is read off the file itself: the offsets of the
    blocks (xg_bgzf_block_index) and the position of a block's first record (xg_bam_block_probe, binary search).
    The halo is verified afterwards: no read of the library may span more than `span` bp (else the cut is redone
    with the span that was seen).  Returns None when the files cannot be split this way (device decoder off,
    records not aligned to blocks, BAMs with different contig lists, too many BAMs): the caller then gives every
    GPU the whole batch (load_reads_multi)."""
    from . import parallel
    n_dev = len(devices)
    if not device_decode_enabled() or n_dev < 2 or len(sam_fn_list) > 8:
        return None
    ctxs = [get_context(d) for d in devices]
    ks = lib.KeySpace()
    bam_refs = [lib.bam_references(fn) for fn in sam_fn_list]
    if any([r[0] for r in refs] != [r[0] for r in bam_refs[0]] for refs in bam_refs[1:]):
        return None
    gid_of, tid_maps = build_tid_maps(bam_refs, list(chroms))
    tid_of_gid = {int(g): t for t, g in enumerate(tid_maps[0]) if g >= 0}
    index = []
    for fn in sam_fn_list:
        off, first, aligned = lib.bgzf_block_index(fn)
        if not aligned:
            return None
        index.append((off, first))
    probe_cache = {}

    def block_key(b, i):
        """(tid, pos) of the first record of block i of BAM b; the unplaced tail and the end sort last"""
        off, _first = index[b]
        if i >= len(off) - 1:
            return _INF_KEY
        k = probe_cache.get((b, i))
        if k is None:
            tid, pos = lib.bam_block_probe(sam_fn_list[b], off[i])
            k = probe_cache[(b, i)] = _INF_KEY if tid < 0 else (tid, pos)
        return k

    def first_block_with(b, key, strictly_greater):
        """first block of BAM b whose first record is >= key (or > key)"""
        off, first = index[b]
        lo, hi = first, len(off) - 1
        while lo < hi:
            mid = (lo + hi) // 2
            k = block_key(b, mid)
            if (k > key) if strictly_greater else (k >= key):
                hi = mid
            else:
                lo = mid + 1
        return lo

    # cut keys from the largest BAM: equal shares of its bytes
    b0 = int(np.argmax([index[b][0][-1] for b in range(len(sam_fn_list))]))
    off0, first0 = index[b0]
    cuts = [(-1, -1)]
    for g in range(1, n_dev):
        i = int(np.searchsorted(off0, off0[first0] + (off0[-1] - off0[first0]) * g // n_dev))
        cuts.append(max(cuts[-1], block_key(b0, max(first0, min(i, len(off0) - 1)))))
    cuts.append(_INF_KEY)
    # units -> chunks by their start
    import bisect
    n_unit = len(unit_beg)
    keys = []
    shards = [[] for _ in range(n_dev)]
    for u in range(n_unit):
        g = gid_of.get(unit_chrom[u], -1)
        t = tid_of_gid.get(g, -1) if unit_end[u] > unit_beg[u] >= 0 else -1
        keys.append((t, int(unit_beg[u])))
        shards[0 if t < 0 else max(0, bisect.bisect_right(cuts, (t, int(unit_beg[u]))) - 1)].append(u)
    shards = [np.array(s, dtype=np.int64) for s in shards]

    def decode_with(span_bp):
        ranges = []
        for k in range(n_dev):
            lo_key, hi_key = cuts[k], cuts[k + 1]
            live = [u for u in shards[k] if keys[u][0] >= 0]
            if live:
                t_min, s_min = min(keys[u] for u in live)
                lo_key = min(lo_key, (t_min, max(0, s_min - span_bp)))
                hi_key = max(hi_key, max((keys[u][0], int(unit_end[u])) for u in live))
            per_bam = []
            for b in range(len(sam_fn_list)):
                off, first = index[b]
                # the block before the first one that begins at or after lo_key: records with key == lo_key may sit
                # at the end of that block (a run of equal starts crosses block boundaries), and none in earlier ones
                i_lo = max(first, first_block_with(b, lo_key, False) - 1)
                i_hi = first_block_with(b, hi_key, False)
                per_bam.append((int(off[i_lo]), int(off[max(i_lo, i_hi)])))
            ranges.append(per_bam)

        def one(k):
            if all(hi <= lo for lo, hi in ranges[k]):
                return None
            return _device_decode_range(ctxs[k], sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, ks, ranges[k])
        return parallel.run_on_devices(n_dev, one), ranges

    for attempt in range(2):
        devs, ranges = decode_with(span)
        if any(d is False for d in devs):           # the device decoder declined
            for d in devs:
                if d:
                    d[0].close()
            return None
        seen_span = max([d[1]["max_span"] for d in devs if d] or [0])
        if seen_span <= span:
            break
        for d in devs:
            if d:
                d[0].close()
        span = int(seen_span)
    else:
        return None
    batches = [ReadBatch(c, d[0], ks, gid_of, d[1]) if d else None for c, d in zip(ctxs, devs)]     # None: empty chunk
    live = [b for b in batches if b is not None]
    stats = {"n_reads": sum(b.stats["n_reads"] for b in live),
             "n_records_seen": sum(b.stats["n_records_seen"] for b in live),
             "max_aln_len": max([b.stats["max_aln_len"] for b in live] or [0]),
             "max_span": max([b.stats["max_span"] for b in live] or [0]),
             "bytes": sum(b.stats["bytes"] for b in live), "decoder": "device, sharded",
             "byte_ranges": ranges, "halo_bp": span,
             # chunk k holds the records whose start (tid, pos) lies in [cuts[k], cuts[k + 1]); tid_map: tid -> gid
             "cuts": cuts, "tid_map": list(tid_maps[0])}
    return ShardedBatch(batches, shards, ks, gid_of, stats)


def _device_decode_range(ctx, sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, keyspace, ranges):
    """(dreads, stats), or False when the device decoder declines."""
    res = ctx.decode_bams(sam_fn_list, tid_maps, cell_tag, umi_tag, want_seq, keyspace, ranges=ranges)
    if res is None:
        return False
    dreads, seen = res
    i = dreads.info()
    return dreads, {"n_reads": i["n_reads"], "n_records_seen": seen, "max_aln_len": i["max_aln_len"],
                    "max_span": i["max_span"], "bytes": i["bytes"], "decoder": "device"}


def make_params(conf, max_aln_len, with_include):
    tab, incl_len = (None, 0)
    if with_include:
        tab, incl_len = include_threshold(conf.min_include, max_aln_len)
    return lib.ParamsBox(min_mapq_int(conf.min_mapq), conf.min_len, conf.incl_flag, conf.excl_flag,
                         conf.no_orphan, conf.use_barcodes(), conf.use_umi(), tab, incl_len)


def write_mtx(path, n_rows_in, row, col, val, emitted, n_cols, n_threads=0):
    """MatrixMarket text exactly as merge_mtx writes it (rdr/fc/utils.py:65-67,80-86): header,
    `%%`, `nrow\tncol\tnnz`, then 1-based `row\tcol\tval` lines with the rows renumbered over
    the emitted features.  (row, col, val): 0-based, sorted by (row, col); emitted: bool per
    input row.  Formatting is done by the library's multi-threaded writer."""
    row = np.asarray(row)
    counts = np.bincount(row, minlength=n_rows_in) if len(row) else np.zeros(n_rows_in, dtype=np.int64)
    row_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    out_row = np.where(emitted, np.cumsum(emitted), 0).astype(np.int32)
    lib.write_mtx(path, row_ptr, out_row, int(np.count_nonzero(emitted)), n_cols, col, val, n_threads)


def n_decode_threads(nproc):
    n = int(nproc) if nproc else 1
    return max(1, min(n, os.cpu_count() or 1))
