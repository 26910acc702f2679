#!/usr/bin/env python
"""bench.py -- reads/sec counted (basefc + baf fc) on synthetic 10x-style batches.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR      (+ the matrices of the last timed step)

A step = one pass of both hot paths over one library:
  basefc on config C3 (10k cells, 300M reads, ~60k features: hg38 genes + seeded nested intervals)
  baf fc  on config C2 (5k cells, 50M reads chr1-22, 200k phased het SNPs)
`value` = reads counted / step time with the records already resident in HBM; `e2e` = the
same through the C-ABI with HOST (pinned) record buffers, H2D upload and D2H result copy
inside the timed region.
Multi-GPU (`--scaling strong`, the default): ONE library cut into N contiguous genomic chunks balanced by
reads, one per GPU -- its features / regions and the reads that can overlap them (halo included); disjoint
rows, no collective in the data path (NCCL carries the barrier, the timing maximum and the parity checksum).
The rows of all ranks are checked against the unsharded matrix (order-independent checksum, outside the timed
region).  `--scaling weak`: one whole library per GPU (round 1's line).
At N=1 the GPU's matrices are compared entry by entry with the CPU oracle's on the SAME batch; a mismatch
fails the run.  The reference arm times the CPU oracle (a C port of the reference's algorithm; the
reference itself is Python on pysam and cannot run on the box) on a bounded sample.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

C_BAR_NOMINAL = 1.43              # mean CIGAR ops per read of the synthetic mix (SURVEY.md 8d); measured per batch below


def matrix_checksum(row, col, val):
    """Order-independent, shard-additive checksum of sparse entries (wraps modulo 2^64)."""
    with np.errstate(over="ignore"):
        x = (np.asarray(row).astype(np.uint64) << np.uint64(32)) ^ np.asarray(col).astype(np.uint64)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
        return int((x * (np.asarray(val).astype(np.uint64) * np.uint64(2) + np.uint64(1))).sum(dtype=np.uint64))


DUMP_LIMIT = 64 * 10 ** 6         # bytes of all --dump-outputs files together
DUMP_ENTRIES = {"basefc": 1 << 21, "baf_ad": 1 << 17, "baf_dp": 1 << 17, "baf_oth": 1 << 17}


def dump_outputs(out_dir, mats):
    """mats = {name: (row, col, val, shape)}, entries sorted by (row, col).  Writes out_dir/<name>_row.npy, _col.npy,
    _val.npy (every entry, or an evenly spaced sample of DUMP_ENTRIES[name] entries when there are more),
    <name>_row_sum.npy (the total of every row, float64) and <name>_shape.npy (rows, cols, nnz): with the same
    arguments two builds can be compared output for output."""
    arrays = {}
    for name, (row, col, val, shape) in mats.items():
        row, col, val = (np.asarray(a) for a in (row, col, val))
        nnz, cap = len(val), DUMP_ENTRIES[name]
        arrays[name + "_shape"] = np.array([shape[0], shape[1], nnz], dtype=np.float64)
        arrays[name + "_row_sum"] = np.bincount(row, weights=val, minlength=shape[0]).astype(np.float64)
        idx = np.arange(nnz) if nnz <= cap else np.arange(cap, dtype=np.int64) * nnz // cap
        exact = max(shape[0], shape[1], int(val.max()) + 1 if nnz else 0) <= 1 << 24     # float32 holds them exactly
        for k, a in (("row", row), ("col", col), ("val", val)):
            arrays["%s_%s" % (name, k)] = a[idx].astype(np.float32 if exact else np.float64)
    total = sum(a.nbytes + 128 for a in arrays.values())      # + the .npy header
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes, more than %d" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as fp:
                return float(json.load(fp)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(local):
    """One process per GPU: run on the CPUs of the GPU's NUMA node, so that the pinned buffers
    this rank allocates (first touch) sit next to its PCIe root instead of across the socket link."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = None
        try:                                    # NVML does not see CUDA_VISIBLE_DEVICES: go by the PCI address
            import torch
            pr = torch.cuda.get_device_properties(local)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(
                ("%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        bind_to_gpu_numa_node(local)
    dist = None
    if world > 1:
        # stdout carries the one JSON line: NCCL's own banner / debug lines go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def barrier_sync(dist, local):
    import torch
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(local)


def max_over_ranks(dist, local, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device="cuda:%d" % local)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(dist, local, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device="cuda:%d" % local)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


class Batch(object):
    """One GPU's workload: device-resident records + the pinned host copy used by e2e."""

    def __init__(self, ctx, args, rank, world):
        from xcltk_b200 import workload
        self.ctx = ctx
        if args.scaling == "strong":
            part = (rank, world) if world > 1 else None
            seed = 7
        else:
            part, seed = None, 7 + 1000 * rank
        self.fc = workload.make_basefc_workload(ctx, args.reads, args.cells, args.features, seed=seed, part=part)
        self.baf = workload.make_baf_workload(ctx, args.baf_reads, args.baf_cells, args.snps, seed=seed + 1, part=part)
        self.n_reads = self.fc.n_reads + self.baf.n_reads          # records this GPU holds (halos included)
        # The two halves of a step are independent calls (xcltk's rdr and baf modules): unless --serial-calls, the baf
        # call is issued from a second host thread through a context (stream, scratch) of its own on the same GPU,
        # so that its host phases and short kernels run beside basefc's instead of after them.
        self.ctx_baf, self.pool = ctx, None
        if not args.serial_calls:
            from concurrent.futures import ThreadPoolExecutor
            from xcltk_b200 import lib
            self.ctx_baf = lib.Context(ctx.device)
            if not os.environ.get("BENCH_NO_PRIORITY"):      # its short kernels go first whenever both contexts wait for SMs
                self.ctx_baf.lib.xg_set_option(self.ctx_baf.h, b"stream_priority", 1)
            self.pool = ThreadPoolExecutor(1)

    # SNP filter of the baf half: min_count = 1, min_maf = 0 (the values xcltk baf passes, baf/pipeline.py:355)

    def step_device(self, checksum=False, keep=False):
        """keep: the result also carries what the two calls returned ("outputs")."""
        ctx, fc, bf = self.ctx, self.fc, self.baf
        launches = 0
        w0 = time.perf_counter()

        def baf_call():
            # pileup -> SNP filter (min_count 1, min_maf 0, on the device) -> region count: one library call
            t = time.perf_counter()
            out = self.ctx_baf.baf_fc(bf.dreads, bf.snp_gid, bf.snp_pos, bf.cell_keys, bf.n_cells, bf.params, bf.snp_ref,
                                      bf.snp_alt, 1, 0.0, bf.reg_ptr, bf.reg_snp, bf.hap_of, True)
            return out, self.ctx_baf.timing(), time.perf_counter() - t

        fut = self.pool.submit(baf_call) if self.pool else None
        # rows in completion order (what the Matrix-Market writer consumes): copied out under the kernels
        seg = ctx.basefc(fc.dreads, fc.gid, fc.beg, fc.end, fc.cell_keys, fc.n_cells, fc.params, segments="tiny")
        w1 = time.perf_counter()
        t_fc = ctx.timing()
        launches += int(t_fc[2])
        (ad, dp, oth), t_c, w_baf = fut.result() if fut else baf_call()
        w2 = time.perf_counter()
        t_p = t_c
        launches += int(t_c[2])
        chk = None
        if checksum:                 # rows numbered as in the whole matrix, so that the shards add up
            r, c, v = seg.to_sorted()
            chk = matrix_checksum(fc.feat_index[r], c, v)
            for k, m in enumerate((ad, dp, oth)):
                chk = (chk + matrix_checksum(bf.feat_index[m[0]] + (k + 1) * (1 << 24), m[1], m[2])) % (1 << 64)
        w4 = time.perf_counter()
        res = dict(nnz=seg.nnz, checksum=chk, wall_ms=[1e3 * (w1 - w0), 1e3 * w_baf, 1e3 * (w2 - w0), 1e3 * (w4 - w2)],
                   launches=launches, t_fc=t_fc, t_pileup=t_p, t_count=t_c, baf_nnz=len(ad[2]) + len(dp[2]) + len(oth[2]),
                   out_bytes=2 * seg.nnz + 16 * len(seg.over[0]) + 8 * (len(ad[2]) + len(dp[2]) + len(oth[2])))
        if keep:
            res["outputs"] = (seg, (ad, dp, oth))
        return res

    def make_host(self):
        self.h_fc = self.fc.dreads.download()         # pinned host record arrays
        self.h_baf = self.baf.dreads.download()

    def step_e2e(self):
        ctx, fc, bf = self.ctx, self.fc, self.baf
        seg = ctx.basefc_host(self.h_fc, fc.gid, fc.beg, fc.end, fc.cell_keys, fc.n_cells, fc.params, segments="tiny")
        h2d_fc = int(ctx.timing()[13])
        d_bf = ctx.map_reads(self.h_baf)          # zero-copy: 8 B/read over PCIe, rest on demand
        ad, dp, oth = ctx.baf_fc(d_bf, bf.snp_gid, bf.snp_pos, bf.cell_keys, bf.n_cells, bf.params, bf.snp_ref,
                                 bf.snp_alt, 1, 0.0, bf.reg_ptr, bf.reg_snp, bf.hap_of, True)
        ctx.timing_pairs = ctx.timing()[6]            # (read, SNP) pairs: records fetched on demand
        d_bf.close()
        return dict(h2d=h2d_fc + 8 * self.h_baf.n + 72 * int(self.ctx.timing_pairs),
                    d2h=2 * seg.nnz + 16 * len(seg.over[0]) + 8 * (len(ad[2]) + len(dp[2]) + len(oth[2])) +
                    12 * len(fc.gid) + 8 * (3 * (len(bf.reg_ptr) - 1) + 3))  # packed entries + row_beg/row_cnt | col + val + row_ptr

    def oracle_parity(self, n_threads):
        """The CPU oracle on this very batch (outside the timed region): its matrices against the GPU's,
        entry by entry; the oracle's wall time is the CPU baseline."""
        from oracle import oracle
        from xcltk_b200 import workload
        ctx, fc, bf = self.ctx, self.fc, self.baf
        conf = workload.Conf()
        conf_b = workload.Conf()
        conf_b.min_include = 0
        letters = "ACGT"
        ref_s, alt_s = "".join(letters[x] for x in bf.snp_ref), "".join(letters[x] for x in bf.snp_alt)
        t = time.perf_counter()
        o_fc = oracle.basefc(self.h_fc, fc.gid, fc.beg, fc.end, fc.cell_keys, fc.n_cells, oracle.params(conf), n_threads)
        t_fc = time.perf_counter() - t
        t = time.perf_counter()
        o_baf = oracle.baf(self.h_baf, bf.snp_gid, bf.snp_pos, ref_s, alt_s, bf.snp_ref_hap, 1 - bf.snp_ref_hap,
                           bf.reg_ptr, bf.reg_snp, bf.cell_keys, bf.n_cells, oracle.params(conf_b), 1, 0, True, n_threads)
        t_baf = time.perf_counter() - t
        seg = ctx.basefc(fc.dreads, fc.gid, fc.beg, fc.end, fc.cell_keys, fc.n_cells, fc.params, segments="tiny")
        g_fc = seg.to_sorted()
        ok_fc = all(np.array_equal(a, b) for a, b in zip(g_fc, o_fc))
        g_baf = ctx.baf_fc(bf.dreads, bf.snp_gid, bf.snp_pos, bf.cell_keys, bf.n_cells, bf.params, bf.snp_ref, bf.snp_alt,
                           1, 0.0, bf.reg_ptr, bf.reg_snp, bf.hap_of, True)
        ok_baf = all(np.array_equal(g[k], o[k]) for g, o in zip(g_baf, o_baf) for k in range(3))
        return dict(basefc=bool(ok_fc), baf=bool(ok_baf), nnz=int(len(o_fc[2])),
                    baf_nnz=int(sum(len(o[2]) for o in o_baf)),
                    against="oracle/xg_oracle.c on the same C3 + C2 batch, entry by entry"), t_fc + t_baf


# The reference's OWN Python path cannot travel to the GPU box (no /root/reference there): timed once in the build
# container (unmodified xcltk v0.5.2 on the pysam shim, 8 worker processes, basefc on the C1 golden: 1M reads in 41.9 s;
# `python oracle/make_golden.py c1_full` prints it) and quoted as a labelled constant next to the C port's live number.
REFERENCE_PYTHON = {"value": 2.39e4, "unit": "reads/s", "cores": 8, "kind": "constant, not timed in this run",
                    "what": "unmodified reference (Python, multiprocessing) on the pysam shim, basefc, C1 golden (1M reads, "
                            "500 barcodes, 33 472 features), build container"}


def cpu_sample(ctx, args, n_sample, n_threads):
    """A bounded sample of the basefc workload (same generator, fewer reads) for the CPU legs."""
    from xcltk_b200 import workload
    from oracle import oracle
    w = workload.make_basefc_workload(ctx, n_sample, args.cells, args.features, seed=99)
    host = w.dreads.download()
    conf = workload.Conf()
    par = oracle.params(conf)

    # ... and the baf half of the step (config 2), scaled with the basefc sample
    n_baf = max(1, int(round(args.baf_reads * (n_sample / float(args.reads)))))
    b = workload.make_baf_workload(ctx, n_baf, args.baf_cells, args.snps, seed=98)
    host_b = b.dreads.download()
    conf_b = workload.Conf()
    conf_b.min_include = 0
    par_b = oracle.params(conf_b)
    letters = "ACGT"
    ref_s, alt_s = "".join(letters[x] for x in b.snp_ref), "".join(letters[x] for x in b.snp_alt)

    def run():
        t = time.perf_counter()
        oracle.basefc(host, w.gid, w.beg, w.end, w.cell_keys, args.cells, par, n_threads)
        oracle.baf(host_b, b.snp_gid, b.snp_pos, ref_s, alt_s, b.snp_ref_hap, 1 - b.snp_ref_hap, b.reg_ptr, b.reg_snp,
                   b.cell_keys, args.baf_cells, par_b, 1, 0, True, n_threads)
        return time.perf_counter() - t
    run.n_reads = n_sample + n_baf
    return run, (host, host_b)


def file_legs(ctx, args):
    """The user's call, file to file: fc_wrapper(BAM, barcodes, features, out_dir) -> features.tsv, barcodes.tsv,
    matrix.mtx on disk (device decode + counting + Matrix-Market writer), on BAM files that hold exactly the records
    of a synthetic batch (xg_write_bam): config C1 at its shape (chr22, 1M reads, 500 barcodes, all 33 472 hg38 gene
    rows) and a slice of config C3 (10k cells, 60k features, --file-reads reads over the whole genome).  The
    matrix.mtx the call wrote must be, byte for byte, the text written from the CPU oracle's matrix of the same
    records (md5)."""
    import hashlib
    import shutil
    import tempfile
    from oracle import oracle
    from xcltk_b200 import lib, workload
    from xcltk_b200.rdr.fc.main import fc_wrapper
    n_thr = os.cpu_count() or 1
    conf = workload.Conf()
    out, host_dec, dev_dec = {}, None, None

    def md5(path):
        h = hashlib.md5()
        with open(path, "rb") as fp:
            for blk in iter(lambda: fp.read(1 << 24), b""):
                h.update(blk)
        return h.hexdigest()

    with tempfile.TemporaryDirectory() as td:
        free = shutil.disk_usage(td).free
        n_c3 = int(min(args.file_reads, max(2e6, (free - (4 << 30)) / 120.0)))       # ~90 B/read on disk + outputs
        for name, n_reads, n_cells, chroms, all_rows in (("C1", 1000000, 500, {"22"}, True),
                                                        ("C3_slice", n_c3, args.cells, None, False)):
            w = workload.make_basefc_workload(ctx, n_reads, n_cells, 33472 if all_rows else args.features, seed=17,
                                              chroms=chroms)
            host = w.dreads.download()
            names = [c for c in workload.HG38_CHROMS if chroms is None or c in chroms]
            contigs = [("chr" + c, workload.HG38_LEN[c]) for c in names]      # BAM says chr22, the features say 22
            bam = os.path.join(td, name + ".bam")
            t = time.perf_counter()
            lib.write_bam(bam, host, contigs, None, "CB", "UB", level=1, n_threads=n_thr)
            t_write = time.perf_counter() - t
            feats = workload.load_genes(None) if all_rows else w.feats
            gid, beg, end = workload.feature_arrays(feats, w.gid_of)
            ks = lib.KeySpace()
            barcodes = [ks.decode(int(k)) for k in w.cell_keys]
            bc_fn, ft_fn = os.path.join(td, name + ".barcodes.tsv"), os.path.join(td, name + ".features.tsv")
            with open(bc_fn, "w") as fp:
                fp.write("".join(b + "\n" for b in barcodes))
            with open(ft_fn, "w") as fp:
                fp.write("".join("%s\t%d\t%d\t%s\n" % f for f in feats))
            # expected text: the oracle's matrix of the same records through the Matrix-Market writer
            o_row, o_col, o_val = oracle.basefc(host, gid, beg, end, w.cell_keys, n_cells, oracle.params(conf), n_thr)
            exp_fn = os.path.join(td, name + ".expected.mtx")
            engine_write = __import__("xcltk_b200.engine", fromlist=["write_mtx"]).write_mtx
            engine_write(exp_fn, len(gid), o_row, o_col, o_val, np.ones(len(gid), dtype=bool), n_cells, n_thr)
            want = md5(exp_fn)
            best = None
            for k in range(3):            # (the page cache's write-back makes single calls jumpy: +/- 100 ms and more)
                out_dir = os.path.join(td, "%s.out%d" % (name, k))
                t = time.perf_counter()
                ret = fc_wrapper(bam, bc_fn, ft_fn, out_dir, ncores=n_thr)
                dt_f = time.perf_counter() - t
                if ret != 0:
                    raise RuntimeError("fc_wrapper returned %d" % ret)
                best = dt_f if best is None else min(best, dt_f)
            got = md5(os.path.join(out_dir, "matrix.mtx"))
            out[name] = {"reads_per_s": n_reads / best, "reads": n_reads, "call_ms": 1e3 * best,
                         "bam_bytes": os.path.getsize(bam), "mtx_bytes": os.path.getsize(os.path.join(out_dir, "matrix.mtx")),
                         "matrix_md5": got, "matches_oracle_text": bool(got == want), "bam_write_s": t_write,
                         "shape": "%d features x %d cells" % (len(gid), n_cells)}
            maps = [np.arange(len(contigs), dtype=np.int32)]
            if name == "C1":            # host decoder (the fallback for files the device decoder declines)
                t = time.perf_counter()
                hr = lib.decode_bams([bam], maps, "CB", "UB", False, lib.KeySpace(), n_thr)
                dt = time.perf_counter() - t
                host_dec = {"reads_per_s": hr.n / dt, "threads": n_thr, "sample_reads": hr.n, "file": "C1 BAM"}
                hr.close()
            else:                       # device decoder alone: file -> HBM-resident batch
                bestd = None
                for _ in range(3):
                    t = time.perf_counter()
                    res = ctx.decode_bams([bam], maps, "CB", "UB", False)
                    dt = time.perf_counter() - t
                    if res is None:
                        break
                    n_dev = res[0].n
                    res[0].close()
                    bestd = dt if bestd is None else min(bestd, dt)
                if bestd is not None:
                    tdv = ctx.timing()
                    dev_dec = {"reads_per_s": n_dev / bestd, "sample_reads": n_dev, "call_ms": 1e3 * bestd,
                               "stream_loop_ms": tdv[4], "extract_ms": tdv[3], "windows": int(tdv[5]), "file": "C3 slice BAM"}
                else:
                    dev_dec = {"declined": getattr(ctx, "decode_fallback_reason", "")}
            host.close()
            w.dreads.close()
            os.remove(bam)
        # ---- config C4 (SMART-seq): 384 per-cell BAMs, no cell / UMI tags: sample IDs, reads collapsed by query name
        n_bams, per_bam = 384, int(args.smartseq_reads)
        chroms4 = None
        names = list(workload.HG38_CHROMS)
        contigs = [(c, workload.HG38_LEN[c]) for c in names]
        paths = []
        t = time.perf_counter()
        w = workload.make_basefc_workload(ctx, per_bam, 40, 33472, seed=1000, chroms=chroms4)
        for b in range(n_bams):
            d = w.dreads if b == 0 else ctx.synth_reads(per_bam, 40, *w.spans, seed=1000 + b, want_seq=False)[0]
            host = d.download()
            p = os.path.join(td, "cell%03d.bam" % b)
            lib.write_bam(p, host, contigs, None, None, None, level=1, n_threads=n_thr, name_from_umi=True)
            paths.append(p)
            host.close()
            d.close()
        t_write = time.perf_counter() - t
        lst, ft_fn = os.path.join(td, "C4.lst"), os.path.join(td, "C4.features.tsv")
        with open(lst, "w") as fp:
            fp.write("".join(p + "\n" for p in paths))
        with open(ft_fn, "w") as fp:
            fp.write("".join("%s\t%d\t%d\t%s\n" % f for f in w.feats))
        ids = ",".join("well%03d" % b for b in range(n_bams))
        best = None
        for k in range(2):
            out_dir = os.path.join(td, "C4.out%d" % k)
            t = time.perf_counter()
            ret = fc_wrapper(None, None, ft_fn, out_dir, sam_list_fn=lst, sample_ids=ids, cell_tag=None, umi_tag=None,
                             ncores=n_thr)
            dt_f = time.perf_counter() - t
            if ret != 0:
                raise RuntimeError("fc_wrapper (C4) returned %d" % ret)
            best = dt_f if best is None else min(best, dt_f)
        # expected: the oracle on the host decoder's records of the same files (query names through the keyspace)
        ks = lib.KeySpace()
        maps = [np.arange(len(contigs), dtype=np.int32)] * n_bams
        hr = lib.decode_bams(paths, maps, None, None, False, ks, n_thr)
        gid, beg, end = workload.feature_arrays(w.feats, w.gid_of)
        conf4 = workload.Conf()
        conf4.excl_flag, conf4.cell_tag, conf4.umi_tag = 1796, None, None      # the no-UMI default (rdr/fc/main.py:425-429)
        conf4.use_barcodes = lambda: False
        conf4.use_umi = lambda: False
        o_row, o_col, o_val = oracle.basefc(hr, gid, beg, end, None, n_bams, oracle.params(conf4), n_thr)
        hr.close()
        exp_fn = os.path.join(td, "C4.expected.mtx")
        __import__("xcltk_b200.engine", fromlist=["write_mtx"]).write_mtx(
            exp_fn, len(gid), o_row, o_col, o_val, np.ones(len(gid), dtype=bool), n_bams, n_thr)
        got = md5(os.path.join(out_dir, "matrix.mtx"))
        out["C4_smartseq"] = {"reads_per_s": n_bams * per_bam / best, "reads": n_bams * per_bam, "bams": n_bams,
                              "call_ms": 1e3 * best, "matrix_md5": got, "matches_oracle_text": bool(got == md5(exp_fn)),
                              "nnz": int(len(o_val)), "bam_write_s": t_write,
                              "shape": "%d features x %d cells, sample IDs, query-name keys" % (len(gid), n_bams)}
    out["note"] = ("fc_wrapper(): BAM file -> features.tsv, barcodes.tsv, matrix.mtx on disk, best of 2-3; the BAMs hold "
                   "the records of device-generated batches (xg_write_bam, htslib block layout, level 1)")
    return out, host_dec, dev_dec


_JSON_FD = None


def claim_stdout():
    """stdout carries exactly one JSON line: keep a private handle on it and point fd 1 at stderr,
    so that nothing a library prints (NCCL's version banner, for one) can get in front of it."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=float, default=300e6, help="basefc reads per GPU (C3: 300M)")
    ap.add_argument("--cells", type=int, default=10000)
    ap.add_argument("--features", type=int, default=60000)
    ap.add_argument("--baf-reads", type=float, default=50e6, help="baf reads per GPU (C2)")
    ap.add_argument("--baf-cells", type=int, default=5000)
    ap.add_argument("--snps", type=int, default=200000)
    ap.add_argument("--cpu-sample", type=float, default=3e8, help="reads of the CPU legs (default: the whole C3 basefc batch)")
    ap.add_argument("--file-reads", type=float, default=6e7, help="reads of the C3 slice written to a BAM for the file-to-matrix leg")
    ap.add_argument("--smartseq-reads", type=float, default=5e4, help="reads per BAM of the 384-BAM SMART-seq leg (C4)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--serial-calls", action="store_true",
                    help="issue the baf call after the basefc call instead of beside it (second host thread + context)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: strong = one library cut into N genomic chunks; weak = one library per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the matrices of the last timed step to DIR/<name>.npy (one GPU; large ones sampled)")
    args = ap.parse_args()
    args.reads, args.baf_reads, args.cpu_sample = int(args.reads), int(args.baf_reads), int(args.cpu_sample)
    args.file_reads = int(args.file_reads)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank, world, local, dist = dist_setup(args.gpus)
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs: the GPU path on one GPU only")
    from xcltk_b200 import engine
    strong = args.scaling == "strong"
    workload_name = ("basefc C3 (%d cells, %.0fM reads, %d features: hg38 genes + nested) + baf fc C2 "
                     "(%d cells, %.0fM reads chr1-22, %d phased het SNPs), %s" % (
                         args.cells, args.reads / 1e6, args.features, args.baf_cells, args.baf_reads / 1e6,
                         args.snps, "one library over all GPUs" if strong else "per GPU"))
    bytes_nominal = args.reads * (28 + 4 * C_BAR_NOMINAL) + args.baf_reads * 8
    config = {"workload": workload_name,
              "reads_per_step": (args.reads + args.baf_reads) * (1 if strong else world),
              "partition": ("contiguous genomic chunks of one library balanced by reads, one per GPU (features / "
                            "regions by start position, reads with halo); disjoint rows, no collective"
                            if strong else "one batch (library) per GPU, no collective"),
              "calls": ("basefc and baf fc issued one after the other" if args.serial_calls else
                        "basefc and baf fc are independent calls, issued side by side from two host threads (a context and stream "
                        "each) on the same GPU; a step ends when both have returned their matrices"),
              "l2_policy": "inputs (%.1f GB of records per step%s) are larger than L2" % (
                  bytes_nominal / 1e9, ", 1/N of it per GPU" if strong else " and GPU")}

    if args.impl == "reference":
        if rank != 0:
            return
        ctx = engine.get_context(local)
        n_thr = os.cpu_count() or 1
        run, host = cpu_sample(ctx, args, args.cpu_sample, n_thr)
        for _ in range(args.warmup):
            run()
        ts = [run() for _ in range(args.steps)]
        v = run.n_reads / (sum(ts) / len(ts))
        line = {"impl": "reference", "metric": "reads/sec counted (basefc + baf fc)", "value": v, "unit": "reads/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * sum(ts) / len(ts), "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "u64 keys / i32 counts", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": "reads/s", "cores": n_thr, "kind": "port",
                                 "sample": "basefc on %d reads of the C3 generator + baf fc on the matching share of C2 "
                                           "(oracle/xg_oracle.c, OpenMP over features / SNPs like the reference's process "
                                           "pool): %d reads per step" % (args.cpu_sample, run.n_reads)},
                "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    ctx = engine.get_context(local)
    batch = Batch(ctx, args, rank, world)
    for k in range(args.warmup):
        info = batch.step_device(checksum=(k == args.warmup - 1))
    checksum = info["checksum"]
    sampler = ClockSampler(local)
    barrier_sync(dist, local)
    sampler.start()
    t0 = time.perf_counter()
    infos = [batch.step_device(keep=bool(args.dump_outputs) and k == args.steps - 1) for k in range(args.steps)]
    barrier_sync(dist, local)
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs:            # the results hold library buffers: let them go before the e2e steps are timed
        seg, baf_out = infos[-1].pop("outputs")
        mats = {"basefc": seg.to_sorted() + (seg.shape,)}
        mats.update(zip(("baf_ad", "baf_dp", "baf_oth"), baf_out))
        dump_outputs(args.dump_outputs, mats)
        del seg, baf_out, mats
    dt = max_over_ranks(dist, local, dt)
    # reads counted per step: the library once (strong: halo reads are not counted twice), or one library per GPU
    total_reads = float(args.reads + args.baf_reads) * (1 if strong else world)
    held_reads = sum_over_ranks(dist, local, float(batch.n_reads))
    value = total_reads * args.steps / dt
    info = infos[-1]
    nnz_all = sum_over_ranks(dist, local, float(info["nnz"]))

    # ---- multi-GPU parity: the shards' rows add up to the unsharded matrices (rank 0 counts the whole library)
    parity = None
    if strong and world > 1:
        import torch
        t = torch.tensor([checksum - (1 << 64) if checksum >= (1 << 63) else checksum], dtype=torch.int64,
                         device="cuda:%d" % local)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)          # int64 addition wraps like the checksum does
        sharded = int(t.item()) % (1 << 64)
        if rank == 0:
            whole = Batch(ctx, args, 0, 1)
            ref = whole.step_device(checksum=True)
            parity = {"sharded_vs_unsharded": bool(ref["checksum"] == sharded), "checksum": sharded,
                      "unsharded_checksum": ref["checksum"], "unsharded_nnz": int(ref["nnz"]), "sharded_nnz": int(nnz_all),
                      "against": "the same library counted on one GPU (rank 0), all four matrices"}
            whole.fc.dreads.close()
            whole.baf.dreads.close()
            del whole
        barrier_sync(dist, local)

    # ---- roofline of the dominant kernel (k_basefc_count): algorithmic bytes / its summed launch time
    peak, peak_src = peaks()
    t_cnt_ms = float(np.mean([i["t_fc"][1] for i in infos]))
    n_epochs = int(info["t_fc"][5])
    # c-bar of THIS batch: CIGAR words stored for the non-simple reads + one op for every simple read
    inf_fc = batch.fc.dreads.info()
    c_bar, c_bar_src = C_BAR_NOMINAL, "nominal mix (SURVEY.md 8d)"
    if not (args.no_e2e and args.no_cpu):
        try:
            batch.make_host()
            n_simple = int(np.count_nonzero((batch.h_fc.fmq >> np.uint32(24)) == 0))
            c_bar = (inf_fc["n_cigar"] + n_simple) / float(max(1, inf_fc["n_reads"]))
            c_bar_src = "this batch: (stored CIGAR words + simple reads) / reads"
        except Exception:
            pass
    bytes_per_read = 28 + 4 * c_bar
    alg_bytes = batch.fc.n_reads * bytes_per_read + 12.0 * info["nnz"]
    achieved = alg_bytes / (t_cnt_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tj = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tj):
        try:
            with open(tj) as fp:
                tr = json.load(fp)
            # measured DRAM bytes per read of the profiled launch, scaled to this run's reads per launch
            traffic = tr["k_basefc_count"]["dram_bytes"] / tr["k_basefc_count"]["reads"] * batch.fc.n_reads / max(1, n_epochs)
            traffic_src = {k: tr.get(k) for k in ("commit", "report", "when")}
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "k_basefc_count", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                "launches_per_step": n_epochs, "avg_launch_ms": t_cnt_ms / max(1, n_epochs),
                "algorithmic_bytes_per_launch": alg_bytes / max(1, n_epochs),
                "c_bar": c_bar, "c_bar_source": c_bar_src, "bytes_per_read": bytes_per_read,
                "reads_this_gpu": batch.fc.n_reads,
                "note": "launch durations from CUDA events on the launching stream; the counting launches of the "
                        "epochs follow one another on one stream (rank 0's GPU)"}
    # ---- and of the baf pileup's scan kernel: 8 B of every read, 71.7 B of the reads that cover a SNP, the
    # SNP table, 12 B per result entry (SURVEY.md 8d).  (read, SNP) pairs stand in for the covering reads.
    t_scan_ms = float(np.mean([i["t_pileup"][1] for i in infos]))
    n_pairs = float(info["t_pileup"][6])
    baf_alg = 8.0 * batch.baf.n_reads + (20 + 4 * c_bar + 46) * n_pairs + 8.0 * len(batch.baf.snp_pos) + 12.0 * info["baf_nnz"]
    roofline_baf = {"bound": "hbm", "kernel": "k_baf_scan", "achieved": baf_alg / (max(t_scan_ms, 1e-6) * 1e-3) / 1e9,
                    "peak": peak, "unit": "GB/s", "frac": baf_alg / (max(t_scan_ms, 1e-6) * 1e-3) / 1e9 / peak,
                    "avg_launch_ms": t_scan_ms, "algorithmic_bytes_per_launch": baf_alg, "read_snp_pairs": n_pairs,
                    "traffic": None}
    try:
        with open(tj) as fp:
            tb = json.load(fp).get("k_baf_scan")
        if tb:       # measured DRAM bytes per read of the profiled launch, scaled to this GPU's reads
            roofline_baf["traffic"] = tb["dram_bytes"] / tb["reads"] * batch.baf.n_reads
            roofline_baf["traffic_source"] = dict(traffic_src or {}, report=tb.get("report", (traffic_src or {}).get("report")))
    except Exception:
        pass

    e2e = None
    if not args.no_e2e:
        try:
            if not hasattr(batch, "h_fc"):
                batch.make_host()
            for _ in range(2):
                batch.step_e2e()
            barrier_sync(dist, local)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                io = batch.step_e2e()
            barrier_sync(dist, local)
            de_local = time.perf_counter() - t0
            de = max_over_ranks(dist, local, de_local)
            e2e = {"value": total_reads * args.steps / de, "unit": "reads/s", "h2d_bytes_per_step": io["h2d"],
                   "d2h_bytes_per_step": io["d2h"], "ms_per_step": 1e3 * de / args.steps,
                   "rank0_h2d_gb_s": io["h2d"] * args.steps / de_local / 1e9,
                   "rank0_d2h_gb_s": io["d2h"] * args.steps / de_local / 1e9,
                   "bytes": "rank 0's; every rank moves its own chunk"}
        except Exception as ex:            # e.g. not enough pinned host memory on the box
            e2e = {"value": None, "unit": "reads/s", "error": str(ex)[:200]}

    # ---- N = 1: parity against the CPU oracle on this batch; its wall time is the CPU baseline
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        if not hasattr(batch, "h_fc"):
            batch.make_host()
        n_thr = os.cpu_count() or 1
        parity, t_cpu = batch.oracle_parity(n_thr)
        cpu = {"value": (args.reads + args.baf_reads) / t_cpu, "unit": "reads/s", "cores": n_thr, "kind": "port",
               "sample": "the whole step on the CPU with the C oracle (oracle/xg_oracle.c, OpenMP over features / SNPs): "
                         "basefc on the %d reads of the C3 batch + baf fc on the %d reads of the C2 batch the GPU "
                         "counted, %.1f s" % (args.reads, args.baf_reads, t_cpu),
               "reference_python": REFERENCE_PYTHON}

    decode = None
    device_decode = None
    file_to_matrix = None
    if rank == 0 and world == 1 and not args.no_cpu:      # the file legs: rank 0 at N=1 only
        try:
            file_to_matrix, decode, device_decode = file_legs(ctx, args)
        except Exception as ex:
            file_to_matrix = {"error": str(ex)[:300]}

    if rank == 0:
        line = {"metric": "reads/sec counted (basefc + baf fc)", "value": value, "unit": "reads/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "u64 keys / i32 counts", "data": "synthetic", "config": config,
                "e2e": e2e, "gpu_launches": int(sum(i["launches"] for i in infos)), "clocks": clocks,
                "parity": parity, "roofline": roofline, "roofline_baf": roofline_baf, "cpu_baseline": cpu, "host_decode": decode, "device_decode": device_decode, "file_to_matrix": file_to_matrix,
                "detail": {"basefc_device_ms": float(np.mean([i["t_fc"][0] for i in infos])),
                           "basefc_epoch_span_ms": float(np.mean([i["t_fc"][3] for i in infos])),
                           "basefc_count_kernel_ms": t_cnt_ms,
                           "baf_device_ms": float(np.mean([i["t_count"][0] for i in infos])),
                           "baf_scan_kernel_ms": float(np.mean([i["t_pileup"][1] for i in infos])),
                           "baf_host_ms_pileup_queued_done": [float(np.mean([i["t_count"][k] for i in infos])) for k in (8, 9, 10)],
                           "basefc_nnz": int(nnz_all), "checksum": checksum, "reads_held_by_all_gpus": held_reads,
                           "wall_ms_basefc_baf_both_checksum": [float(x) for x in np.mean(
                               [i["wall_ms"] for i in infos], axis=0)],
                           "basefc_host_ms_index_windows_plan_upload_call": [float(x) for x in info["t_fc"][8:13]],
                           "basefc_reads_per_s_kernels_only": batch.fc.n_reads / (
                               float(np.mean([i["t_fc"][3] for i in infos])) * 1e-3)}}
        emit(line)
    if dist is not None:
        dist.destroy_process_group()
    bad_file = [k for k, v in (file_to_matrix or {}).items() if isinstance(v, dict) and v.get("matches_oracle_text") is False]
    if rank == 0 and ((parity is not None and not all(v for v in parity.values() if isinstance(v, bool))) or bad_file):
        sys.stderr.write("bench.py: PARITY MISMATCH %r %r\n" % (parity, bad_file))
        sys.exit(3)


if __name__ == "__main__":
    main()
