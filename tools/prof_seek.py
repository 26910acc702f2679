"""Seek with the BAM index vs reading the whole BAM: `pileup_wrapper --chrom 22`, `afc_wrapper` on a 1 % gene
subset and `pileup_wrapper` with a dense 200 000-SNP panel, over a synthetic library of chr1..chr22
(synth.write_fast_bam: fixed-size records, whole records per BGZF block), with and without a .bai.  Runs alternate; the median wall time of each, the compressed bytes the decoder read
and the card's name and power limit are printed as one JSON line.  Everything is written to a temporary directory.

    python tools/prof_seek.py --reads 6e7 --runs 3
"""

import argparse
import json
import os
import random
import shutil
import statistics
import struct
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def reg2bin(beg, end):
    """SAMv1 section 5.3, vectorised over 0-based [beg, end)."""
    end = end - 1
    out = np.zeros(len(beg), dtype=np.int64)
    done = np.zeros(len(beg), dtype=bool)
    for shift, first in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        hit = ~done & ((beg >> shift) == (end >> shift))
        out[hit] = first + (beg[hit] >> shift)
        done |= hit
    return out


def write_bai(bam, n_ref, tid, pos, end, rec_len):
    """The .bai of a write_fast_bam file: record i sits in data block 1 + i // k at offset (i % k) * rec_len."""
    from xcltk_b200 import lib
    off, first, aligned = lib.bgzf_block_index(bam)
    assert aligned and first == 1
    k = (0xff00 // rec_len)
    i = np.arange(len(pos), dtype=np.int64)
    blk = 1 + i // k
    vb = (off[blk].astype(np.int64) << 16) | ((i % k) * rec_len)
    ve = (off[blk].astype(np.int64) << 16) | ((i % k + 1) * rec_len)      # what bgzf_tell gives after the record
    bins = reg2bin(pos, end)
    buf = bytearray(b"BAI\1" + struct.pack("<i", n_ref))
    for t in range(n_ref):
        sel = np.nonzero(tid == t)[0]
        if len(sel) == 0:
            buf += struct.pack("<ii", 0, 0)
            continue
        b, p, e, s, f = bins[sel], pos[sel], end[sel], vb[sel], ve[sel]
        cut = np.nonzero(np.diff(b) != 0)[0] + 1                  # chunks: runs of consecutive records of one bin
        starts = np.concatenate([[0], cut])
        ends = np.concatenate([cut, [len(b)]]) - 1
        cb, ce, cbin = s[starts], f[ends], b[starts]
        order = np.lexsort((cb, cbin))
        cb, ce, cbin = cb[order], ce[order], cbin[order]
        ub, at, cnt = np.unique(cbin, return_index=True, return_counts=True)
        buf += struct.pack("<i", len(ub))
        for u, a, c in zip(ub, at, cnt):
            buf += struct.pack("<Ii", int(u), int(c))
            buf += np.stack([cb[a:a + c], ce[a:a + c]], axis=1).astype("<u8").tobytes()
        n_win = int((e.max() - 1) >> 14) + 1
        big = np.iinfo(np.int64).max
        lin = np.full(n_win, big, dtype=np.int64)
        np.minimum.at(lin, p >> 14, s)                            # reads of 91 bp touch one or two windows
        np.minimum.at(lin, (e - 1) >> 14, s)
        lin = np.maximum.accumulate(np.where(lin == big, -1, lin))   # holes: the previous window's offset
        lin[lin < 0] = s[0]
        buf += struct.pack("<i", n_win) + lin.astype("<u8").tobytes()
    buf += struct.pack("<Q", 0)
    with open(bam + ".bai", "wb") as fp:
        fp.write(bytes(buf))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=float, default=6e7)
    ap.add_argument("--cells", type=int, default=5000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None, help="JSON result file (besides stdout)")
    a = ap.parse_args()
    from xcltk_b200 import engine, lib, synth, workload
    from xcltk_b200.baf.fc.main import afc_wrapper
    from xcltk_b200.baf.pileup import pileup_wrapper
    logging_off = __import__("logging")
    logging_off.disable(logging_off.WARNING)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    td = tempfile.mkdtemp(prefix="prof_seek_")
    try:
        contigs = [("chr" + c, workload.HG38_LEN[c]) for c in workload.HG38_CHROMS[:22]]
        bam = os.path.join(td, "lib.bam")
        t0 = time.time()
        barcodes = synth.write_fast_bam(bam, int(a.reads), contigs, n_cells=a.cells, seed=7, level=1, threads=16)
        t_write = time.time() - t0
        ctx = engine.get_context(0)
        dev, _seen = ctx.decode_bams([bam], [np.arange(len(contigs), dtype=np.int32)], "CB", "UB", False)
        host = dev.download()
        dev.close()
        pos = host.pos_end[:, 0].astype(np.int64)
        end = host.pos_end[:, 1].astype(np.int64)
        tid = np.zeros(host.n, dtype=np.int64)
        for _b, g, rb, re_ in host.runs:
            tid[rb:re_] = g
        host.close()
        rec_len = 4 + 32 + 11 + 4 + 46 + 91 + 4 + 22 + 16
        t0 = time.time()
        write_bai(bam, len(contigs), tid, pos, end, rec_len)
        t_index = time.time() - t0
        os.rename(bam + ".bai", bam + ".bai.off")
        bc = os.path.join(td, "barcodes.tsv")
        synth.write_lines(bc, barcodes)
        genes = [g for g in workload.load_genes() if g[0] in workload.HG38_CHROMS[:22]]
        rng = random.Random(3)
        sub = sorted(rng.sample(genes, max(1, len(genes) // 100)), key=lambda g: (int(g[0]), g[1]))
        ft = os.path.join(td, "genes.tsv")
        synth.write_features(ft, [("chr" + c, s, e, n) for c, s, e, n in sub])
        snps = synth.gen_snps(5, sub, 20000)
        st = os.path.join(td, "snps.tsv")
        synth.write_snp_tsv(st, snps, chr_prefix="chr")
        # a dense candidate panel: 200 000 SNPs over all autosomes (ranges closer than XG_BAM_INDEX_MERGE_GAP merge)
        prng = random.Random(9)
        dense = {}
        for c, ln in ((c, workload.HG38_LEN[c]) for c in workload.HG38_CHROMS[:22]):
            n_c = max(1, int(200000 * ln / 2.9e9))
            dense[c] = [(pp, "A", "C", 0) for pp in sorted(prng.sample(range(1, ln), n_c))]
        panel = os.path.join(td, "panel.tsv")
        synth.write_snp_tsv(panel, dense, chr_prefix="chr")
        read = []
        real = engine.load_reads

        def spy(*x, **kw):
            b = real(*x, **kw)
            read.append(b.stats.get("bytes_read"))
            return b
        engine.load_reads = spy
        # ~1.9x depth of random bases: min_count 8 keeps a few 10k sites on chr22
        jobs = {"pileup_chrom22": lambda out: pileup_wrapper(bam, bc, None, out, ncores=16, chrom="22", min_count=8,
                                                             min_maf=0.1),
                "afc_genes_1pct": lambda out: afc_wrapper(bam, bc, ft, st, out, ncores=16),
                "pileup_panel_200k": lambda out: pileup_wrapper(bam, bc, panel, out, ncores=16)}
        res = {}
        for name, job in jobs.items():
            times = {False: [], True: []}
            nread = {}
            outs = {}
            for r in range(a.runs + 1):                            # the first pair warms up
                for with_index in (False, True):
                    if with_index:
                        os.rename(bam + ".bai.off", bam + ".bai")
                    out = os.path.join(td, "%s_%d_%d" % (name, r, with_index))
                    del read[:]
                    t0 = time.time()
                    assert job(out) == 0
                    dt = time.time() - t0
                    if with_index:
                        os.rename(bam + ".bai", bam + ".bai.off")
                    if r:
                        times[with_index].append(dt)
                    nread[with_index] = read[-1]
                    outs[with_index] = {f: open(os.path.join(out, f), "rb").read() for f in sorted(os.listdir(out))}
                    shutil.rmtree(out)
                assert outs[False] == outs[True], name
            res[name] = {"median_s_whole": statistics.median(times[False]),
                         "median_s_index": statistics.median(times[True]),
                         "runs_whole": times[False], "runs_index": times[True],
                         "bytes_read_whole": nread[False], "bytes_read_index": nread[True]}
        line = {"card": card, "reads": int(a.reads), "bam_bytes": os.path.getsize(bam), "write_s": t_write,
                "index_s": t_index, "runs": a.runs, "results": res}
        print(json.dumps(line))
        if a.out:
            with open(a.out, "w") as fp:
                fp.write(json.dumps(line) + "\n")
    finally:
        shutil.rmtree(td, ignore_errors=True)


if __name__ == "__main__":
    main()
