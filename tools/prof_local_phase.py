"""Local phasing from the reads: xg_local_phase on the config-2 shape (50M device-synthesised reads, 5k cells, 200k
SNPs inside hg38 genes).  The SNPs of the long genes (>= 50 kb, >= 2 SNPs, SNP span >= 50 kb) are piled up with
xg_snp_pileup (filter (0, 0)); then
  device  local_phasing_device over all long genes, 5 warm calls: EM kernel time and device span (median), the
          longest single region, waves, regions, SNPs, non-zeros, inner EM iterations;
  host    reg_local_phasing region by region in list order on the same matrices, for as many regions as fit in
          --host-budget seconds (a prefix in list order, so that the device can be run on the same prefix and the
          flips compared);
  e2e     afc_wrapper(phase_from_reads=True) against pileup_wrapper -> afc_wrapper(cellsnp_dir=...) on the
          c1_chr22_10x golden BAM (small: overheads, not throughput), best of 3 each, same output bytes.
Prints the card's name and power limit.

usage: python tools/prof_local_phase.py [n_reads] [--host-budget S] [--out DIR]"""

import json
import os
import subprocess
import sys
import tempfile
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from xcltk_b200 import engine, workload  # noqa: E402
from xcltk_b200.baf.fc.config import Config  # noqa: E402
from xcltk_b200.baf.fc.gfeature import SNP, BlockRegion  # noqa: E402
from xcltk_b200.baf.fc.phasing import (csr_from_coo, is_long_region, local_phasing_device,  # noqa: E402
                                       reg_local_phasing)

BASES = "ACGT"


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def arg(name, default):
    return sys.argv[sys.argv.index(name) + 1] if name in sys.argv else default


def same(a, b):
    return (a is None and b is None) or (a is not None and b is not None and np.array_equal(a, b))


def build(w):
    """Fresh SNP objects and long gene regions (the EM changes both)."""
    snps = []
    for i in range(len(w.snp_pos)):
        s = SNP(w.contigs[w.snp_gid[i]], int(w.snp_pos[i]) + 1, BASES[w.snp_ref[i]], BASES[w.snp_alt[i]],
                int(w.snp_ref_hap[i]), 1 - int(w.snp_ref_hap[i]))
        s.index = i
        snps.append(s)
    conf = Config()
    regs = []
    for k, (c, s, e, name) in enumerate(w.feats):
        ids = w.reg_snp[w.reg_ptr[k]:w.reg_ptr[k + 1]]
        if len(ids) == 0:
            continue
        reg = BlockRegion(c, s, e + 1, name, [snps[i] for i in ids])
        if is_long_region(conf, reg):
            regs.append(reg)
    return snps, regs


def e2e(tmp):
    from xcltk_b200.baf.fc.main import afc_wrapper
    from xcltk_b200.baf.pileup import pileup_wrapper
    g = os.path.join(ROOT, "tests", "golden", "c1_chr22_10x")
    inp = (os.path.join(g, "a.bam"), os.path.join(g, "barcodes.tsv"))
    feats, snp_fn = os.path.join(g, "features.tsv"), os.path.join(g, "snps.tsv")
    files = ("xcltk.region.tsv", "xcltk.samples.tsv", "xcltk.AD.mtx", "xcltk.DP.mtx", "xcltk.OTH.mtx")

    def two_step(out):
        csd = out + "_csp"
        assert pileup_wrapper(*inp, snp_fn, csd, ncores=4) == 0
        assert afc_wrapper(*inp, feats, snp_fn, out, ncores=4, cellsnp_dir=csd, output_all_reg=True) == 0

    def one_call(out):
        assert afc_wrapper(*inp, feats, snp_fn, out, ncores=4, phase_from_reads=True, output_all_reg=True) == 0

    res, same = {"two_step": [], "phase_from_reads": []}, True
    for k in range(4):                           # the first pair warms up
        got = {}
        for name, f in (("two_step", two_step), ("phase_from_reads", one_call)):
            out = os.path.join(tmp, "%s%d" % (name, k))
            t0 = time.perf_counter()
            f(out)
            if k:
                res[name].append(time.perf_counter() - t0)
            got[name] = [open(os.path.join(out, x), "rb").read() for x in files]
        same = same and got["two_step"] == got["phase_from_reads"]
    return {"e2e_c1_two_step_s_best": min(res["two_step"]),
            "e2e_c1_phase_from_reads_s_best": min(res["phase_from_reads"]), "e2e_c1_same_bytes": same}


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_dir = arg("--out", None)
    budget = float(arg("--host-budget", 120))
    args = [a for a in args if a not in (out_dir, arg("--host-budget", None))]
    n_reads = int(float(args[0])) if args else 50000000
    ctx = engine.get_context(0)
    w = workload.make_baf_workload(ctx, n_reads, 5000, 200000, seed=11)
    snps, regs = build(w)
    ids = np.unique(np.concatenate([[s.index for s in r.snp_list] for r in regs]))
    t0 = time.perf_counter()
    ad, dp, _oth = ctx.snp_pileup(w.dreads, w.snp_gid[ids], w.snp_pos[ids], w.cell_keys, 5000, w.params,
                                  w.snp_ref[ids], w.snp_alt[ids], 0, 0.0)
    t_pileup = time.perf_counter() - t0

    def coo(m):
        return ids[np.asarray(m[0], dtype=np.int64)], np.asarray(m[1]), np.asarray(m[2])
    csr = csr_from_coo(len(snps), coo(ad), coo(dp), np.ones(5000, dtype=bool))

    def device(n_regions=None):
        s, r = build(w)
        r = r[:n_regions] if n_regions is not None else r
        t0 = time.perf_counter()
        flips, t = local_phasing_device(ctx, r, s, csr, 5000)
        return flips, t, time.perf_counter() - t0, r

    device()                                       # warm-up
    runs = [device() for _ in range(5)]
    t = runs[-1][1]
    flips_all = runs[-1][0]
    assert all(same(a, b) for r in runs for a, b in zip(r[0], flips_all)), "device runs differ"
    # host reference: a prefix of the regions in list order, within the budget
    s_h, r_h = build(w)
    row_ptr, col, a_v, d_v = csr
    host_flips, t_host, n_host = [], 0.0, 0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for reg in r_h:
            sel = [s.index for s in reg.snp_list]
            AD = np.zeros((5000, len(sel)), dtype=np.int64)
            DP = np.zeros_like(AD)
            for j, g in enumerate(sel):
                AD[col[row_ptr[g]:row_ptr[g + 1]], j] = a_v[row_ptr[g]:row_ptr[g + 1]]
                DP[col[row_ptr[g]:row_ptr[g + 1]], j] = d_v[row_ptr[g]:row_ptr[g + 1]]
            t0 = time.perf_counter()
            _reg, f = reg_local_phasing(reg, AD, DP)
            t_host += time.perf_counter() - t0
            host_flips.append(f)
            n_host += 1
            if t_host > budget:
                break
    dev_prefix = device(n_host)
    equal = all(same(a, b) for a, b in zip(host_flips, dev_prefix[0]))
    lists_equal = all([s.index for s in a.snp_list] == [s.index for s in b.snp_list]
                      for a, b in zip(r_h[:n_host], dev_prefix[3]))
    with tempfile.TemporaryDirectory() as tmp:
        ee = e2e(tmp)
    summary = {
        "card": card(), "n_reads": n_reads, "n_cells": 5000, "n_snps": len(snps),
        "long_regions": len(regs), "region_snp_slots": int(sum(len(r.snp_list) for r in runs[-1][3])),
        "snps_piled_up": int(len(ids)), "dp_nnz": int(len(csr[1])), "entries": t[7], "waves": t[2],
        "inner_iterations": t[4], "device_calls": t[9], "tie_regions_decided_on_host": t[10], "failed": int(sum(f is None for f in flips_all)),
        "pileup_wall_s": t_pileup,
        "device_em_ms_median": float(np.median([r[1][1] for r in runs])),
        "device_span_ms_median": float(np.median([r[1][0] for r in runs])),
        "device_call_wall_ms_median": float(np.median([1e3 * r[2] for r in runs])),
        "largest_region_ms": t[5], "largest_region_share": t[6],
        "host_regions_timed": n_host, "host_s": t_host,
        "device_em_ms_same_prefix": dev_prefix[1][1],
        "flips_equal_on_prefix": bool(equal), "pruned_lists_equal_on_prefix": bool(lists_equal),
    }
    summary.update(ee)
    print(json.dumps(summary, indent=1))
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "prof_local_phase.json"), "w") as fp:
            json.dump(summary, fp, indent=1)


if __name__ == "__main__":
    main()
