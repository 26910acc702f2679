"""SNP-level counting: xg_snp_pileup against xg_baf_fc with one region per SNP (GT 0|1) on the config-2 shape
(50M device-synthesised reads, 5k cells, 200k SNPs).  The two routes alternate in one process, 20 warm calls each;
per call: device span (timing()[0]), host wall time to the results on the host.  A separate profiled pass gives
the time of the reduction kernels of each route (CUDA activity records).  The matrices of the two routes must be
identical.  Prints the card's name and power limit.

usage: python tools/prof_snp_pileup.py [n_reads] [--out DIR]"""

import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from xcltk_b200 import engine, workload  # noqa: E402

# kernels after the pileup (k_baf_first / k_baf_resolve and the scan are shared by both routes)
SNP_KERNELS = ("k_snp_hist", "k_snp_scatter", "k_snp_finalize")
FC_KERNELS = ("k_baf_count_combos", "k_baf_region_masks", "k_baf_finalize")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_dir = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out_dir in args:
        args.remove(out_dir)
    n_reads = int(float(args[0])) if args else 50000000
    ctx = engine.get_context(0)
    b = workload.make_baf_workload(ctx, n_reads, 5000, 200000, seed=11)
    n = len(b.snp_pos)
    reg_ptr, reg_snp = np.arange(n + 1, dtype=np.int64), np.arange(n, dtype=np.int32)
    hap = np.full((n, 8), 2, np.uint8)
    hap[np.arange(n), b.snp_ref] = 0
    hap[np.arange(n), b.snp_alt] = 1

    def snp():
        return ctx.snp_pileup(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 5000, b.params, b.snp_ref, b.snp_alt, 0, 0.0)

    def fc():
        return ctx.baf_fc(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 5000, b.params, b.snp_ref, b.snp_alt, 0, 0.0,
                          reg_ptr, reg_snp, hap, True)

    routes = {"snp_pileup": snp, "baf_fc_one_region_per_snp": fc}
    a, c = snp(), fc()                              # warm-up, and the two results must be identical
    for x, y in zip(a, c):
        for k in range(3):
            assert np.array_equal(np.asarray(x[k]), np.asarray(y[k])), "routes differ"
    res = {name: {"span_ms": [], "wall_ms": []} for name in routes}
    for _ in range(20):
        for name, f in routes.items():
            t0 = time.perf_counter()
            f()
            res[name]["wall_ms"].append(1e3 * (time.perf_counter() - t0))
            res[name]["span_ms"].append(ctx.timing()[0])
    t = ctx.timing()
    snp()
    ts = ctx.timing()
    # kernel times, profiled pass of its own
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            snp()
            fc()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        for k in SNP_KERNELS + FC_KERNELS:
            if k in ev.key:
                kern[k] = kern.get(k, 0.0) + ev.device_time_total / 1e3 / 5    # ms per call
    summary = {
        "card": card(), "n_reads": n_reads, "n_cells": 5000, "n_snps": n,
        "pairs": ts[6], "winners": ts[7], "warp_path_snps": ts[14], "cta_path_snps": ts[15], "launches_fc": t[2],
        "launches_snp": ts[2], "dp_nnz": int(len(a[1][2])),
        "kernel_ms_per_call": kern,
        "snp_reduction_ms": sum(kern.get(k, 0.0) for k in SNP_KERNELS),
        "fc_reduction_ms": sum(kern.get(k, 0.0) for k in FC_KERNELS),
    }
    for name, r in res.items():
        for key in ("span_ms", "wall_ms"):
            v = np.array(r[key])
            summary["%s_%s_median" % (name, key)] = float(np.median(v))
            summary["%s_%s_min" % (name, key)] = float(v.min())
            summary["%s_%s_max" % (name, key)] = float(v.max())
    print(json.dumps(summary, indent=1))
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "prof_snp_pileup.json"), "w") as fp:
            json.dump(dict(summary, raw=res), fp, indent=1)


if __name__ == "__main__":
    main()
