"""SNP discovery (xg_snp_discover) on the config-2 shape: 50M device-synthesised reads, 5k cells, a pseudo-reference
at 0.1 % base errors and 200k planted heterozygous SNPs, discovered on the whole autosomes with min_count 20 /
min_maf 0.1 (the command line's defaults) and with min_count 3 / min_maf 0.1 (the shape has about 3 reads per
position, so only the second filter leaves work for the exact stage).  20 warm calls each:
medians of the raw scan, the exact stage and the whole call (device time, timing()[1] / [3] / [0]) and the host wall
time, the positions scanned, raw candidates and kept sites; then snp_pileup on the planted SNPs in the same process
for comparison.  Prints the card's name and power limit.

usage: python tools/prof_snp_discover.py [n_reads] [--out DIR]"""

import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from xcltk_b200 import engine, workload  # noqa: E402


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
    b = workload.make_baf_workload(ctx, n_reads, 5000, 200000, seed=11, ref_error=0.001)
    tg = (np.arange(len(b.contigs), dtype=np.int32), np.zeros(len(b.contigs), np.int32),
          np.array([workload.HG38_LEN[c] for c in b.contigs], np.int32))             # whole autosomes
    n = len(b.snp_pos)

    def snp():
        return ctx.snp_pileup(b.dreads, b.snp_gid, b.snp_pos, b.cell_keys, 5000, b.params, b.snp_ref, b.snp_alt, 0, 0.0)

    planted = set(zip(b.snp_gid.tolist(), b.snp_pos.tolist()))
    summary = {"card": card(), "n_reads": n_reads, "n_cells": 5000, "planted_snps": n}
    snp()
    res = {"snp_pileup_span_ms": [], "snp_pileup_wall_ms": []}
    for _ in range(20):
        t0 = time.perf_counter()
        snp()
        res["snp_pileup_wall_ms"].append(1e3 * (time.perf_counter() - t0))
        res["snp_pileup_span_ms"].append(ctx.timing()[0])
    # the command line's defaults (20, 0.1), and a filter the shape's depth of about 3 reads per position can pass
    for min_count, min_maf in ((20, 0.1), (3, 0.1)):
        name = "discover_%g_%g" % (min_count, min_maf)

        def disc():
            return ctx.snp_discover(b.dreads, tg[0], tg[1], tg[2], b.cell_keys, 5000, b.params, min_count, min_maf)
        sites = disc()
        r = {"whole_ms": [], "raw_scan_ms": [], "exact_ms": [], "wall_ms": []}
        for _ in range(20):
            t0 = time.perf_counter()
            disc()
            r["wall_ms"].append(1e3 * (time.perf_counter() - t0))
            t = ctx.timing()
            r["whole_ms"].append(t[0])
            r["raw_scan_ms"].append(t[1])
            r["exact_ms"].append(t[3])
        found = set(zip(sites["gid"].tolist(), sites["pos"].tolist()))
        summary[name] = {"covered_windows": t[5], "positions_scanned": t[6], "raw_candidates": t[7],
                         "kept_sites": t[14], "read_window_entries": t[13], "pileup_slices": t[11],
                         "launches": t[2], "planted_found": len(planted & found)}
        for k, v in r.items():
            summary[name][k + "_median"] = float(np.median(v))
            summary[name][k + "_min"] = float(np.min(v))
            summary[name][k + "_max"] = float(np.max(v))
        res[name] = r
    for k in ("snp_pileup_span_ms", "snp_pileup_wall_ms"):
        summary[k + "_median"] = float(np.median(res[k]))
    print(json.dumps(summary, indent=1))
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "prof_snp_discover.json"), "w") as fp:
            json.dump(dict(summary, raw=res), fp, indent=1)


if __name__ == "__main__":
    main()
