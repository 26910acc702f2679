"""Read-assignment summary (xg_basefc_summary) next to the counting kernel it accompanies.

1. Config-3 shape (300M device-synthesised reads, ~60k features with nested ones, 10k cells): basefc and the summary
   alternate in one process, `reps` warm calls each after one warm-up of both; per call the device time of
   k_basefc_count (timing()[1] of basefc: the sum over its epochs) and of k_basefc_summary (timing()[1] of the
   summary), CUDA events on the library's stream.  The 2.4 GB of pos / end alone exceed the 126 MB L2.
2. fc_wrapper wall time on tests/golden/c1_chr22_10x (rdr_defaults) with and without summary=True, alternating,
   after one warm-up call of each.
Medians and every sample go to <out>/prof_basefc_summary.json, with the card's name and power limit.

usage: python tools/prof_basefc_summary.py [n_reads] [reps] [--out DIR]"""

import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from xcltk_b200 import engine, workload  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def kernel_times(n_reads, reps):
    ctx = engine.get_context(0)
    w = workload.make_basefc_workload(ctx, n_reads, 10000, 60000, seed=7)
    cnt, summ, wall = [], [], []
    table = None
    for k in range(reps + 1):
        ctx.basefc(w.dreads, w.gid, w.beg, w.end, w.cell_keys, w.n_cells, w.params)
        t_cnt = ctx.timing()[1]
        t0 = time.perf_counter()
        t = ctx.basefc_summary(w.dreads, w.gid, w.beg, w.end, w.cell_keys, w.n_cells, w.params)
        t_wall = (time.perf_counter() - t0) * 1e3
        assert table is None or (t == table).all(), "the summary changed between calls"
        table = t
        if k:                       # the first round is the warm-up
            cnt.append(t_cnt)
            summ.append(ctx.timing()[1])
            wall.append(t_wall)
    w.dreads.close()
    return {"n_reads": n_reads, "n_features": int(len(w.gid)), "n_cells": w.n_cells, "reps": reps,
            "k_basefc_count_ms": cnt, "k_basefc_summary_ms": summ, "summary_call_wall_ms": wall,
            "median_count_ms": float(np.median(cnt)), "median_summary_ms": float(np.median(summ)),
            "median_summary_wall_ms": float(np.median(wall)),
            "records_in_range": int(table.sum()), "fates": table.sum(axis=0).tolist()}


def wrapper_times(reps):
    import logging
    from util import resolve
    from xcltk_b200.rdr.fc.main import fc_wrapper
    logging.disable(logging.CRITICAL)
    r = resolve("c1_chr22_10x", "rdr_defaults")
    td = tempfile.mkdtemp(prefix="prof_summary_")
    res = {False: [], True: []}
    try:
        for k in range(reps + 1):
            for summary in (False, True):
                out = os.path.join(td, "o%d_%d" % (k, summary))
                t0 = time.perf_counter()
                assert fc_wrapper(r["sam"][0], r["barcodes"], r["features"], out, summary=summary, **r["kwargs"]) == 0
                if k:
                    res[summary].append((time.perf_counter() - t0) * 1e3)
    finally:
        shutil.rmtree(td, ignore_errors=True)
    return {"case": "c1_chr22_10x/rdr_defaults", "reps": reps, "wall_ms_plain": res[False], "wall_ms_summary": res[True],
            "median_plain_ms": float(np.median(res[False])), "median_summary_ms": float(np.median(res[True]))}


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_dir = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out_dir in args:
        args.remove(out_dir)
    n_reads = int(float(args[0])) if args else 300000000
    reps = int(args[1]) if len(args) > 1 else 10
    res = {"card": card(), "kernels": kernel_times(n_reads, reps), "fc_wrapper": wrapper_times(reps)}
    print(json.dumps(res))
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "prof_basefc_summary.json"), "w") as fp:
            json.dump(res, fp, indent=1)


if __name__ == "__main__":
    main()
