"""Exact path on log-normalised counts (general arithmetic): the candidate filter against full evaluation of every row.

    python tools/exact_general_time.py OUTDIR [--quick]

1. The config-5 shape (50k cells x 20k genes, 1000 stored values per cell) with log1p counts: the filter path and option
   "exact_filter" = 1 (every row evaluated in full), alternating, 3 runs each; medians and ranges of scan_ms / total_ms,
   the stats counters, and whether the two outputs are equal bit for bit.
2. 200k cells x 30k genes x 1500 per cell, which full evaluation could not serve before (more than 25,600 genes): the filter
   path alone, its time and counters.
The GPU's name and power limit are read in the same run.  Writes OUTDIR/exact_general_time.json."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402

KEYS = ("scan_ms", "total_ms", "filter_cells", "filter_uncertain", "candidates_appended", "kernel_launches", "variant_used")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def data(n, G, per_cell, seed):
    toc, genes, counts = synthetic.gen_expression_matrix_fast(n, G, per_cell, seed=seed, clusters=64)
    return toc, genes, (np.log1p(counts) * np.float32(1.7)).astype(np.float32)


def run(eng, toc, pairs, G, k, thr, full):
    eng.set_option("exact_filter", 1 if full else 0)
    n = len(toc) - 1
    out = np.zeros((n, k), em2.SIMPAIR_DTYPE)
    used = np.zeros(n, np.uint32)
    eng.exact_similar_pairs_into(toc, pairs, G, k, thr, out, used)
    st = eng.stats()
    return {key: st[key] for key in KEYS}, out, used


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "runs": [float(x) for x in xs]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--quick", action="store_true", help="small shapes (a rehearsal of the script)")
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--threshold", type=float, default=0.2)
    a = ap.parse_args()
    os.makedirs(a.outdir, exist_ok=True)
    shape5 = (4000, 2000, 100) if a.quick else (50_000, 20_000, 1000)
    big = (8000, 3000, 150) if a.quick else (200_000, 30_000, 1500)
    res = {"gpu": gpu_info(), "k": a.k, "threshold": a.threshold}
    with em2.Engine(0) as eng:
        toc, genes, counts = data(*shape5, seed=5)
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = synthetic.to_pairs(genes, counts)
        G = shape5[1]
        run(eng, toc, pairs, G, a.k, a.threshold, False)                 # warm-up: module load, scratch allocation
        runs = {"filter": [], "full": []}
        outs = {}
        for _ in range(3):
            for mode in ("filter", "full"):
                st, out, used = run(eng, toc, pairs, G, a.k, a.threshold, mode == "full")
                runs[mode].append(st)
                outs[mode] = (out.view(np.uint64).copy(), used.copy())
        res["config5"] = {"cells": shape5[0], "genes": shape5[1], "per_cell": shape5[2],
                          "outputs_equal": bool(np.array_equal(outs["filter"][0], outs["full"][0])
                                                and np.array_equal(outs["filter"][1], outs["full"][1]))}
        for mode in runs:
            res["config5"][mode] = {"scan_ms": summary([r["scan_ms"] for r in runs[mode]]),
                                    "total_ms": summary([r["total_ms"] for r in runs[mode]]),
                                    "counters": {key: runs[mode][-1][key] for key in KEYS[2:]}}
        del toc, genes, counts, pairs, outs
        toc, genes, counts = data(*big, seed=7)
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = synthetic.to_pairs(genes, counts)
        st, out, used = run(eng, toc, pairs, big[1], a.k, a.threshold, False)
        res["large"] = {"cells": big[0], "genes": big[1], "per_cell": big[2], "filter": st,
                        "used_mean": float(used.mean())}
        eng.set_option("exact_filter", 0)
    res["gpu_after"] = gpu_info()
    path = os.path.join(a.outdir, "exact_general_time.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
