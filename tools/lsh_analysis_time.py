"""LSH accuracy analysis (em2_analyze_lsh) against the exact similar-pairs job at the same shape.

    python tools/lsh_analysis_time.py OUTDIR [--quick]

Shapes: config 5 (50k cells x 20k genes) and 200k cells x 20k genes, integer clustered counts with 1000 stored per cell,
L = 1024, 20 bins.  Per shape, after one warm-up call of each: 3 runs of analyze_lsh (similarity stage = scan_ms, binning =
finalize_ms, total_ms; medians and ranges; pairs per second of the whole call and of the binning) and 3 runs of
exact_similar_pairs (k = 100, threshold 0.2) at the same shape, plus the ordered pairs each similarity stage computes.  The
GPU's name and power limit are read in the same run.  Writes OUTDIR/lsh_analysis_time.json."""
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


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "runs": [float(x) for x in xs]}


def computed_pairs(n, budget=48 << 30):
    """Ordered pairs the similarity stages compute (the host's chunk rule in em2_analyze_lsh and exactRect)."""
    def up(x, m):
        return -(-x // m) * m
    ld = up(n, 256)
    budget_rows = max(128, budget // (ld * 4) // 128 * 128)
    full = n * n if budget_rows < n else n * n // 2     # the full job's symmetric GEMM computes tiles on or above the diagonal
    if budget_rows >= n:
        return n * n // 2, full
    chunk = min(budget_rows, max(4096, up(up(n, 8) // 8, 128)), up(n, 128))
    cap, r0, total = chunk * ld, 0, 0
    while r0 < n:
        ldc = up(n - r0, 256)
        rows = min(n - r0, max(128, cap // ldc // 128 * 128))
        total += rows * (n - r0)
        r0 += rows
    return total, full


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--quick", action="store_true", help="small shapes (a rehearsal of the script)")
    args = ap.parse_args()
    os.makedirs(args.outdir, exist_ok=True)
    G, per_cell, L, B, k, thr = 20000, 1000, 1024, 20, 100, 0.2
    shapes = [4000, 9000] if args.quick else [50000, 200000]
    if args.quick:
        G, per_cell = 2000, 100
    result = {"gpu": gpu_info(), "genes": G, "stored_per_cell": per_cell, "lsh_count": L, "bins": B, "shapes": []}
    with em2.Engine(0) as eng:
        result["device"] = eng.device_name
        for n in shapes:
            toc, genes, counts = synthetic.gen_expression_matrix_fast(n, G, per_cell, seed=5, clusters=64)
            pairs = em2.to_pairs(genes, counts)
            sig = eng.compute_signatures(toc, pairs, em2.generate_lsh_vectors(G, L, 231))
            pair_total = n * (n - 1) // 2
            runs = {"scan_ms": [], "finalize_ms": [], "total_ms": []}
            eng.analyze_lsh(toc, pairs, G, sig, L, B)                          # warm-up
            for _ in range(3):
                out = eng.analyze_lsh(toc, pairs, G, sig, L, B)
                st = eng.stats()
                for key in runs:
                    runs[key].append(st[key])
            assert int(out["pair_count"].sum()) + int(out["undefined_pairs"]) == pair_total
            ids = np.zeros((n, k), em2.SIMPAIR_DTYPE)
            used = np.zeros(n, np.uint32)
            exact = {"scan_ms": [], "total_ms": []}
            eng.exact_similar_pairs_into(toc, pairs, G, k, thr, ids, used)      # warm-up
            for _ in range(3):
                eng.exact_similar_pairs_into(toc, pairs, G, k, thr, ids, used)
                st = eng.stats()
                for key in exact:
                    exact[key].append(st[key])
            window, full = computed_pairs(n)
            shape = {
                "cells": n, "pairs": pair_total, "variant_used": st["variant_used"],
                "analyze": {key: summary(v) for key, v in runs.items()},
                "analyze_pairs_per_s": pair_total / (np.median(runs["total_ms"]) * 1e-3),
                "binning_pairs_per_s": pair_total / (np.median(runs["finalize_ms"]) * 1e-3),
                "binning_share_of_similarity_stage": float(np.median(runs["finalize_ms"]) / np.median(runs["scan_ms"])),
                "exact_similar_pairs": {key: summary(v) for key, v in exact.items()},
                "ordered_pairs_computed": {"analyze": window, "exact_similar_pairs": full, "ratio": window / full},
                "bins": {key: np.asarray(out[key]).tolist() for key in ("pair_count", "sum_error", "sum_squared_error")},
                "undefined_pairs": int(out["undefined_pairs"]),
            }
            result["shapes"].append(shape)
            print(json.dumps({key: shape[key] for key in ("cells", "analyze", "binning_share_of_similarity_stage",
                                                           "exact_similar_pairs", "ordered_pairs_computed")}), flush=True)
    with open(os.path.join(args.outdir, "lsh_analysis_time.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
