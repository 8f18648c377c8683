"""Time of extending a findSimilarPairs0 (exact Pearson) job to appended cells against a full rerun.

    python tools/extend_exact_time.py OUTDIR [--n 50000,200000] [--m 1000,10000] [--genes 20000] [--nnz 1000] [--runs 3]

For each N: N + max(M) seeded clustered integer counts (synthetic.gen_expression_matrix_fast, 20k genes, 1000 stored counts
per cell as config 5 of bench.py), k = 50, threshold 0.2.  The old lists (exact_similar_pairs on the first N cells) are
computed once and not timed.  For each M the two calls run alternately, `runs` times each after one warm-up of both:
exact_similar_pairs on all N + M cells, and extend_exact_similar_pairs from the old lists.  Reported: medians and ranges of
the calls' scan_ms and total_ms (total includes the host-to-device copy of all counts, which both calls make), the path the
extension took, whether the outputs are equal, and the GPU's name and power limit.  Writes OUTDIR/extend_exact_time.json.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit": power}


def summary(values):
    v = sorted(values)
    return {"median": float(np.median(v)), "min": v[0], "max": v[-1], "runs": v}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--n", default="50000,200000")
    ap.add_argument("--m", default="1000,10000")
    ap.add_argument("--genes", type=int, default=20000)
    ap.add_argument("--nnz", type=int, default=1000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--threshold", type=float, default=0.2)
    ap.add_argument("--clusters", type=int, default=64)
    a = ap.parse_args()
    Ns = [int(x) for x in a.n.split(",")]
    Ms = [int(x) for x in a.m.split(",")]
    os.makedirs(a.outdir, exist_ok=True)
    result = {"gpu": gpu_info(), "genes": a.genes, "nnz_per_cell": a.nnz, "k": a.k, "threshold": a.threshold,
              "clusters": a.clusters, "cases": []}
    G, k, thr = a.genes, a.k, a.threshold
    with em2.Engine(0) as eng:
        for N in Ns:
            toc, genes, counts = synthetic.gen_expression_matrix_fast(N + max(Ms), G, a.nnz, seed=N, clusters=a.clusters)
            pairs = synthetic.to_pairs(genes, counts)
            del genes, counts
            e = int(toc[N])
            old = eng.exact_similar_pairs(toc[: N + 1], pairs[:e], G, k, thr)
            for M in Ms:
                t, p = toc[: N + M + 1], pairs[: int(toc[N + M])]
                full_t, ext_t, paths, equal = {"scan_ms": [], "total_ms": []}, {"scan_ms": [], "total_ms": []}, [], True
                eng.exact_similar_pairs(t, p, G, k, thr)                             # warm-up of both shapes
                eng.extend_exact_similar_pairs(t, p, G, N, *old, k, thr)
                for _ in range(a.runs):
                    want = eng.exact_similar_pairs(t, p, G, k, thr)
                    st = eng.stats()
                    full_t["scan_ms"].append(st["scan_ms"])
                    full_t["total_ms"].append(st["total_ms"])
                    got = eng.extend_exact_similar_pairs(t, p, G, N, *old, k, thr)
                    st = eng.stats()
                    ext_t["scan_ms"].append(st["scan_ms"])
                    ext_t["total_ms"].append(st["total_ms"])
                    paths.append(st["scan_symmetric"])
                    equal = equal and all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(got, want))
                case = {"cells": N, "appended": M, "full": {q: summary(v) for q, v in full_t.items()},
                        "extend": {q: summary(v) for q, v in ext_t.items()}, "extend_scan_symmetric": paths,
                        "outputs_equal": equal}
                result["cases"].append(case)
                print(json.dumps({"cells": N, "appended": M, "full_scan_ms": case["full"]["scan_ms"]["median"],
                                  "extend_scan_ms": case["extend"]["scan_ms"]["median"], "paths": paths, "equal": equal}), flush=True)
            del toc, pairs, old
    with open(os.path.join(a.outdir, "extend_exact_time.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
