"""Time of extending a findSimilarPairs4 job to appended cells against a full rerun.

    python tools/extend_time.py OUTDIR [--n 1000000] [--m 1000,10000,100000] [--runs 3]

N clustered signatures (L = 1024, 512 clusters) plus M appended cells drawn from the same clusters; k = 50, threshold 0.2.
The old lists (find_similar_pairs on the first N cells) are computed once and not timed.  For each M the two calls run
alternately, `runs` times each: find_similar_pairs on all N + M cells, and extend_similar_pairs from the old lists.
Reported: medians and ranges of the calls' scan_ms and total_ms, the path the extension took, whether the outputs are
equal, and the GPU's name and power limit.  Writes OUTDIR/extend_time.json.
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
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--m", default="1000,10000,100000")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--lsh", type=int, default=1024)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--threshold", type=float, default=0.2)
    ap.add_argument("--clusters", type=int, default=512)
    a = ap.parse_args()
    Ms = [int(x) for x in a.m.split(",")]
    os.makedirs(a.outdir, exist_ok=True)
    sig = synthetic.gen_signatures(a.n + max(Ms), a.lsh, seed=2024, clusters=a.clusters)
    result = {"gpu": gpu_info(), "cells": a.n, "lsh_count": a.lsh, "k": a.k, "threshold": a.threshold, "clusters": a.clusters,
              "cases": []}
    with em2.Engine(0) as eng:
        old = eng.find_similar_pairs(sig[: a.n], a.lsh, a.k, a.threshold)
        for M in Ms:
            s = sig[: a.n + M]
            full_t, ext_t, paths, equal = {"scan_ms": [], "total_ms": []}, {"scan_ms": [], "total_ms": []}, [], True
            eng.find_similar_pairs(s, a.lsh, a.k, a.threshold)                       # warm-up of both shapes
            eng.extend_similar_pairs(s, a.n, *old, a.lsh, a.k, a.threshold)
            for _ in range(a.runs):
                want = eng.find_similar_pairs(s, a.lsh, a.k, a.threshold)
                st = eng.stats()
                full_t["scan_ms"].append(st["scan_ms"])
                full_t["total_ms"].append(st["total_ms"])
                got = eng.extend_similar_pairs(s, a.n, *old, a.lsh, a.k, a.threshold)
                st = eng.stats()
                ext_t["scan_ms"].append(st["scan_ms"])
                ext_t["total_ms"].append(st["total_ms"])
                paths.append(st["scan_symmetric"])
                equal = equal and all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(got, want))
            case = {"appended": M, "full": {k: summary(v) for k, v in full_t.items()},
                    "extend": {k: summary(v) for k, v in ext_t.items()}, "extend_scan_symmetric": paths, "outputs_equal": equal}
            result["cases"].append(case)
            print(json.dumps({"appended": M, "full_scan_ms": case["full"]["scan_ms"]["median"],
                              "extend_scan_ms": case["extend"]["scan_ms"]["median"], "paths": paths, "equal": equal}), flush=True)
    with open(os.path.join(a.outdir, "extend_time.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
