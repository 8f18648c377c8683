"""Time and quality of rescoring LSH candidate lists with the exact (Pearson) similarities, against the full exact job.

    python tools/rescore_time.py OUTDIR [--n 50000,200000,1000000] [--widths 50,100,200,500,1000] [--genes 20000]
                                        [--nnz 1000] [--runs 3]

For each N: seeded clustered integer counts (synthetic.gen_expression_matrix_fast, 20k genes, 1000 stored counts per cell, the
shapes of extend_exact_time.py).  For each candidate width k', the candidates are lsh_similar_pairs lists (L = 1024,
threshold 0.2, k'; k' > 112 takes the one-directional scan), timed once as "the LSH job".  rescore_similar_pairs to k = 50
runs once as a warm-up, then `runs` times: medians and ranges of scan_ms (the rescoring stage) and total_ms (which includes
the host-to-device copy of the counts and the candidates), whether the outputs are equal across runs, the bytes of candidate
CSR the kernel reads (stored counts of every listed candidate x 8 B, from the shapes) and those bytes over the median scan
time.  At N <= 200k the full exact_similar_pairs (k = 50) is timed the same way and is the reference for quality:
  id_recall: |rescored ids & exact ids| / |exact ids| over all rows;
  above_kth: the fraction of rescored entries whose similarity is at least the row's exact k-th similarity (every passing
             entry when the exact row is not full) -- ties make id recall understate quality on clustered data;
and the same two figures for the plain k' = 50 LSH lists (their entries' exact similarities from the k' = 50 rescoring).
1 M cells run when the host has the memory for them (about 48 GB).  The GPU's name and power limit are read in the same run.
Writes OUTDIR/rescore_time.json.
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


def entry_keys(ids, used):
    """row * 2^32 + id of every used entry."""
    mask = np.arange(ids.shape[1])[None, :] < used[:, None]
    rows = np.nonzero(mask)[0].astype(np.uint64)
    return (rows << np.uint64(32)) | ids[mask].astype(np.uint64)


def quality(ids, sims, used, exact):
    """id recall against the exact lists, and the fraction of entries at or above the row's exact k-th similarity (every
    listed entry counts in the denominator, so entries the threshold rejected count as misses)."""
    eids, esims, eused = exact
    k = eids.shape[1]
    recall = float(np.isin(entry_keys(eids, eused), entry_keys(ids, used)).sum() / max(1, int(eused.sum())))
    kth = np.where(eused == k, esims[:, k - 1], -np.inf).astype(np.float64)
    mask = np.arange(ids.shape[1])[None, :] < used[:, None]
    above = int((sims.astype(np.float64) >= kth[:, None])[mask].sum())
    return recall, above


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--n", default="50000,200000,1000000")
    ap.add_argument("--widths", default="50,100,200,500,1000")
    ap.add_argument("--genes", type=int, default=20000)
    ap.add_argument("--nnz", type=int, default=1000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--threshold", type=float, default=0.2)
    ap.add_argument("--lsh-count", type=int, default=1024)
    ap.add_argument("--clusters", type=int, default=64)
    ap.add_argument("--exact-max", type=int, default=200000, help="largest N at which the full exact job runs")
    a = ap.parse_args()
    Ns = [int(x) for x in a.n.split(",")]
    widths = [int(x) for x in a.widths.split(",")]
    os.makedirs(a.outdir, exist_ok=True)
    result = {"gpu": gpu_info(), "genes": a.genes, "nnz_per_cell": a.nnz, "k": a.k, "threshold": a.threshold,
              "lsh_count": a.lsh_count, "clusters": a.clusters, "runs": a.runs, "cases": [], "skipped": []}
    G, k, thr, L = a.genes, a.k, a.threshold, a.lsh_count
    avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    U = em2.generate_lsh_vectors(G, L, 231)
    path = os.path.join(a.outdir, "rescore_time.json")
    with em2.Engine(0) as eng:
        for N in Ns:
            need = N * a.nnz * 8 * 3 + N * max(widths) * 8 * 3
            if need > avail:
                result["skipped"].append({"cells": N, "host_bytes_needed": need, "host_bytes_available": avail})
                print(json.dumps(result["skipped"][-1]), flush=True)
                continue
            toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, a.nnz, seed=N, clusters=a.clusters)
            pairs = synthetic.to_pairs(genes, counts)
            del genes, counts
            nnz = np.diff(toc).astype(np.int64)
            case = {"cells": N, "widths": []}
            exact = None
            if N <= a.exact_max:
                t = {"scan_ms": [], "total_ms": []}
                eng.exact_similar_pairs(toc, pairs, G, k, thr)
                for _ in range(a.runs):
                    exact = eng.exact_similar_pairs(toc, pairs, G, k, thr)
                    st = eng.stats()
                    t["scan_ms"].append(st["scan_ms"])
                    t["total_ms"].append(st["total_ms"])
                case["exact"] = {q: summary(v) for q, v in t.items()}
                print(json.dumps({"cells": N, "exact_scan_ms": case["exact"]["scan_ms"]["median"]}), flush=True)
            for w in widths:
                cids, _, cused = eng.lsh_similar_pairs(toc, pairs, U, w, thr)
                st = eng.stats()
                lsh = {"total_ms": st["total_ms"], "signatures_ms": st["signatures_ms"], "scan_ms": st["scan_ms"],
                       "scan_symmetric": st["scan_symmetric"]}
                t = {"scan_ms": [], "total_ms": []}
                first = eng.rescore_similar_pairs(toc, pairs, G, cids, cused, k, thr)
                equal = True
                for _ in range(a.runs):
                    got = eng.rescore_similar_pairs(toc, pairs, G, cids, cused, k, thr)
                    st = eng.stats()
                    t["scan_ms"].append(st["scan_ms"])
                    t["total_ms"].append(st["total_ms"])
                    equal = equal and all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(got, first))
                cand_bytes = int(nnz[cids[np.arange(w)[None, :] < cused[:, None]]].sum()) * 8
                row = {"width": w, "candidates": int(cused.sum()), "lsh": lsh, "rescore": {q: summary(v) for q, v in t.items()},
                       "outputs_equal_across_runs": equal, "variant_used": st["variant_used"],
                       "candidate_csr_bytes": cand_bytes,
                       "candidate_csr_bytes_per_s": cand_bytes / (1e-3 * float(np.median(t["scan_ms"])))}
                if exact is not None:
                    recall, above = quality(*got, exact)
                    row["id_recall"] = recall
                    row["above_kth"] = above / max(1, int(got[2].sum()))
                    if w == k:     # the plain LSH lists, with their entries' exact similarities (threshold -1 keeps them all)
                        full = eng.rescore_similar_pairs(toc, pairs, G, cids, cused, w, -1.0)
                        case["plain_lsh"] = {"id_recall": quality(cids, full[1], cused, exact)[0],
                                             "above_kth": quality(*full, exact)[1] / max(1, int(cused.sum()))}
                case["widths"].append(row)
                print(json.dumps({"cells": N, "width": w, "rescore_scan_ms": row["rescore"]["scan_ms"]["median"],
                                  "lsh_total_ms": lsh["total_ms"], "GB_per_s": row["candidate_csr_bytes_per_s"] / 1e9,
                                  "recall": row.get("id_recall"), "above_kth": row.get("above_kth"), "equal": equal}), flush=True)
                del cids, cused, got, first
            result["cases"].append(case)
            with open(path, "w") as f:          # partial results survive a later case running out of time
                json.dump(result, f, indent=1)
            del toc, pairs, exact, nnz
    with open(path, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
