#!/usr/bin/env python
"""bench.py -- LSH cell-similarity hot path on B200 (BASELINE.json metric: cell-pairs/sec).

A step = one pass of the hot path over the synthetic batch: per-cell sums -> LSH signatures ->
(all-gather when N>1) -> all-pairs Hamming scan with fused top-k -> SimilarPairs payload.
Workload (default "m1" = the configuration BASELINE.json's metric is quoted on): 1,000,000 cells x 30k genes, 5% density
(1500 stored counts per cell, 12 GB of CSR), L=1024, k=50, similarityThreshold 0.2, synthetic clustered counts (512
clusters; benchdata.py, generated on the device per rank), hyperplanes from seed 231.  `--workload c2` is
BASELINE.json configs[1] (100k cells), c1/c3/c4/c5 the other configs.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference          # the reference's own CPU code (oracle/_ref) on a bounded sample

`value`   : unordered cell pairs N(N-1)/2 per second of the whole job, inputs resident in HBM,
            CUDA-event timed, max over ranks.
`e2e`     : same metric through the reference-facing C-ABI call on HOST buffers (H2D + D2H inside).
`roofline`: the dominant kernel (the Hamming scan) against its governing pipe, measured live.

`--dump-outputs DIR` writes what the last timed step computed, for the cells listed in DIR/cells.npy (all cells, or a
seeded sample of them that keeps the files under 64 MB): neighbour_ids, similarities and used (the SimilarPairs rows),
and on the counts workloads also sum1, sum2 and signatures (each 64-bit signature word as two 32-bit halves, low
half first).  Inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: cells, genes, nnz/cell, L, k, threshold
    "m1": dict(cells=1_000_000, genes=30_000, nnz_per_cell=1500, lsh=1024, k=50, thr=0.2, clusters=512, hashed=True,
               note="the metric's configuration: 1M cells x 30k genes, 5% density, full counts -> lists pipeline"),
    "m1s": dict(cells=60_000, genes=30_000, nnz_per_cell=1500, lsh=1024, k=50, thr=0.2, clusters=32, hashed=True,
                note="reduced m1 for quick checks (NOT a bench line)"),
    "c1": dict(cells=10_000, genes=20_000, nnz_per_cell=1000, lsh=1024, k=50, thr=0.2,
               note="BASELINE configs[0]: 10k x 20k, 5% density"),
    "c2": dict(cells=100_000, genes=30_000, nnz_per_cell=1500, lsh=1024, k=50, thr=0.2,
               note="BASELINE configs[1]: 100k x 30k, 5% density"),
    "c3": dict(cells=1_300_000, genes=28_000, nnz_per_cell=2000, lsh=1024, k=50, thr=0.2, clusters=64, hashed=True,
               note="BASELINE configs[2]: 1.3M x 28k (10x mouse-brain shape, ~2.0k nnz/cell assumed), meant for 8 GPUs"),
    "c4": dict(kind="sig", cells=1_000_000, genes=0, lsh=1024, k=50, thr=0.2, clusters=500,
               note="BASELINE configs[3]: 1M cells, signatures-only synthetic (500 planted clusters, 12% bit flips); "
                    "--lsh 256/1024/4096 and --variant popc/mma give the sweep"),
    "c4s": dict(kind="sig", cells=200_000, genes=0, lsh=1024, k=50, thr=0.2, clusters=100,
                note="reduced c4 for quick checks (NOT a bench line)"),
    "c5": dict(kind="exact", cells=50_000, genes=20_000, nnz_per_cell=1000, lsh=0, k=50, thr=0.2,
               note="BASELINE configs[4]: exact Pearson brute force on 50k cells x 20k genes @ 5%"),
    "c2s": dict(cells=20_000, genes=30_000, nnz_per_cell=1500, lsh=1024, k=50, thr=0.2,
                note="reduced c2 for quick checks (NOT a bench line)"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


_INT8 = {}


def int8_peak(peaks, kernel_ms, device_index=0):
    """Tensor-pipe roofline denominator of the int8 scan, MEASURED: tools/mma_peak.cu (back-to-back
    tcgen05.mma.kind::i8 M=128 N=256 K=32, A in tensor memory -- the highest int8 issue rate the pipe gives) run live on
    this GPU; else the committed run of the same tool (profiles/r2_mma_peak.json); else 2 x the bf16 figure of
    MEASURED_PEAKS.json.  Burst figure for a kernel timed alone, sustained (power-capped clocks) for one that runs
    for more than ~100 ms at a time (B200_PROFILING.md)."""
    which = "sustained" if kernel_ms > 100.0 else "burst"
    if not _INT8:
        exe = os.path.join(ROOT, "expressionmatrix2_b200", "build", "mma_peak")
        try:
            out = subprocess.check_output([exe], env=dict(os.environ, CUDA_VISIBLE_DEVICES=str(device_index)), timeout=120).decode()
            _INT8.update(json.loads(out), source="tools/mma_peak.cu run live on this GPU by bench.py")
        except Exception:
            try:
                _INT8.update(json.load(open(os.path.join(ROOT, "profiles", "r2_mma_peak.json"))),
                             source="profiles/r2_mma_peak.json (tools/mma_peak.cu, committed run)")
            except Exception:
                _INT8.update(source="fallback")
    key = "i8_ts_n256_tops_sustained" if which == "sustained" else "i8_ts_n256_tops"
    if _INT8.get(key):
        note = (f"{key} = {_INT8[key]} TOP/s, {_INT8['source']}; same run: operands in shared memory N=256 "
                f"{_INT8.get('i8_ss_n256_tops')} (the scan kernels' instruction shape), sustained "
                f"{_INT8.get('i8_ss_n256_tops_sustained')}; bf16 {_INT8.get('bf16_ss_n256_tflops')}")
        return float(_INT8[key]), which, note
    bf = peaks["bf16_tflops_sustained"] if which == "sustained" else peaks["bf16_tflops"]
    return 2.0 * bf, which, f"2 x bf16 TF/s of MEASURED_PEAKS.json ({peaks['source']}, {which}): tools/mma_peak could not run"


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                    samples=len(sm))


def _synthetic_module():
    """expressionmatrix2_b200/synthetic.py loaded by path: the numpy generators of the small workloads without
    importing the product package (the reference arm must not touch it)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_em2_synthetic", os.path.join(ROOT, "expressionmatrix2_b200", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def host_counts(w, cell_begin, cell_end, seed=12345):
    """(toc, gene_ids, counts) of cells [cell_begin, cell_end) of the workload, on the host."""
    if w.get("hashed"):
        import benchdata as bd
        g, c = bd.counts_to_numpy(bd.gen_counts(cell_begin, cell_end, w["genes"], w["nnz_per_cell"], seed=seed,
                                                clusters=w["clusters"]))
        return bd.toc_of(cell_end - cell_begin, w["nnz_per_cell"]), g, c
    toc, genes, counts = _synthetic_module().gen_expression_matrix_fast(w["cells"], w["genes"], w["nnz_per_cell"], seed=seed)
    b, e = int(toc[cell_begin]), int(toc[cell_end])
    return (toc[cell_begin:cell_end + 1] - toc[cell_begin]).astype(np.uint64), genes[b:e], counts[b:e]


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref), bounded sample per step
# ------------------------------------------------------------------------------------------------
def cpu_sample(w, head, signatures, loop_rows, lsh=None):
    """Times the reference's two instrumented regions on a bounded sample of the workload:
    Lsh::computeCellLshSignatures on the cells of `head` = (toc, genes, counts) of the first cells (its own timer,
    Lsh.cpp:160,209) and the findSimilarPairs4 pair loop (ExpressionMatrixLsh.cpp:217,270) for the last `loop_rows`
    cells against all earlier cells.  Returns the extrapolated whole-job figures.  head=None: signatures-only
    workload (config 4), only the pair loop is timed."""
    import oracle
    N, L, k, thr = w["cells"], lsh or w["lsh"], w["k"], w["thr"]
    kind = "reference" if oracle.have_ref() else "port"
    loop_rows = min(loop_rows, N)
    t0 = time.time()
    t_sig, ref_sig, sig_cells = 0.0, None, 0
    if head is not None:
        toc, genes, counts = head
        sig_cells = len(toc) - 1
        if kind == "reference":
            with oracle.Reference.from_csr(toc, genes, counts, w["genes"], L, 231) as R:
                t_sig = R.signature_seconds
                ref_sig = R.signatures()
        else:
            U = oracle.generate_lsh_vectors(w["genes"], L, 231)
            s1, _ = oracle.cell_sums(toc, counts)
            t1 = time.time()
            ref_sig, _ = oracle.signatures(toc, genes, counts, s1, U)
            t_sig = time.time() - t1
    if kind == "reference":
        with oracle.Reference.from_signatures(signatures, L) as R:
            r = R.find_similar_pairs4_loop(k, thr, N - loop_rows, N, want_pairs=False)
            t_loop, pairs = r["seconds"], r["pairs"]
    else:
        t_loop, pairs, _ = oracle.pair_loop(signatures, L, thr, N - loop_rows, N)
    total_pairs = N * (N - 1) / 2
    sig_s_per_cell = t_sig / max(sig_cells, 1)
    ns_per_pair = 1e9 * t_loop / max(pairs, 1)
    full_seconds = sig_s_per_cell * N + ns_per_pair * 1e-9 * total_pairs
    what = (f"signatures of the first {sig_cells} cells + " if head is not None else "")
    out = dict(value=total_pairs / full_seconds, unit="cell-pairs/s", cores=1, kind=kind,
               sample=what + f"findSimilarPairs4 pair loop for the last {loop_rows} cells x all earlier cells "
                             f"({pairs} pairs), extrapolated to the whole job",
               ns_per_pair=ns_per_pair, signature_s_per_cell=sig_s_per_cell, extrapolated_job_seconds=full_seconds,
               sample_seconds=time.time() - t0)
    if ref_sig is not None:
        out["_ref_sig"] = ref_sig
    return out


def sample_sizes(N, per_step=False):
    """Bounded CPU samples (about 15 s for the cpu_baseline leg, about 2 s per step of the reference arm):
    (cells whose signatures the reference computes, rows of the pair loop)."""
    budget = 1.0e8 if per_step else 1.0e9           # pair evaluations at ~13 ns each
    rows = int(max(16, min(2048, budget // max(N, 1))))
    return (128 if per_step else 1024), rows


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path returned in its last step, so that two builds can be compared output for output
# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 60_000_000          # array bytes; with the .npy headers the files stay under 64 MB in all


def dump_rows(n: int, bytes_per_row: int) -> np.ndarray:
    """Cells whose outputs are written: all of them when they fit, else a sorted sample drawn with a fixed seed, so that
    runs with the same arguments write the same cells."""
    r = min(n, DUMP_BYTES // bytes_per_row)
    if r == n:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(n, r, replace=False)).astype(np.int64)


def list_outputs(pairs, used):
    """SimilarPairs rows (pairs int32 [R, k, 2] = cell id, float bits; used [R]) as float arrays.  Entries past a row's
    used count are not part of the result and are written as 0."""
    import torch
    valid = torch.arange(pairs.shape[1], device=pairs.device)[None, :] < used.to(torch.int64)[:, None]
    ids = torch.where(valid, pairs[..., 0].to(torch.int64) & 0xFFFFFFFF, 0).to(torch.float64)
    sims = torch.where(valid, pairs[..., 1].contiguous().view(torch.float32), 0.0)
    return dict(neighbour_ids=ids, similarities=sims, used=used.to(torch.float64))


def write_dump(directory: str, arrays: dict) -> None:
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a))


def run_reference(args, w):
    """The reference's own CPU code (oracle/_ref; the C port when the reference build is absent) on a bounded sample
    of the same workload per step, one core (the reference is single threaded).  Imports nothing of the product:
    counts from the bench generators, hyperplanes from the reference's own Lsh constructor, and -- for the pair
    loop, which needs the signatures of ALL cells -- synthetic signatures with the workload's cluster structure."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    import benchdata as bd
    oracle.build()
    kind = w.get("kind", "lsh")
    N, L = w["cells"], args.lsh or w["lsh"]
    samples = []
    if kind == "exact":
        G = w["genes"]
        toc, genes, counts = host_counts(w, 0, N)
        s1, s2 = oracle.cell_sums(toc, counts)
        for i in range(args.warmup + args.steps):
            t0 = time.time()
            oracle.exact_rows(G, toc, genes, counts, s1, s2, 4 * i, 4 * i + 4)
            dt = time.time() - t0
            if i >= args.warmup:
                samples.append(dict(value=4 * N / dt, wall_ms=1e3 * dt, kind="port", ns_per_pair=1e9 * dt / (4 * N),
                                    signature_s_per_cell=0.0, extrapolated_job_seconds=N * (N - 1) / 2 / (4 * N / dt),
                                    sample=f"computeCellSimilarity for 4 cells against all {N} cells ({4 * N} pairs)"))
        sig_note = "n/a (exact path)"
        metric = "cell-pairs/sec (exact Pearson, top-50)"
    else:
        sig_cells, loop_rows = sample_sizes(N, per_step=True)
        head = host_counts(w, 0, min(sig_cells, N)) if kind == "lsh" else None
        signatures = bd.gen_signatures(0, N, L, clusters=w.get("clusters", 64)).numpy().view(np.uint64)
        sig_note = ("pair loop on synthetic signatures with the workload's cluster structure (benchdata.gen_signatures); "
                    "signature timing on the workload's own counts")
        for i in range(args.warmup + args.steps):
            t0 = time.time()
            sm = cpu_sample(w, head, signatures, loop_rows, lsh=L)
            sm.pop("_ref_sig", None)
            sm["wall_ms"] = 1e3 * (time.time() - t0)
            if i >= args.warmup:
                samples.append(sm)
        metric = "cell-pairs/sec (1024-bit LSH, top-50)"
    value = float(np.median([sm["value"] for sm in samples]))
    best = samples[0]
    line = dict(impl="reference", metric=metric, value=value, unit="cell-pairs/s",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=float(np.mean([sm["wall_ms"] for sm in samples])), higher_is_better=True,
                scaling="strong", vs_baseline=None, dtype="u64 popcount + f64 projections" if kind != "exact" else "f32 products, f64 sums",
                data="synthetic",
                config=dict(workload=args.workload, cells=N, genes=w["genes"], nnz_per_cell=w.get("nnz_per_cell"), lsh=L,
                            k=w["k"], thr=w["thr"], note=w["note"], signatures=sig_note),
                cpu_baseline=dict(kind=best["kind"], cores=1, value=value, unit="cell-pairs/s", sample=best["sample"],
                                  ns_per_pair=best["ns_per_pair"], signature_s_per_cell=best["signature_s_per_cell"],
                                  extrapolated_job_seconds=best["extrapolated_job_seconds"]),
                e2e=dict(value=value, unit="cell-pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def _setup_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local_rank, dev


def _timed_steps(args, world, dev, local_rank, step, n_marks, launch_counter=None, after_timed=None):
    """W warm-up steps, then exactly K steps bracketed by barrier + synchronize; CUDA events; max over ranks.
    `after_timed` runs once right after the K-th step, before any untimed step can overwrite its outputs."""
    import torch
    import torch.distributed as dist

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # nvidia-smi samples every 100 ms; a multi-GPU step of this workload can be a few ms, so the sampler also covers the
    # warm-up steps (same kernels, same clocks) -- otherwise a short timed region would end before its first sample
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(n_marks)] for _ in range(args.steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = launch_counter() if launch_counter else 0
    t_begin.record()
    for i in range(args.steps):
        step(ev[i])
    t_end.record()
    launches = (launch_counter() - launches0) if launch_counter else 0      # kernels of this library enqueued by the K timed steps
    barrier()
    if after_timed:
        after_timed()
    total_ms = t_begin.elapsed_time(t_end)
    if total_ms < 300.0:          # keep the GPU busy with the same step until the sampler has something to report
        t0 = time.time()
        while time.time() - t0 < 0.35:
            step()
        torch.cuda.synchronize()
    clocks = sampler.stop()
    clocks["window"] = "warm-up + timed steps" + (" + identical extra steps (timed region shorter than the 100 ms sampling period)" if total_ms < 300.0 else "")
    stage = [float(np.mean([ev[i][j].elapsed_time(ev[i][j + 1]) for i in range(args.steps)])) for j in range(n_marks - 1)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / args.steps, stage, clocks, barrier, launches


def _scan_roofline(em2, eng, peaks, variant, variant_used, rows, N, L, W, k, world, pairs_total, scan_ms, local_rank,
                   symmetric=False):
    scan_s = scan_ms * 1e-3
    ordered = rows * N                      # pair evaluations this GPU executed per launch
    if symmetric:      # every unordered pair once: near window (2w + 1 tiles of 256 columns, both owners) + offsets w+1 .. S/2
        S = (N + 255) // 256
        wn = max(16, (N // 32 + 511) // 512)
        wn = min(wn, (S - 1) // 2)
        ordered = rows * 256.0 * (2 * wn + 1 + max(0, S // 2 - wn))
    alg_pairs = pairs_total / world         # algorithmic units per GPU per launch
    if variant_used == em2.VARIANT_MMA_I8:
        peak, which, note = int8_peak(peaks, scan_ms, local_rank)
        K = (L + 127) // 128 * 128
        roof = dict(bound="tensor", unit="TOP/s", achieved=alg_pairs * 2 * L / scan_s / 1e12, peak=peak,
                    peak_source=note,
                    executed=ordered * 2 * K / scan_s / 1e12)
    else:
        mb = os.path.join(ROOT, "expressionmatrix2_b200", "build", "microbench")
        popc_peak = None
        try:
            popc_peak = json.loads(subprocess.check_output([mb], env=dict(os.environ, CUDA_VISIBLE_DEVICES=str(local_rank))).decode())["popc_per_s"]
        except Exception:
            pass
        popc_peak = popc_peak or 4.6e12
        # algorithmic unit = one unordered pair = 2W 32-bit popcount-words (SURVEY.md 8d)
        # the kernel folds three words into two POPCs with carry-save adders: (2W * 2 / 3, rounded up) + 1 POPC per ordered pair
        popc_per_pair = (2 * W * 2 + 2) // 3 + 1
        roof = dict(bound="alu", unit="Gpopc32/s", achieved=alg_pairs * 2 * W / scan_s / 1e9, peak=popc_peak / 1e9,
                    peak_source="POPC.b32 issue rate measured by tools/microbench.cu on this GPU",
                    executed=ordered * popc_per_pair / scan_s / 1e9)
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["executed_frac"] = roof["executed"] / roof["peak"]
    roof["kernel"] = "scan_topk (encode + scanMmaKernel/scanPopc*Kernel + finalize)"
    roof["kernel_ms"] = scan_ms
    roof["traffic"] = None      # filled by the caller from profiles/r2_traffic.json (ncu --set full captures)
    roof["note"] = ("achieved = algorithmic ops (one evaluation per UNORDERED pair, 2L bit-ops each); executed = what the "
                    "row-block design runs (every ordered pair): executed_frac is the kernel-quality figure, frac is capped "
                    "at half of it")
    alg_bytes = N * L / 8 + rows * L / 8 + rows * (8 * k + 4)
    roof["hbm"] = dict(bound="hbm", unit="GB/s", algorithmic_bytes=alg_bytes, achieved=alg_bytes / scan_s / 1e9,
                       peak=peaks["hbm_gbs"], frac=alg_bytes / scan_s / 1e9 / peaks["hbm_gbs"],
                       note="compulsory bytes only; the scan is compute bound by construction")
    return roof


def run_b200(args, w):
    import torch
    import torch.distributed as dist
    import expressionmatrix2_b200 as em2
    from expressionmatrix2_b200 import synthetic
    from expressionmatrix2_b200.parallel import Partition, all_gather_signatures

    world, rank, local_rank, dev = _setup_dist()
    variant = dict(auto=em2.VARIANT_AUTO, popc=em2.VARIANT_POPC, mma=em2.VARIANT_MMA_I8)[args.variant]
    kind = w.get("kind", "lsh")
    N, G, k, thr = w["cells"], w["genes"], w["k"], w["thr"]
    L = args.lsh or w["lsh"]
    W = em2.word_count(L)
    part = Partition(N, world, rank)          # same rule as em2_dist_partition
    assert (part.row_begin, part.row_end, part.shard) == em2.dist_partition(N, world, rank)
    rows = part.rows
    eng = em2.Engine(local_rank)
    cpu_group = None
    if world > 1:
        # torch.distributed is the plumbing: it carries the library's communicator id to the ranks; the collectives of
        # the data path (signature all-gather, candidate exchange) run inside libem2b200 on its own NCCL communicator
        ident = [em2.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        eng.comm_init(ident[0], rank, world)
        cpu_group = dist.new_group(backend="gloo")      # host-side waits that must not put a spinning kernel on the GPUs
    if args.symmetric:
        eng.set_option("scan_symmetric", 2)
    if args.one_directional:
        eng.set_option("scan_symmetric", 1)
    for nv in args.option:
        name, value = nv.split("=")
        eng.set_option(name, int(value))
    stream = torch.cuda.current_stream().cuda_stream
    peaks = load_peaks()
    pairs_total = N * (N - 1) / 2
    cfg = dict(workload=args.workload, cells=N, genes=G, nnz_per_cell=w.get("nnz_per_cell"), lsh=L, k=k, thr=thr,
               note=w["note"])
    line = dict(metric="cell-pairs/sec (1024-bit LSH, top-50)", unit="cell-pairs/s", n_gpus=world, steps=args.steps,
                warmup=args.warmup, higher_is_better=True, scaling="strong", vs_baseline=None, data="synthetic")

    if kind == "exact":
        # ---------------- config 5: exact Pearson brute force (single GPU; N>1 = replicas of the row blocks) ------
        if world > 1:
            raise SystemExit("the exact workload (config 5) is a single-GPU validation run")
        toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, w["nnz_per_cell"], seed=12345)
        lpairs = em2.to_pairs(genes, counts)
        p_toc = torch.from_numpy(toc.view(np.int64)).pin_memory()
        p_counts = torch.from_numpy(lpairs.view(np.int64)).pin_memory()
        h_pairs = torch.empty((N, k, 2), dtype=torch.int32).pin_memory()
        h_used = torch.empty(N, dtype=torch.int32).pin_memory()
        n_toc, n_counts = p_toc.numpy().view(np.uint64), p_counts.numpy().view(em2.PAIR_DTYPE)
        sampler = ClockSampler(local_rank)
        ms, st = [], None
        for i in range(args.warmup + args.steps):
            if i == args.warmup:
                sampler.start()
            t0 = time.perf_counter()
            eng.exact_similar_pairs_into(n_toc, n_counts, G, k, thr, h_pairs.numpy().view(em2.SIMPAIR_DTYPE).reshape(N, k),
                                         h_used.numpy().view(np.uint32))
            if i >= args.warmup:
                ms.append(1e3 * (time.perf_counter() - t0))
            st = eng.stats()
        clocks = sampler.stop()
        if args.dump_outputs:
            cells = torch.from_numpy(dump_rows(N, 8 + 12 * k + 8))
            write_dump(args.dump_outputs, dict({n: t.numpy() for n, t in list_outputs(h_pairs[cells], h_used[cells]).items()},
                                               cells=cells.numpy().astype(np.float64)))
        e2e_t = float(np.mean(ms))
        dev_ms = st["sums_ms"] + st["scan_ms"]
        Gpad = (G + 127) // 128 * 128
        peak, which, peak_note = int8_peak(peaks, st["scan_ms"], local_rank)
        roof = dict(bound="tensor", unit="TOP/s", achieved=pairs_total * 2 * G / (st["scan_ms"] * 1e-3) / 1e12,
                    # the N x N float matrix fits (<= 48 GB) for N <= ~109k: only tiles on or above the diagonal are computed
                    executed=(float(N) * N / 2 + 128.0 * N if 4.0 * N * N <= 48 * 2 ** 30 else float(N) * N) * 2 * Gpad
                    / (st["scan_ms"] * 1e-3) / 1e12, peak=peak,
                    peak_source=peak_note, kernel="exactGemmKernel + exactSelectKernel",
                    kernel_ms=st["scan_ms"], traffic=None)
        roof["frac"] = roof["achieved"] / peak
        roof["executed_frac"] = roof["executed"] / peak
        line.update(metric="cell-pairs/sec (exact Pearson, top-50)", value=pairs_total / (dev_ms * 1e-3), ms_per_step=dev_ms,
                    dtype="u8 x u8 -> s32 tcgen05 (scalar products), f64 (correlation)", config=dict(cfg, variant="exact"),
                    stage_ms=dict(sums=st["sums_ms"], exact=st["scan_ms"]), roofline=roof,
                    e2e=dict(value=pairs_total / (e2e_t * 1e-3), unit="cell-pairs/s", ms=e2e_t, h2d_bytes_per_step=int(st["h2d_bytes"]),
                             d2h_bytes_per_step=int(st["d2h_bytes"]), api="em2_exact_similar_pairs (C-ABI, host buffers)"),
                    gpu_launches=int(st["kernel_launches"]) * args.steps, clocks=clocks)
        # ---- what config 5 is for: the LSH path's neighbour recall against the exact lists, at the config's 50k cells
        exact_pairs = h_pairs.numpy().view(em2.SIMPAIR_DTYPE).reshape(N, k).copy()
        exact_used = h_used.numpy().view(np.uint32).copy()
        Lr = 1024
        U = em2.generate_lsh_vectors(G, Lr, 231)
        lids, lsims, lused = eng.lsh_similar_pairs(toc, lpairs, U, k, thr)
        lsh_ms = eng.stats()["total_ms"]
        hits = pairs_in_both = 0
        err2 = 0.0
        sample_rows = np.arange(0, N, max(1, N // 5000))
        for c in sample_rows:
            e_ids = exact_pairs["cell"][c, :exact_used[c]]
            l_ids = lids[c, :lused[c]]
            common, ei, li = np.intersect1d(e_ids, l_ids, return_indices=True)
            hits += len(common)
            pairs_in_both += len(common)
            err2 += float(np.sum((lsims[c, li].astype(np.float64) - exact_pairs["similarity"][c, ei].astype(np.float64)) ** 2))
        denom = int(np.sum(np.minimum(exact_used[sample_rows], k)))
        line["recall"] = dict(cells=N, lsh_bits=Lr, k=k, sampled_rows=int(len(sample_rows)),
                              recall_at_k=hits / max(denom, 1),
                              note="fraction of the exact top-k (Pearson > threshold) that the 1024-bit LSH top-k contains; on tightly "
                                   "clustered synthetic data many mates are equally near, so id-set recall understates list quality",
                              rms_similarity_error_of_common_pairs=(err2 / max(pairs_in_both, 1)) ** 0.5,
                              theoretical_sigma_max=float(np.pi / (2 * np.sqrt(Lr))),
                              mean_stored_exact=float(exact_used.mean()), mean_stored_lsh=float(lused.mean()),
                              lsh_job_ms_host_buffers=lsh_ms)
        if not args.no_cpu_baseline:
            import oracle
            oracle.build()
            s1, s2 = oracle.cell_sums(toc, counts)
            t0 = time.time()
            r = oracle.exact_rows(G, toc, genes, counts, s1, s2, 0, 4)
            dt = time.time() - t0
            ids_np = h_pairs.numpy().view(em2.SIMPAIR_DTYPE).reshape(N, k)
            wi, ws, wu, _ = oracle.exact_topk(G, toc, genes, counts, k, thr, 0, 4)
            line["cpu_baseline"] = dict(value=4 * N / dt, unit="cell-pairs/s", cores=1, kind="port",
                                        sample=f"computeCellSimilarity for cells 0..3 against all {N} cells ({4 * N} pairs)",
                                        extrapolated_job_seconds=pairs_total / (4 * N / dt),
                                        sample_rows_match_gpu=bool(np.array_equal(wi, ids_np["cell"][:4]) and
                                                                   np.array_equal(ws.view(np.uint32), ids_np["similarity"][:4].view(np.uint32))))
        print(json.dumps(line))
        eng.close()
        return

    # ---------------- LSH workloads: "lsh" (counts -> lists) and "sig" (signatures-only scan, config 4) -----------
    import benchdata as bd
    hashed = bool(w.get("hashed"))
    d_lut = torch.from_numpy(em2.similarity_table(L).astype(np.float32)).to(dev)
    d_pairs = torch.zeros((rows, k, 2), dtype=torch.int32, device=dev)
    d_used = torch.zeros(rows, dtype=torch.int32, device=dev)
    d_sig_local = torch.zeros((part.shard, W), dtype=torch.int64, device=dev)
    mm = em2.mismatch_max(L, thr)
    if kind == "lsh":
        m = w["nnz_per_cell"]
        if hashed:
            # every rank synthesises its own cells on its GPU (the 1M-cell CSR is 12 GB); benchdata is counter based, so
            # any other rank / the host can reproduce any range of cells
            d_counts = torch.empty(rows * m, dtype=torch.int64, device=dev)
            step_cells = 20_000
            for b0 in range(part.row_begin, part.row_end, step_cells):
                e0 = min(part.row_end, b0 + step_cells)
                d_counts[(b0 - part.row_begin) * m:(e0 - part.row_begin) * m] = bd.gen_counts(
                    b0, e0, G, m, clusters=w["clusters"], device=dev)
            d_toc = torch.arange(rows + 1, dtype=torch.int64, device=dev) * m
            nnz_local = rows * m
        else:
            toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, m, seed=12345)
            ltoc, lgenes, lcounts = part.slice_csr(toc, genes, counts)
            lpairs = em2.to_pairs(lgenes, lcounts)
            nnz_local = int(ltoc[-1])
            d_toc = torch.from_numpy(ltoc.view(np.int64)).to(dev)
            d_counts = torch.from_numpy(lpairs.view(np.int64)).to(dev)
        U = em2.generate_lsh_vectors(G, L, 231)
        d_U = torch.from_numpy(U).to(dev)
        d_sum1 = torch.empty(rows, dtype=torch.float64, device=dev)
        d_sum2 = torch.empty(rows, dtype=torch.float64, device=dev)
        d_nz = torch.zeros(8, dtype=torch.int64, device=dev)
    else:
        d_sig_local[:rows] = bd.gen_signatures(part.row_begin, part.row_end, L, clusters=w.get("clusters", 500), device=dev)
    torch.cuda.empty_cache()

    if kind == "lsh":
        stage_names = ["sums", "signatures", "scan_topk"]
    else:
        stage_names = ["scan_topk"]

    def step(events=None):
        def mark(i):
            if events is not None:
                events[i].record()
        j = 0
        mark(j)
        if kind == "lsh":
            eng.cell_sums_device(rows, d_toc, d_counts, d_sum1, d_sum2, stream=stream)
            j += 1
            mark(j)
            eng.signatures_device(rows, G, d_toc, d_counts, d_sum1, d_sum2, d_U, L, L, d_sig_local, d_nz, stream=stream,
                                  nnz=nnz_local)
            j += 1
            mark(j)
        if world > 1:      # collective: signature all-gather (+ the symmetric scan's exchange) on NCCL inside the library
            eng.scan_topk_dist_device(d_sig_local, N, L, k, mm, d_lut, d_pairs, d_used, variant=variant, stream=stream)
        else:
            eng.scan_topk_device(d_sig_local, N, L, 0, N, k, mm, d_lut, d_pairs, d_used, variant=variant, stream=stream)
        j += 1
        mark(j)

    dump = {}

    def take_outputs():
        """Lists (and, from counts, the sums and signatures) of the sampled cells; each rank contributes the cells it owns."""
        cells = torch.from_numpy(dump_rows(N, 8 + 12 * k + 8 + (16 + 16 * W if kind == "lsh" else 0))).to(dev)
        mine = (cells >= part.row_begin) & (cells < part.row_end)
        at = (cells - part.row_begin).clamp(0, max(rows - 1, 0))
        pick = (lambda t: t[at]) if rows else (lambda t: t.new_zeros((len(cells),) + t.shape[1:]))
        out = list_outputs(pick(d_pairs), pick(d_used))
        if kind == "lsh":      # signature words as their two 32-bit halves, low half first
            out.update(sum1=pick(d_sum1), sum2=pick(d_sum2),
                       signatures=(pick(d_sig_local).view(torch.int32).to(torch.int64) & 0xFFFFFFFF).to(torch.float64))
        for name, t in out.items():
            t = torch.where(mine.view(-1, *[1] * (t.dim() - 1)), t, 0)
            if world > 1:      # every cell is owned by exactly one rank
                dist.all_reduce(t)
            dump[name] = t.cpu().numpy()
        dump["cells"] = cells.cpu().numpy().astype(np.float64)

    ms_per_step, stage, clocks, barrier, launches = _timed_steps(args, world, dev, local_rank, step, len(stage_names) + 1,
                                                                 launch_counter=lambda: eng.stats()["kernel_launches"],
                                                                 after_timed=take_outputs if args.dump_outputs else None)
    if dump and rank == 0:
        write_dump(args.dump_outputs, dump)
    stage_ms = dict(zip(stage_names, stage))
    value = pairs_total / (ms_per_step * 1e-3)
    if world > 1:      # one more step, bracketed by the library's own events: the collectives inside scan_topk
        torch.cuda.synchronize()
        s0 = eng.stats()
        step()
        torch.cuda.synchronize()
        s1 = eng.stats()
        stage_ms["allgather_inside_scan_topk"] = s1["allgather_ms"] - s0["allgather_ms"]
        stage_ms["exchange_inside_scan_topk"] = s1["exchange_ms"] - s0["exchange_ms"]
        stage_ms["exchange_bytes_sent_rank0"] = int(s1["exchange_bytes"] - s0["exchange_bytes"])
    variant_used = eng.stats()["variant_used"] or (em2.VARIANT_POPC if variant != em2.VARIANT_MMA_I8 else variant)
    sym_used = int(eng.stats()["scan_symmetric"])
    used_mean = float(d_used.float().mean().item()) if rows else 0.0

    # ---- e2e: host buffers -> host lists ----------------------------------------------------------
    # One blocking library call on HOST buffers, as the reference's host layer makes it: em2_lsh_similar_pairs on one
    # GPU, em2_multi_lsh_similar_pairs over all N GPUs (rank 0 drives them from one process, exactly like the C++
    # ExpressionMatrix::findSimilarPairs4 of host/; the other ranks have released their GPUs and wait on the host).
    e2e_t, h2d, d2h, api, e2e_stats = float('nan'), 0, 0, 'skipped (--no-e2e)', {}
    sig_all_host = None
    if not args.no_e2e:
        own_pairs = d_pairs.cpu()
        own_used = d_used.cpu()
        sig_all_host = d_sig_local[:rows].cpu().numpy().view(np.uint64) if world == 1 else None
        if kind == "lsh":
            n_toc = (np.arange(N + 1, dtype=np.uint64) * np.uint64(m)) if hashed else toc
            if rank == 0:
                p_counts = torch.empty(int(n_toc[-1]), dtype=torch.int64).pin_memory()
                if hashed:
                    if world == 1:
                        p_counts.copy_(d_counts)
                    else:      # rank 0 needs the whole job's counts on the host: regenerate the other ranks' cells here
                        for b0 in range(0, N, 20_000):
                            e0 = min(N, b0 + 20_000)
                            p_counts[b0 * m:e0 * m].copy_(bd.gen_counts(b0, e0, G, m, clusters=w["clusters"], device=dev))
                else:
                    p_counts.copy_(torch.from_numpy(em2.to_pairs(genes, counts).view(np.int64)))
                p_toc = torch.from_numpy(n_toc.view(np.int64)).pin_memory()
                p_U = torch.from_numpy(U).pin_memory()
        elif rank == 0:
            p_sig = torch.empty((N, W), dtype=torch.int64).pin_memory()
            for b0 in range(0, N, 100_000):
                e0 = min(N, b0 + 100_000)
                p_sig[b0:e0].copy_(bd.gen_signatures(b0, e0, L, clusters=w.get("clusters", 500), device=dev))
        # release the device-resident leg's memory on every rank before the library allocates its own
        eng.close()
        del d_pairs, d_used, d_sig_local
        if kind == "lsh":
            del d_counts, d_toc, d_U, d_sum1, d_sum2
        torch.cuda.empty_cache()
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier(group=cpu_group)
        if rank == 0:
            h_pairs = torch.empty((N, k, 2), dtype=torch.int32).pin_memory()
            h_used = torch.empty(N, dtype=torch.int32).pin_memory()
            o_pairs = h_pairs.numpy().view(em2.SIMPAIR_DTYPE).reshape(N, k)
            o_used = h_used.numpy().view(np.uint32)
            runner = em2.Engine(local_rank) if world == 1 else em2.MultiEngine(devices=list(range(world)))
            if args.symmetric:
                runner.set_option("scan_symmetric", 2)
            if args.one_directional:
                runner.set_option("scan_symmetric", 1)
            for nv in args.option:
                name, value = nv.split("=")
                runner.set_option(name, int(value))
            if kind == "lsh":
                a_toc, a_counts, a_U = p_toc.numpy().view(np.uint64), p_counts.numpy().view(em2.PAIR_DTYPE), p_U.numpy()
                call = lambda: runner.lsh_similar_pairs_into(a_toc, a_counts, a_U, k, thr, o_pairs, o_used, variant=variant)
                api = ("em2_lsh_similar_pairs" if world == 1 else f"em2_multi_lsh_similar_pairs over {world} GPUs") + " (C-ABI, host buffers)"
            else:
                a_sig = p_sig.numpy().view(np.uint64)
                call = lambda: runner.find_similar_pairs_into(a_sig, L, k, thr, o_pairs, o_used, variant=variant)
                api = ("em2_find_similar_pairs" if world == 1 else f"em2_multi_find_similar_pairs over {world} GPUs") + " (C-ABI, host buffers)"
            e2e_ms, st = [], None
            for i in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                call()
                if i >= args.warmup:
                    e2e_ms.append(1e3 * (time.perf_counter() - t0))
                st = runner.stats()
            e2e_t = float(np.mean(e2e_ms))
            h2d, d2h = int(st["h2d_bytes"]), int(st["d2h_bytes"])
            e2e_stats = {k2: st[k2] for k2 in ("h2d_ms", "sums_ms", "signatures_ms", "scan_ms", "d2h_ms", "allgather_ms", "exchange_ms")}
            e2e_stats["note"] = ("per-stage times are device-side maxima over the GPUs; h2d overlaps sums/signatures (chunked copy "
                                 "stream); inputs and outputs are pinned host buffers")
            e2e_stats["scan_symmetric"] = int(st["scan_symmetric"])
            # the host-buffer call and the device-resident steps must have produced the same lists (rank 0's rows)
            e2e_stats["lists_equal_device_path"] = bool(
                torch.equal(h_pairs[part.row_begin:part.row_end], own_pairs) and torch.equal(h_used[part.row_begin:part.row_end], own_used))
            runner.close()
        if world > 1:
            dist.barrier(group=cpu_group)

    # ---- rooflines ---------------------------------------------------------------------------------
    roof = _scan_roofline(em2, eng, peaks, variant, variant_used, rows, N, L, W, k, world, pairs_total,
                          stage_ms["scan_topk"], local_rank, symmetric=(sym_used == 1))
    if sym_used == 1:
        roof["kernel"] = "scan_topk (grouping + encode + scanMmaSymKernel near window and far sweep + scatter + merge)"
        roof["note"] = ("symmetric scan: achieved = algorithmic ops (one evaluation per unordered pair, 2L bit-ops); executed adds "
                        "the near window, whose tiles both owners evaluate")
    try:       # DRAM bytes per launch of the dominant kernel, from the committed ncu --set full capture of this workload
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        ent = tr.get(f"{args.workload}@L{L}@n{world}@sym{1 if sym_used == 1 else 0}")
        if ent:
            roof["traffic"] = ent["bytes"]
            roof["traffic_kernel"] = ent["kernel"]
            roof["traffic_source"] = ent["source"]
    except Exception:
        pass
    sig_roof = None
    if kind == "lsh":
        sig_s = stage_ms["signatures"] * 1e-3
        sig_bytes = 8 * nnz_local + 8 * (rows + 1) + 8 * rows + 8 * G * L + rows * L / 8
        density = nnz_local / (rows * float(G))
        filtered = density >= 0.012 and rows >= 4096 and G >= 1024 and L >= 128
        sig_roof = dict(kernel="signatures (columnStats + quantize + densify + sigFilterKernel + fixup)" if filtered
                        else "signatures (columnStats + signatureKernel, FP64)",
                        path="tensor-core filter + FP64 fix-up" if filtered else "fp64",
                        kernel_ms=stage_ms["signatures"], flops=2.0 * nnz_local * L,
                        achieved_gflops=2.0 * nnz_local * L / sig_s / 1e9, algorithmic_bytes=sig_bytes,
                        achieved_gbs=sig_bytes / sig_s / 1e9, hbm_frac=sig_bytes / sig_s / 1e9 / peaks["hbm_gbs"])
        if filtered:
            Gpad, Lp = (G + 127) // 128 * 128, (L + 127) // 128 * 128
            ex = 2.0 * rows * Gpad * 3 * Lp
            pk, _, pk_note = int8_peak(peaks, stage_ms["signatures"], local_rank)
            sig_roof.update(bound="tensor", executed_int8_tops=ex / sig_s / 1e12, peak=pk, peak_source=pk_note,
                            executed_frac=ex / sig_s / 1e12 / pk,
                            note="executed = dense G x 3L int8 MACs per cell over the whole stage time (dense expansion, "
                                 "column statistics and fix-up included)")

    if rank == 0:
        line.update(value=value, ms_per_step=ms_per_step,
                    dtype=("s8 tcgen05 / u64 popc (scan), u8 x s8 tcgen05 filter + f64 fix-up (signatures)" if kind == "lsh"
                           else "s8 tcgen05 / u64 popc (scan)"),
                    config=dict(cfg, variant={1: "popc", 2: "mma_i8"}.get(variant_used, "popc"), scan_symmetric=sym_used,
                                parallelism=f"cell-row blocks x{world}" + ((", NCCL inside libem2b200: 1 all-gather of signatures" +
                                             (" + 1 all-gather of bounds + 1 all-to-all of column-direction candidates (symmetric scan)"
                                              if sym_used == 1 else "")) if world > 1 else ""),
                                l2=("inputs (CSR + hyperplanes, >1.4 GB) exceed the 126 MB L2; no flush needed" if kind == "lsh" else
                                    "encoded signatures (N x L bytes) exceed the 126 MB L2 for N*L > 1.3e8; candidate buffers are rewritten every step"),
                                ordered_evaluations_per_s=N * float(N) / (ms_per_step * 1e-3),
                                mean_neighbours_stored=used_mean),
                    stage_ms=stage_ms, roofline=roof,
                    e2e=None if args.no_e2e else dict(value=pairs_total / (e2e_t * 1e-3), unit="cell-pairs/s", ms=e2e_t,
                                                      h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, stage_ms=e2e_stats, api=api),
                    gpu_launches=int(launches), clocks=clocks)
        if sig_roof:
            line["signature_roofline"] = sig_roof
        if world == 1 and kind == "lsh" and hashed and not args.no_e2e and not args.no_api_e2e:
            # the reference's own call on a data directory, everything it contains inside the timed region (tools/e2e_host.py;
            # a subprocess: the C++ layer prints its progress to stdout, and a failure here must not cost the bench line).
            # Its data directory and result live in a private temporary directory: the tree may be read-only and the
            # machine shared.
            try:
                torch.cuda.empty_cache()
                with tempfile.TemporaryDirectory(prefix="em2-e2e-", dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
                    api_out = os.path.join(tmp, "e2e_api.json")
                    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "e2e_host.py"), "--workload", args.workload,
                                    "--repeat", str(args.steps), "--dir", os.path.join(tmp, "data"), "--out", api_out],
                                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=420, check=True,
                                   env=dict(os.environ, EM2_DEVICES=str(local_rank)))
                    with open(api_out) as f:
                        api = json.load(f)
                line["e2e_api"] = dict(value=api["cell_pairs_per_s"], unit="cell-pairs/s", ms=1e3 * api["best_seconds"], api=api["api"],
                                       includes=api["includes"], runs=api["runs"],
                                       note="ingest (addCells into the mapped CellExpressionCounts file) is outside the timed region, as in the "
                                            "reference; `e2e` above is the same job through the C-ABI call on pinned host buffers")
            except Exception as ex:      # noqa: BLE001
                line["e2e_api"] = dict(error=f"{type(ex).__name__}: {ex}"[:300])
        if world == 1 and not args.no_cpu_baseline:
            import oracle
            oracle.build()
            sig_np = sig_all_host if sig_all_host is not None else d_sig_local[:rows].cpu().numpy().view(np.uint64)
            sig_cells, loop_rows = sample_sizes(N)
            head = host_counts(w, 0, min(sig_cells, N)) if kind == "lsh" else None
            cb = cpu_sample(w, head, sig_np, loop_rows, lsh=L)
            ref_sig = cb.pop("_ref_sig", None)
            if ref_sig is not None:      # the reference's signatures of the sampled cells against the GPU's
                cb["sample_signatures_match_gpu"] = bool(np.array_equal(ref_sig, sig_np[:len(ref_sig)]))
            line["cpu_baseline"] = cb
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="m1", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", default="auto", choices=["auto", "popc", "mma"])
    ap.add_argument("--lsh", type=int, default=0, help="override the workload's LSH bit count (config 4 sweep)")
    ap.add_argument("--symmetric", action="store_true",
                    help="whole-matrix scans evaluate every unordered pair once (em2_set_option scan_symmetric = 2; N = 1 only)")
    ap.add_argument("--one-directional", action="store_true", help="never use the symmetric scan (scan_symmetric = 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--option", action="append", default=[], metavar="NAME=VALUE",
                    help="em2_set_option on the engine (tuning / diagnosis runs), e.g. --option debug_flags=8")
    ap.add_argument("--no-api-e2e", action="store_true", help="skip the API-level leg (tools/e2e_host.py on a data directory)")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: skip the host-buffer end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32/float64; "
                         "a fixed, seeded sample of the cells when all of them would exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm (--impl b200)")
    args.warmup = max(args.warmup, 0)
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_b200(args, w)


if __name__ == "__main__":
    main()
