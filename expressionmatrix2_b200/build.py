"""In-tree build of libem2b200.so (CUDA kernels + C-ABI) for sm_100a with nvcc.

    python -m expressionmatrix2_b200.build            # build if stale
    python -m expressionmatrix2_b200.build --force

The shared library lands next to this file so that it travels with the repo snapshot to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libem2b200.so")
SOURCES = ["capi.cu", "signatures.cu", "sig_filter.cu", "scan_popc.cu", "scan_mma.cu", "extend.cu", "exact.cu", "subset.cu", "cellgraph.cu", "siggraph.cu", "bucketed.cu", "multi.cu", "hostgen.cpp"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-ffp-contract=off,-pthread", "-Xptxas=-v",
    "-ccbin", "/usr/bin/g++", "-I/usr/include",
]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "em2b200.h"),
                                                                os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src + ".o")
        objs.append(obj)
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if src.endswith(".cpp"):
            cmd.insert(1, "-x")
            cmd.insert(2, "cu")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(HERE, "build", "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    subprocess.check_call([NVCC, "-shared", "-o", LIB, *objs, "-lcudart", "-lpthread", "-ldl", "-ccbin", "/usr/bin/g++"])
    return LIB


TOOLS = os.path.join(HERE, "..", "tools")


def build_tools(force: bool = False) -> None:
    """Pipe-rate microbenchmarks (tools/*.cu) -> build/<name>; bench.py runs them for the roofline denominators."""
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for name in ("mma_peak", "microbench"):
        src = os.path.join(TOOLS, name + ".cu")
        out = os.path.join(HERE, "build", name)
        if not os.path.exists(src):
            continue
        if not force and os.path.exists(out) and os.path.getmtime(out) >= os.path.getmtime(src):
            continue
        subprocess.check_call([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-ccbin", "/usr/bin/g++",
                               "-o", out, src], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
