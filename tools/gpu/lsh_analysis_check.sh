#!/bin/sh
# LSH accuracy analysis (em2_analyze_lsh) on one B200: build, the analysis test files and the exact path's GPU test files, smoke,
# then tools/lsh_analysis_time.py.  Usage: tools/gpu/lsh_analysis_check.sh OUTDIR [tests|time|all]
[ -n "$1" ] || { echo "usage: $0 OUTDIR [tests|time|all]" >&2; exit 2; }
OUT=$1
WHAT=${2:-all}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1 || { tail -40 "$OUT/build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
rc=0
if [ "$WHAT" != time ]; then
    python -m pytest -q -p no:cacheprovider tests/test_gpu_lsh_analysis.py tests/test_host_lsh_analysis.py tests/test_lsh_analysis_ref.py \
        > "$OUT/tests_analysis.log" 2>&1 || rc=1
    tail -25 "$OUT/tests_analysis.log"
    python -m pytest -q -p no:cacheprovider tests/test_gpu_exact_filter.py tests/test_gpu_extend_exact.py tests/test_gpu_rescore.py \
        tests/test_host_exact_general.py tests/test_host_extend_exact.py tests/test_host_rescore.py > "$OUT/tests_exact.log" 2>&1 || rc=1
    tail -8 "$OUT/tests_exact.log"
    python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1 || rc=1
    tail -3 "$OUT/smoke.log"
fi
if [ "$WHAT" != tests ]; then
    python tools/lsh_analysis_time.py "$OUT" > "$OUT/lsh_analysis_time.log" 2>&1 || rc=1
    tail -6 "$OUT/lsh_analysis_time.log"
fi
exit $rc
