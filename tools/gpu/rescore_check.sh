#!/bin/bash
# Exact rescoring of candidate lists: build, the rescoring tests and the exact path's full-job and extension tests, then
# tools/rescore_time.py with the arguments after the output directory (default: its full set of shapes).
OUT=${1:?usage: bash tools/gpu/rescore_check.sh OUTPUT_DIR [rescore_time.py arguments]}
shift
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1 || { echo build failed; tail -30 $OUT/build.log; exit 1; }
timeout 1200 python -m pytest tests/test_gpu_rescore.py tests/test_host_rescore.py tests/test_gpu_extend_exact.py \
  tests/test_host_extend_exact.py -q -p no:cacheprovider > $OUT/tests_rescore.log 2>&1
echo "tests rc=$?"; tail -15 $OUT/tests_rescore.log
timeout 2400 python tools/rescore_time.py $OUT "$@" > $OUT/rescore_time.log 2>&1
echo "rescore_time rc=$?"; tail -30 $OUT/rescore_time.log
