#!/bin/bash
# FP4 symmetric scan, step 0: sustained CTA-pair issue rates of kind::mxf4 (N = 128, 256) against kind::i8 (N = 256) on
# random +-1 operands, with SM clock / clock-event reasons / power read in the same run; plus one bench line of the
# current tree.
OUT=${1:?usage: bash tools/gpu/fp4_gate.sh OUTPUT_DIR}
OUT=$(mkdir -p "$OUT" && cd "$OUT" && pwd)
{ nvidia-smi --query-gpu=name,memory.total,power.limit,clocks.max.sm --format=csv; } > $OUT/box.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1 || { echo build failed; tail -30 $OUT/build.log; exit 1; }
timeout 120 expressionmatrix2_b200/build/mma_peak fp4 2 3 > $OUT/mma_peak_fp4.json 2> $OUT/mma_peak_fp4.err
echo "gate rc=$?"; cat $OUT/mma_peak_fp4.json
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 3 > $OUT/bench_m1.json 2> $OUT/bench_m1.err
echo "bench rc=$?"; tail -c 400 $OUT/bench_m1.err; cat $OUT/box.txt
