#!/bin/bash
# FP4 symmetric scan: GPU test suite and smoke on this tree, then the outputs of bench.py on m1 and c4 from this tree
# and from a copy of the parent commit in _parent/ (git archive), compared array for array.
OUT=${1:?usage: bash tools/gpu/fp4_check.sh OUTPUT_DIR}
OUT=$(mkdir -p "$OUT" && cd "$OUT" && pwd)      # absolute: the parent arm runs from _parent/
python -c "import __graft_entry__ as g; g.build()" > $OUT/build_new.log 2>&1 || { echo new build failed; tail -30 $OUT/build_new.log; exit 1; }
(cd _parent && python -c "import __graft_entry__ as g; g.build()") > $OUT/build_parent.log 2>&1 || { echo parent build failed; exit 1; }
timeout 900 python -m pytest tests -q -m gpu -p no:cacheprovider > $OUT/tests_gpu.log 2>&1
echo "gpu tests rc=$?"; tail -15 $OUT/tests_gpu.log
timeout 300 python __graft_entry__.py --smoke > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -2 $OUT/smoke.log
for w in m1 c4; do
  for arm in new parent; do
    d=$OUT/dump_${w}_$arm
    if [ $arm = new ]; then dir=.; else dir=_parent; fi
    (cd $dir && timeout 400 python bench.py --gpus 1 --workload $w --steps 1 --warmup 1 --no-cpu-baseline --no-api-e2e --dump-outputs $d) \
      > $OUT/dump_${w}_$arm.json 2> $OUT/dump_${w}_$arm.err
    echo "dump $w $arm rc=$?"
  done
done
OUT="$OUT" python - <<'EOF'
import glob, json, os
import numpy as np
for w in ("m1", "c4"):
    a, b = f"{os.environ['OUT']}/dump_{w}_new", f"{os.environ['OUT']}/dump_{w}_parent"
    names = sorted(os.path.basename(p) for p in glob.glob(a + "/*.npy"))
    same = names == sorted(os.path.basename(p) for p in glob.glob(b + "/*.npy"))
    eq = {n: bool(np.array_equal(np.load(f"{a}/{n}"), np.load(f"{b}/{n}"))) for n in names}
    line = json.loads(open(f"{os.environ['OUT']}/dump_{w}_new.json").read().strip().splitlines()[-1])
    print(w, "files", names, "same set", same, "equal", eq, "scan_symmetric", line["config"].get("scan_symmetric"),
          "lists_equal_device_path", line.get("e2e", {}).get("stage_ms", {}).get("lists_equal_device_path"))
EOF
rm -rf $OUT/dump_m1_new $OUT/dump_m1_parent $OUT/dump_c4_new $OUT/dump_c4_parent
