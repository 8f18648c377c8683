#!/bin/bash
# FP4 symmetric scan: this tree against a copy of the parent commit in _parent/ (git archive), alternating in one
# session: 3 runs each of the default bench line (m1), then 2 each of c4 and c2.
OUT=${1:?usage: bash tools/gpu/fp4_timing.sh OUTPUT_DIR}
OUT=$(mkdir -p "$OUT" && cd "$OUT" && pwd)      # absolute: the parent arm runs from _parent/
{ nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv; } > $OUT/timing_box.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/build_new.log 2>&1 || { echo new build failed; exit 1; }
(cd _parent && python -c "import __graft_entry__ as g; g.build()") > $OUT/build_parent.log 2>&1 || { echo parent build failed; exit 1; }
run() {   # arm workload index extra-args...
  local arm=$1 w=$2 i=$3; shift 3
  local dir=.; [ $arm = parent ] && dir=_parent
  (cd $dir && timeout 300 python bench.py --gpus 1 --steps 5 --warmup 3 --workload $w "$@") \
    > $OUT/t_${w}_${arm}_$i.json 2> $OUT/t_${w}_${arm}_$i.err
  echo "$w $arm $i rc=$?"
}
for i in 1 2 3; do run parent m1 $i; run new m1 $i; done
for w in c4 c2; do
  for i in 1 2; do run parent $w $i --no-cpu-baseline --no-api-e2e; run new $w $i --no-cpu-baseline --no-api-e2e; done
done
OUT="$OUT" python - <<'EOF' | tee $OUT/timing_summary.json
import glob, json, os, statistics
out = {}
for w in ("m1", "c4", "c2"):
    for arm in ("parent", "new"):
        lines = []
        for f in sorted(glob.glob(f"{os.environ['OUT']}/t_{w}_{arm}_*.json")):
            try:
                lines.append(json.loads(open(f).read().strip().splitlines()[-1]))
            except Exception:
                pass
        if not lines:
            continue
        ms = [l["ms_per_step"] for l in lines]
        scan = [l["stage_ms"].get("scan_topk") for l in lines]
        out[f"{w}_{arm}"] = dict(ms_per_step=ms, median_ms=statistics.median(ms), spread_ms=max(ms) - min(ms),
                                 scan_topk_ms=scan, median_scan_ms=statistics.median(scan),
                                 scan_symmetric=[l["config"].get("scan_symmetric") for l in lines],
                                 lists_equal_device_path=[l.get("e2e", {}).get("stage_ms", {}).get("lists_equal_device_path") for l in lines],
                                 clocks=[l.get("clocks") for l in lines])
    if f"{w}_new" in out and f"{w}_parent" in out:
        out[f"{w}_ratio"] = dict(step=out[f"{w}_new"]["median_ms"] / out[f"{w}_parent"]["median_ms"],
                                 scan=out[f"{w}_new"]["median_scan_ms"] / out[f"{w}_parent"]["median_scan_ms"])
print(json.dumps(out, indent=1))
EOF
