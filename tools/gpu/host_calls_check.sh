#!/bin/bash
# Blocking host-buffer calls against the parent commit: build this tree and a copy of the parent in _parent/ (git archive).
# "check": the test suite and smoke on this tree, then both arms on the same seeded inputs -- every blocking call of
# tests/test_gpu_host_calls.py (this tree's file, run against each arm's library) with pageable and with pinned buffers, and
# bench.py's c5 outputs -- compared byte for byte, and em2_stats field by field but the times and bounced_bytes.
# "time": three runs of each arm, alternated, of bench.py on m1 and c5, and the pageable-buffer em2_stats of
# em2_compute_signatures (200k cells x 20k genes, 1000 counts per cell, L = 1024), em2_find_similar_pairs and
# em2_find_similar_pairs7 (1 M cells x 1024 bits); ROUNDS picks some of the three rounds, the summary reads every round found
# in OUTPUT_DIR.  "all": both.
OUT=${1:?usage: bash tools/gpu/host_calls_check.sh OUTPUT_DIR [check|time|all] [ROUNDS]}
MODE=${2:-check}
ROUNDS=${3:-1 2 3}
OUT=$(mkdir -p "$OUT" && cd "$OUT" && pwd)      # absolute: the parent arm runs from _parent/
NEW=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/gpu.csv
python -c "import __graft_entry__ as g; g.build()" > $OUT/build_new.log 2>&1 || { echo new build failed; tail -30 $OUT/build_new.log; exit 1; }
(cd _parent && python -c "import __graft_entry__ as g; g.build()") > $OUT/build_parent.log 2>&1 || { echo parent build failed; exit 1; }
arm_dir() { if [ $1 = new ]; then echo .; else echo _parent; fi; }

if [ $MODE = check ] || [ $MODE = all ]; then
timeout 1500 python -m pytest tests -q -p no:cacheprovider > $OUT/tests.log 2>&1
echo "tests rc=$?"; tail -8 $OUT/tests.log
timeout 300 python __graft_entry__.py --smoke > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -2 $OUT/smoke.log

# ---- outputs and stats of both arms ----
for arm in new parent; do
  (cd $(arm_dir $arm) && NEW=$NEW timeout 600 python - $OUT/parity_$arm <<'EOF'
import importlib.util, json, os, sys
import numpy as np
import expressionmatrix2_b200 as em2

out = sys.argv[1]
os.makedirs(out, exist_ok=True)
assert os.path.dirname(em2.__file__) == os.path.join(os.getcwd(), "expressionmatrix2_b200"), em2.__file__
spec = importlib.util.spec_from_file_location("host_calls", os.path.join(os.environ["NEW"], "tests", "test_gpu_host_calls.py"))
hc = importlib.util.module_from_spec(spec)
spec.loader.exec_module(hc)
outs, stats = {}, {}
with em2.Engine(0) as e, em2.MultiEngine(devices=[0]) as m:
    d = hc.Data(e)
    for name, fn in hc.CALLS.items():
        for mode in ("pageable", "pinned"):
            eng = m if name.startswith("multi_") else e
            res = fn(eng, hc.Mem(mode), d)[0]
            for i, o in enumerate(res):
                outs[f"{name}_{mode}_{i}"] = o.copy()
            stats[f"{name}_{mode}"] = eng.stats()
np.savez(f"{out}/outputs.npz", **outs)
json.dump(stats, open(f"{out}/stats.json", "w"), indent=1)
print("ok", len(stats))
EOF
  ) > $OUT/parity_$arm.log 2>&1
  echo "parity $arm rc=$?"; tail -2 $OUT/parity_$arm.log
  d=$OUT/dump_c5_$arm
  (cd $(arm_dir $arm) && timeout 600 python bench.py --gpus 1 --workload c5 --steps 1 --warmup 1 --no-cpu-baseline --no-api-e2e --dump-outputs $d) \
    > $OUT/dump_c5_$arm.json 2> $OUT/dump_c5_$arm.err
  echo "dump c5 $arm rc=$?"
done
OUT="$OUT" python - <<'EOF' | tee $OUT/parity_summary.txt
import glob, json, os
import numpy as np
o = os.environ["OUT"]
a, b = np.load(f"{o}/parity_new/outputs.npz"), np.load(f"{o}/parity_parent/outputs.npz")
# analyze_lsh's error sums (outputs 1 and 2) are float sums in an order the device chooses: compared to rounding
sums = [f"analyze_lsh_{m}_{i}" for m in ("pageable", "pinned") for i in (1, 2)]
print("outputs: same names", sorted(a.files) == sorted(b.files), "unequal",
      [n for n in a.files if (not np.allclose(a[n], b[n], rtol=1e-9, atol=1e-12) if n in sums else a[n].tobytes() != b[n].tobytes())])
sa, sb = json.load(open(f"{o}/parity_new/stats.json")), json.load(open(f"{o}/parity_parent/stats.json"))
for n in sa:
    diff = {f: (sa[n][f], sb[n][f]) for f in sa[n] if not f.endswith("_ms") and f != "bounced_bytes" and sa[n][f] != sb[n][f]}
    print(n, "stats differ (new, parent):" if diff else "stats equal", diff or "",
          "bounced new/parent", sa[n]["bounced_bytes"], sb[n]["bounced_bytes"])
x, y = f"{o}/dump_c5_new", f"{o}/dump_c5_parent"
names = sorted(os.path.basename(p) for p in glob.glob(x + "/*.npy"))
print("c5 dump files", names, "same set", names == sorted(os.path.basename(p) for p in glob.glob(y + "/*.npy")),
      "equal", all(np.array_equal(np.load(f"{x}/{n}"), np.load(f"{y}/{n}")) for n in names))
EOF
rm -rf $OUT/dump_c5_new $OUT/dump_c5_parent
fi

if [ $MODE = time ] || [ $MODE = all ]; then
for i in $ROUNDS; do
  for arm in parent new; do
    dir=$(arm_dir $arm)
    (cd $dir && timeout 600 python bench.py --gpus 1 --workload m1 --no-cpu-baseline --no-api-e2e) > $OUT/m1_${arm}_$i.json 2> $OUT/m1_${arm}_$i.err
    (cd $dir && timeout 600 python bench.py --gpus 1 --workload c5 --no-cpu-baseline) > $OUT/c5_${arm}_$i.json 2> $OUT/c5_${arm}_$i.err
    (cd $dir && timeout 900 python - $OUT/calls_${arm}_$i.json <<'EOF'
import json, sys
import expressionmatrix2_b200 as em2
from expressionmatrix2_b200 import synthetic

res = {}
with em2.Engine(0) as e:        # numpy buffers: pageable; each call once to warm up, then the one whose stats are kept
    N, G, L = 200_000, 20_000, 1024
    toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, 1000, seed=5)
    pairs = synthetic.to_pairs(genes, counts)
    del genes, counts
    U = em2.generate_lsh_vectors(G, L, 231)
    for _ in range(2):
        e.compute_signatures(toc, pairs, U)
    res["compute_signatures"] = e.stats()
    del toc, pairs, U
    sig = synthetic.gen_signatures(1_000_000, L, seed=6, clusters=500)
    for _ in range(2):
        e.find_similar_pairs(sig, L, 50, 0.2)
    res["find_similar_pairs"] = e.stats()
    for _ in range(2):
        e.find_similar_pairs7(sig, L, 50, 0.2, [24, 16, 12], 200, 20)
    res["find_similar_pairs7"] = e.stats()
json.dump(res, open(sys.argv[1], "w"), indent=1)
EOF
    ) > $OUT/calls_${arm}_$i.log 2>&1
    echo "timing $arm $i done"
  done
done
OUT="$OUT" python - <<'EOF' | tee $OUT/timing_summary.txt
import json, os
o = os.environ["OUT"]
for arm in ("parent", "new"):
    for i in (1, 2, 3):
        for w in ("m1", "c5"):
            try:
                line = json.loads(open(f"{o}/{w}_{arm}_{i}.json").read().strip().splitlines()[-1])
                print(arm, i, w, "ms_per_step %.3f e2e_ms %.2f" % (line["ms_per_step"], line["e2e"]["ms"]))
            except Exception as ex:
                print(arm, i, w, "unreadable", ex)
        try:
            c = json.load(open(f"{o}/calls_{arm}_{i}.json"))
            print(arm, i, " ".join("%s total_ms %.1f h2d_ms %.1f d2h_ms %.1f bounced %d" % (n, s["total_ms"], s["h2d_ms"], s["d2h_ms"],
                                                                                           s["bounced_bytes"]) for n, s in c.items()))
        except Exception as ex:
            print(arm, i, "calls unreadable", ex)
EOF
fi
exit 0
