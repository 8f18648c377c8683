#!/bin/bash
# Exact path host side: build this tree and a copy of the parent commit in _parent/ (git archive), the test suite and smoke
# on this tree, then both arms on the same seeded inputs -- the full job, an extension (N = 3000, M = 1000) and a rescoring,
# each with pageable and with pinned buffers, and bench.py's c5 outputs -- compared byte for byte with every em2_stats field
# but the times and bounced_bytes.  Second argument "time": instead, c5, tools/extend_exact_time.py and
# tools/rescore_time.py, three runs of each arm, alternated.
OUT=${1:?usage: bash tools/gpu/exact_host_check.sh OUTPUT_DIR [check|time]}
OUT=$(mkdir -p "$OUT" && cd "$OUT" && pwd)      # absolute: the parent arm runs from _parent/
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/gpu.csv
python -c "import __graft_entry__ as g; g.build()" > $OUT/build_new.log 2>&1 || { echo new build failed; tail -30 $OUT/build_new.log; exit 1; }
(cd _parent && python -c "import __graft_entry__ as g; g.build()") > $OUT/build_parent.log 2>&1 || { echo parent build failed; exit 1; }
if [ "${2:-check}" = check ]; then
timeout 1500 python -m pytest tests -q -p no:cacheprovider > $OUT/tests.log 2>&1
echo "tests rc=$?"; tail -8 $OUT/tests.log
timeout 300 python __graft_entry__.py --smoke > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -2 $OUT/smoke.log

# ---- outputs and stats of both arms ----
for arm in new parent; do
  if [ $arm = new ]; then dir=.; else dir=_parent; fi
  (cd $dir && timeout 600 python - $OUT/parity_$arm <<'EOF'
import json, os, sys
import numpy as np
import torch
import expressionmatrix2_b200 as em2
from expressionmatrix2_b200 import synthetic

out = sys.argv[1]
os.makedirs(out, exist_ok=True)
P = em2._ptr


def pin(a):
    t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory()
    return t.numpy().view(a.dtype).reshape(a.shape), t


res, keep = {}, []
with em2.Engine(0) as e:
    L = e._L
    for name, frac in (("int", False), ("general", True)):
        N, M, G, k, thr = 4000, 1000, 2000, 30, 0.1
        toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.05, seed=77, mode="clustered", clusters=12)
        if frac:
            counts = np.log1p(counts).astype(np.float32) * np.float32(1.7)
        pairs = em2.to_pairs(genes, counts)
        oldN = N - M
        U = em2.generate_lsh_vectors(G, 256, 231)
        cids, _, cused = e.lsh_similar_pairs(toc, pairs, U, 60, 0.0)
        cand = np.zeros(cids.shape, em2.SIMPAIR_DTYPE)
        cand["cell"] = cids
        for mem in ("pageable", "pinned"):
            conv = (lambda a: a) if mem == "pageable" else (lambda a: keep.append(pin(a)) or keep[-1][0])
            t, p = conv(toc), conv(pairs)
            # the full job over the old cells, then over all cells
            o_old, u_old = conv(np.zeros((oldN, k), em2.SIMPAIR_DTYPE)), conv(np.zeros(oldN, np.uint32))
            rc = L.em2_exact_similar_pairs(e._h, oldN, G, P(t), P(p), k, thr, P(o_old), P(u_old))
            assert rc == 0, L.em2_last_error(e._h)
            o, u = conv(np.zeros((N, k), em2.SIMPAIR_DTYPE)), conv(np.zeros(N, np.uint32))
            rc = L.em2_exact_similar_pairs(e._h, N, G, P(t), P(p), k, thr, P(o), P(u))
            assert rc == 0, L.em2_last_error(e._h)
            res[f"{name}_{mem}_full"] = (o.copy(), u.copy(), e.stats())
            o, u = conv(np.zeros((N, k), em2.SIMPAIR_DTYPE)), conv(np.zeros(N, np.uint32))
            rc = L.em2_extend_exact_similar_pairs(e._h, oldN, N, G, P(t), P(p), k, thr, P(o_old), P(u_old), P(o), P(u))
            assert rc == 0, L.em2_last_error(e._h)
            res[f"{name}_{mem}_extend"] = (o.copy(), u.copy(), e.stats())
            c, cu = conv(cand), conv(cused)
            o, u = conv(np.zeros((N, 20), em2.SIMPAIR_DTYPE)), conv(np.zeros(N, np.uint32))
            rc = L.em2_rescore_similar_pairs(e._h, N, G, P(t), P(p), cand.shape[1], P(c), P(cu), 20, thr, P(o), P(u))
            assert rc == 0, L.em2_last_error(e._h)
            res[f"{name}_{mem}_rescore"] = (o.copy(), u.copy(), e.stats())
np.savez(f"{out}/lists.npz", **{f"{n}_pairs": v[0] for n, v in res.items()}, **{f"{n}_used": v[1] for n, v in res.items()})
json.dump({n: v[2] for n, v in res.items()}, open(f"{out}/stats.json", "w"), indent=1)
print("ok", len(res))
EOF
  ) > $OUT/parity_$arm.log 2>&1
  echo "parity $arm rc=$?"; tail -2 $OUT/parity_$arm.log
  d=$OUT/dump_c5_$arm
  (cd $dir && timeout 600 python bench.py --gpus 1 --workload c5 --steps 1 --warmup 1 --no-cpu-baseline --no-api-e2e --dump-outputs $d) \
    > $OUT/dump_c5_$arm.json 2> $OUT/dump_c5_$arm.err
  echo "dump c5 $arm rc=$?"
done
OUT="$OUT" python - <<'EOF'
import glob, json, os
import numpy as np
o = os.environ["OUT"]
a, b = np.load(f"{o}/parity_new/lists.npz"), np.load(f"{o}/parity_parent/lists.npz")
print("lists: same names", sorted(a.files) == sorted(b.files),
      "unequal", [n for n in a.files if a[n].tobytes() != b[n].tobytes()])
sa, sb = json.load(open(f"{o}/parity_new/stats.json")), json.load(open(f"{o}/parity_parent/stats.json"))
for n in sa:
    diff = {f: (sa[n][f], sb[n][f]) for f in sa[n] if not f.endswith("_ms") and f != "bounced_bytes" and sa[n][f] != sb[n][f]}
    print(n, "stats differ:" if diff else "stats equal", diff or "", "bounced new/parent", sa[n]["bounced_bytes"], sb[n]["bounced_bytes"],
          "total_ms new/parent %.1f/%.1f" % (sa[n]["total_ms"], sb[n]["total_ms"]))
x, y = f"{o}/dump_c5_new", f"{o}/dump_c5_parent"
names = sorted(os.path.basename(p) for p in glob.glob(x + "/*.npy"))
print("c5 dump files", names, "same set", names == sorted(os.path.basename(p) for p in glob.glob(y + "/*.npy")),
      "equal", all(np.array_equal(np.load(f"{x}/{n}"), np.load(f"{y}/{n}")) for n in names))
EOF
rm -rf $OUT/dump_c5_new $OUT/dump_c5_parent
exit 0
fi

# ---- timing, arms alternated ----
for i in 1 2 3; do
  for arm in new parent; do
    if [ $arm = new ]; then dir=.; else dir=_parent; fi
    (cd $dir && timeout 600 python bench.py --gpus 1 --workload c5 --no-cpu-baseline) > $OUT/c5_${arm}_$i.json 2> $OUT/c5_${arm}_$i.err
    (cd $dir && timeout 600 python tools/extend_exact_time.py $OUT/ext_${arm}_$i --n 50000 --m 1000 --runs 1) > $OUT/ext_${arm}_$i.log 2>&1
    (cd $dir && timeout 900 python tools/rescore_time.py $OUT/res_${arm}_$i --n 50000 --widths 100 --runs 1) > $OUT/res_${arm}_$i.log 2>&1
    echo "timing $arm $i done"
  done
done
OUT="$OUT" python - <<'EOF'
import json, os
o = os.environ["OUT"]
for arm in ("new", "parent"):
    for i in (1, 2, 3):
        try:
            line = json.loads(open(f"{o}/c5_{arm}_{i}.json").read().strip().splitlines()[-1])
            print(arm, i, "c5 ms_per_step %.3f e2e_ms %.2f" % (line["ms_per_step"], line["e2e"]["ms"]))
        except Exception as ex:
            print(arm, i, "c5 unreadable", ex)
        try:
            c = json.load(open(f"{o}/ext_{arm}_{i}/extend_exact_time.json"))["cases"][0]
            print(arm, i, "full scan/total %.2f/%.2f extend scan/total %.2f/%.2f" % (
                c["full"]["scan_ms"]["median"], c["full"]["total_ms"]["median"], c["extend"]["scan_ms"]["median"],
                c["extend"]["total_ms"]["median"]), "equal", c["outputs_equal"])
            c = json.load(open(f"{o}/res_{arm}_{i}/rescore_time.json"))["cases"][0]
            r = c["widths"][0]["rescore"]
            print(arm, i, "exact scan/total %.2f/%.2f rescore scan/total %.2f/%.2f" % (
                c["exact"]["scan_ms"]["median"], c["exact"]["total_ms"]["median"], r["scan_ms"]["median"], r["total_ms"]["median"]))
        except Exception as ex:
            print(arm, i, "tool output unreadable", ex)
EOF
