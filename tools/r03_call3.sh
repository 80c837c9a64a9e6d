#!/bin/bash
# round 3, call 3 (1 GPU): the final tree against the parent commit's build in $1, alternated in one call: bench.py 5 x each without the
# per-P sweep, then once each with it (every run dumps its MatMult_Elliptic result; the dumps must agree bit for bit), then the per-launch
# times of both under torch.profiler.
set -u
O=${OUT_DIR:-r03_out}; mkdir -p $O  # results directory (relative to the repository root)
PARENT=${1:-_parent}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r03c3_gpu.csv
: > $O/r03_ab_parent.jsonl; : > $O/r03_ab_pair.jsonl
for rep in 1 2 3 4 5 6; do
  date +%T
  X=--no-extras; [ $rep = 6 ] && X=
  (cd $PARENT && timeout 200 python bench.py --steps 200 --no-cpu-baseline --no-ksp $X --dump-outputs ../$O/dump_parent_$rep 2>/dev/null | tail -1) >> $O/r03_ab_parent.jsonl
  timeout 200 python bench.py --steps 200 --no-cpu-baseline --no-ksp $X --dump-outputs $O/dump_pair_$rep 2>/dev/null | tail -1 >> $O/r03_ab_pair.jsonl
done
date +%T
O=$O python - <<'PY' | tee $O/r03_ab_summary.txt
import glob, json, os, statistics
import numpy as np
O = os.environ["O"]
ref = np.load(f"{O}/dump_parent_1/matmult_elliptic.npy")
same = [bool(np.array_equal(ref, np.load(f))) for f in sorted(glob.glob(f"{O}/dump_*_*/matmult_elliptic.npy"))]
print("dumps:", len(same), "all bit-identical to parent run 1:", all(same))
for tag in ("parent", "pair"):
    L = [json.loads(l) for l in open(f"{O}/r03_ab_{tag}.jsonl") if l.strip()]
    ms = [d["ms_per_step"] for d in L]
    warm = [d["value_l2_warm"] for d in L]
    print(tag, "runs", len(L), "ms_per_step median %.5f min %.5f max %.5f" % (statistics.median(ms), min(ms), max(ms)), [round(x, 5) for x in ms])
    print(tag, "value_l2_warm GDOF/s median %.3f" % statistics.median(warm), [round(x, 3) for x in warm])
    print(tag, "parity ok", [d["parity"]["ok"] for d in L])
    print(tag, "stokes", json.dumps(L[-1].get("stokes"))[:600])
    ps = L[-1].get("p_sweep")
    rows = ps.get("rows", ps) if isinstance(ps, dict) else ps
    for r in rows if isinstance(rows, list) else []:
        if r.get("op") == "MatMult_Elliptic":
            print(tag, "p_sweep", r.get("P"), r.get("path"), round(r["ms"], 5))
PY
rm -rf $O/dump_parent_* $O/dump_pair_*
cp tools/persist_launch_times.py $PARENT/tools/
(cd $PARENT && timeout 200 python tools/persist_launch_times.py 128 100 2>/dev/null) > $O/r03_launches_parent.jsonl
timeout 200 python tools/persist_launch_times.py 128 100 2>/dev/null > $O/r03_launches_pair.jsonl
cat $O/r03_launches_parent.jsonl $O/r03_launches_pair.jsonl
date +%T
