#!/bin/bash
# round 3, call 1 (1 GPU): persistent chain with pair-split items.  Start stagger and whole / split configuration at P = 128, split items
# at the other even-MT extents, per-launch times, and a first output comparison against the parent commit's build in $1.
# (Run on an intermediate build whose SB200_PERSIST_CFG selected 1 = 12 whole-item warps at P = 128, 4 = split items at P = 32 / 64 / 96,
# unset = split items at P = 128 only; the final build has no such switch.)
set -u
O=${OUT_DIR:-r03_out}; mkdir -p $O  # results directory (relative to the repository root)
PARENT=${1:-_parent}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r03_gpu.csv
for rep in 1 2 3; do
  for cs in "1 6000" "0 0" "0 3000" "0 6000"; do set -- $cs
    echo "cfg=$1 stagger=$2 rep=$rep $(SB200_PERSIST_CFG=$1 SB200_STAGGER=$2 timeout 120 python tools/time_ops.py elliptic 128 200 2>&1 | head -1)"
  done
done | tee $O/r03_stagger_cfg.log
for rep in 1 2; do for P in 32 64 96; do for cfg in 1 4; do
  echo "cfg=$cfg P=$P rep=$rep $(SB200_PERSIST_CFG=$cfg timeout 120 python tools/time_ops.py elliptic $P 200 2>&1 | head -1)"
done; done; done | tee $O/r03_extents.log
cp tools/persist_launch_times.py $PARENT/tools/
(cd $PARENT && timeout 300 python tools/persist_launch_times.py 128 50) > $O/r03_launches_parent.jsonl 2>&1
timeout 300 python tools/persist_launch_times.py 128 50 > $O/r03_launches_pair.jsonl 2>&1
cat $O/r03_launches_parent.jsonl $O/r03_launches_pair.jsonl
(cd $PARENT && timeout 300 python bench.py --steps 20 --no-cpu-baseline --no-ksp --no-extras --no-stokes --dump-outputs ../$O/dump_parent) > $O/r03_bench_parent_quick.json 2>&1
timeout 300 python bench.py --steps 20 --no-cpu-baseline --no-ksp --no-extras --no-stokes --dump-outputs $O/dump_pair > $O/r03_bench_pair_quick.json 2>&1
python -c "import numpy as np; a=np.load('$O/dump_parent/matmult_elliptic.npy'); b=np.load('$O/dump_pair/matmult_elliptic.npy'); print('bit-identical', np.array_equal(a,b), 'maxdiff', float(np.abs(a-b).max()))" | tee $O/r03_bitident_quick.txt
tail -c 600 $O/r03_bench_pair_quick.json
timeout 900 python -m pytest tests/test_gpu_elliptic.py -m gpu -q -x 2>&1 | tail -5 | tee $O/r03_gpu_elliptic.log
rm -rf $O/dump_parent $O/dump_pair
