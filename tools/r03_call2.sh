#!/bin/bash
# round 3, call 2 (1 GPU): the final tree builds (no spills in the persistent kernels), smoke() and the whole GPU suite pass.
set -u
O=${OUT_DIR:-r03_out}; mkdir -p $O  # results directory (relative to the repository root)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r03c2_gpu.csv
date +%T; python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('build + smoke ok')" 2>&1 | tail -2 | tee $O/r03_smoke.log
grep -A3 "Compiling entry.*persist_kernel" build/elliptic_persist.ptxas.log | grep -E "Compiling|spill|registers" > $O/r03_ptxas_persist.txt
echo "persist_kernel instantiations: $(grep -c Compiling $O/r03_ptxas_persist.txt), with spills: $(grep 'spill stores' $O/r03_ptxas_persist.txt | grep -vc ' 0 bytes spill stores')"
date +%T; timeout 1000 python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -15 | tee $O/r03_gputests.log; date +%T
