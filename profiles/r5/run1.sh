#!/bin/bash
# The whole -m gpu suite and smoke() on both builds: the parent commit (BASE_TREE) and
# this tree.
set -u
BASE_TREE=${BASE_TREE:?set BASE_TREE to a built checkout of the parent commit}
O=${OUT_DIR:-profiles/r5/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/card1.txt
for t in . "$BASE_TREE"; do
  n=$([ $t = . ] && echo new || echo old)
  (cd $t && timeout 720 python -m pytest tests -m gpu -q -p no:cacheprovider) > $O/tests_gpu_$n.log 2>&1
  echo "$n tests rc=$?"; tail -n 3 $O/tests_gpu_$n.log
  (cd $t && timeout 120 python -c "import __graft_entry__ as g; g.smoke()") > $O/smoke_$n.log 2>&1
  echo "$n smoke rc=$?"; tail -n 1 $O/smoke_$n.log
done
