#!/bin/bash
# One-stream batch-32 step: headline three times per build, alternating, and the timeline
# of each build with the frame-copy marks.  BASE_TREE: a built checkout of the parent
# commit.  Both trees need their trace library
# (B2R_TRACE_GT=1 python -m dopamine_b200.csrc.build --trace --force).
set -u
BASE_TREE=${BASE_TREE:?set BASE_TREE to a built checkout of the parent commit}
O=${OUT_DIR:-profiles/r6/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $O/card1.txt
for i in 1 2 3; do
  for t in "$BASE_TREE" .; do
    n=$([ $t = . ] && echo new || echo old)
    (cd $t && timeout 120 python bench.py --no-sweep --no-e2e --no-cpu-baseline) 2> $O/headline_${n}_$i.err | tail -n 1 > $O/headline_${n}_$i.json
    python -c "
import json
r = json.load(open('$O/headline_${n}_$i.json'))
print('$n run $i: ms_per_step', r['ms_per_step'])"
  done
done
for t in "$BASE_TREE" .; do
  n=$([ $t = . ] && echo new || echo old)
  echo "== timeline $n"
  (cd $t && B2R_LIB=profiles/micro/libb200replay_trace.so timeout 120 python profiles/micro/timeline.py 32) 2>&1 | tail -n 24 | tee $O/timeline_$n.txt
done
nvidia-smi --query-gpu=name,power.limit,clocks.sm --format=csv,noheader
