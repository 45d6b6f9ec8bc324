#!/bin/bash
# Staged loss tail: new tests, timelines, headline (old and new builds alternating), dumps.
# BASE_TREE: a built checkout of the parent commit (old build, timed alternately).
set -u
BASE_TREE=${BASE_TREE:?set BASE_TREE to a built checkout of the parent commit}
O=${OUT_DIR:-profiles/r4/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/card.txt
timeout 900 python -m pytest tests/test_tail_staging.py tests/test_gpu_step.py -m gpu -x -q > $O/tests1.log 2>&1
echo "tests rc=$?"; tail -n 3 $O/tests1.log
for t in "$BASE_TREE" .; do
  echo "== timeline $t"
  (cd $t && B2R_LIB=profiles/micro/libb200replay_trace.so timeout 300 python profiles/micro/timeline.py 32) 2>&1 | tail -n 22
done
for i in 1 2 3; do
  for t in "$BASE_TREE" .; do
    n=$([ $t = . ] && echo new || echo old)
    (cd $t && timeout 600 python bench.py --no-sweep --no-e2e --no-cpu-baseline) 2> $O/headline_${n}_$i.err | tail -n 1 > $O/headline_${n}_$i.json
    python -c "
import json, sys
r = json.load(open('$O/headline_${n}_$i.json'))
print('$n run $i: ms_per_step', r['ms_per_step'], 'clocks', json.dumps(r.get('clocks'))[:160])"
  done
done
for t in "$BASE_TREE" .; do
  n=$([ $t = . ] && echo new || echo old)
  (cd $t && timeout 600 python bench.py --steps 20 --no-sweep --no-e2e --no-cpu-baseline --dump-outputs /tmp/r4dump_$n) > $O/dump_$n.json 2> $O/dump_$n.err
  echo "dump $n rc=$?"
done
ls /tmp/r4dump_new | wc -l
for f in /tmp/r4dump_old/*.npy; do cmp -s $f /tmp/r4dump_new/$(basename $f) && echo "same $(basename $f)" || echo "DIFFERENT $(basename $f)"; done
