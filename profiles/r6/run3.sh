#!/bin/bash
# The full default bench once per build, parent (BASE_TREE) and this tree, in one call.
set -u
BASE_TREE=${BASE_TREE:?set BASE_TREE to a built checkout of the parent commit}
O=${OUT_DIR:-profiles/r6/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
for t in "$BASE_TREE" .; do
  n=$([ $t = . ] && echo new || echo old)
  (cd $t && timeout 270 python bench.py) 2> /dev/null | tail -n 1 > $O/full_$n.json
  python -c "
import json
r = json.load(open('$O/full_$n.json'))
print('$n', 'ms_per_step', r['ms_per_step'], 'sweep', json.dumps(r.get('sweep_summary'))[:300], 'e2e', json.dumps(r.get('e2e'))[:120])"
done
