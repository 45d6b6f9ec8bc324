#!/bin/bash
# The full default bench once per build, old (BASE_TREE) and new, in the same call.
set -u
BASE_TREE=${BASE_TREE:?set BASE_TREE to a built checkout of the parent commit}
O=${OUT_DIR:-profiles/r4/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
for t in "$BASE_TREE" .; do
  n=$([ $t = . ] && echo new || echo old)
  (cd $t && timeout 280 python bench.py) 2> $O/full_$n.err | tail -n 1 > $O/full_$n.json
  python -c "
import json
r = json.load(open('$O/full_$n.json'))
print('$n', 'ms_per_step', r['ms_per_step'], 'sweep', json.dumps(r.get('sweep_summary')), 'e2e', json.dumps(r.get('e2e'))[:400])"
done
