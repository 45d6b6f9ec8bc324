#!/bin/bash
# Same bits (dumps at 32 / 256 / 1024 / 4096), same speed (headline three times per build,
# alternating; the full default bench once per build) and the one-kernel-loss step with
# 101 atoms, for the parent commit (BASE_TREE) and this tree, in one call.
set -u
BASE_TREE=${BASE_TREE:?set BASE_TREE to a built checkout of the parent commit}
O=${OUT_DIR:-profiles/r5/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/card2.txt
D=$(mktemp -d)
for b in 32 256 1024 4096; do
  for t in "$BASE_TREE" .; do
    n=$([ $t = . ] && echo new || echo old)
    (cd $t && timeout 300 python bench.py --steps 20 --no-sweep --no-e2e --no-cpu-baseline \
      --batch $b --dump-outputs $D/$n/$b) > $O/dump_${n}_$b.json 2> $O/dump_${n}_$b.err
    echo "dump $n $b rc=$?"
  done
  same=0; diff=0
  for f in $D/old/$b/*.npy; do
    if cmp -s $f $D/new/$b/$(basename $f); then same=$((same + 1)); else diff=$((diff + 1)); echo "DIFFERENT $b $(basename $f)"; fi
  done
  echo "batch $b: $same identical, $diff different, $(ls $D/new/$b | wc -l) files in new"
done
mkdir -p $BASE_TREE/profiles/r5
cp profiles/r5/unsplit_writeback.py $BASE_TREE/profiles/r5/
for t in "$BASE_TREE" .; do
  n=$([ $t = . ] && echo new || echo old)
  (cd $t && timeout 300 python profiles/r5/unsplit_writeback.py --out $D/unsplit_$n) 2>&1 | tail -n 2
  cp $D/unsplit_$n/times.json $O/unsplit_$n.json
done
for f in $D/unsplit_old/*.npy; do
  cmp -s $f $D/unsplit_new/$(basename $f) && echo "unsplit same $(basename $f)" || echo "unsplit DIFFERENT $(basename $f)"
done
for i in 1 2 3; do
  for t in "$BASE_TREE" .; do
    n=$([ $t = . ] && echo new || echo old)
    (cd $t && timeout 300 python bench.py --no-sweep --no-e2e --no-cpu-baseline) 2> $O/headline_${n}_$i.err | tail -n 1 > $O/headline_${n}_$i.json
    python -c "
import json
r = json.load(open('$O/headline_${n}_$i.json'))
print('$n run $i: ms_per_step', r['ms_per_step'])"
  done
done
for t in "$BASE_TREE" .; do
  n=$([ $t = . ] && echo new || echo old)
  (cd $t && timeout 400 python bench.py) 2> $O/full_$n.err | tail -n 1 > $O/full_$n.json
  python -c "
import json
r = json.load(open('$O/full_$n.json'))
print('$n', 'ms_per_step', r['ms_per_step'], 'sweep', json.dumps(r.get('sweep_summary'))[:300], 'e2e', json.dumps(r.get('e2e'))[:200])"
done
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
rm -rf $D
