#!/bin/bash
# Same bits (bench dumps at 32 and 256 rows of both builds), the whole -m gpu suite and
# smoke() on this tree.  BASE_TREE: a built checkout of the parent commit.
set -u
BASE_TREE=${BASE_TREE:?set BASE_TREE to a built checkout of the parent commit}
O=${OUT_DIR:-profiles/r6/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
D=$(mktemp -d)
for b in 32 256; do
  for t in "$BASE_TREE" .; do
    n=$([ $t = . ] && echo new || echo old)
    (cd $t && timeout 100 python bench.py --steps 20 --no-sweep --no-e2e --no-cpu-baseline \
      --batch $b --dump-outputs $D/$n/$b) > /dev/null 2>&1
    echo "dump $n $b rc=$?"
  done
  same=0; diff=0
  for f in $D/old/$b/*.npy; do
    if cmp -s $f $D/new/$b/$(basename $f); then same=$((same + 1)); else diff=$((diff + 1)); echo "DIFFERENT $b $(basename $f)"; fi
  done
  echo "batch $b: $same identical, $diff different, $(ls $D/new/$b | wc -l) files in new"
done
rm -rf $D
timeout 60 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -n 1
timeout 360 python -m pytest tests -m gpu -q -p no:cacheprovider > $O/tests_gpu.log 2>&1
echo "gpu suite rc=$?"; tail -n 1 $O/tests_gpu.log
