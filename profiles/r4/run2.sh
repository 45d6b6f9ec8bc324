#!/bin/bash
# The whole GPU suite and smoke() on the staged-tail tree.
set -u
O=${OUT_DIR:-profiles/r4/out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
timeout 480 python -m pytest tests -m gpu -q > $O/tests_all.log 2>&1
echo "tests rc=$?"; tail -n 5 $O/tests_all.log
timeout 90 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -n 2
