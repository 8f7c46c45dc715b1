#!/bin/bash
# A/B of builds on one box: tools/ab_bench.sh "" /tmp/parent/mocha_sigasia2023_b200/libmocha_b200.so ...
#   -> ms per 128-clip step for each library ("" = the in-tree build; any other argument is loaded through MOCHA_LIB)
for lib in "$@"; do
  ms=$(MOCHA_LIB="$lib" python bench.py --steps 300 --no-latency --no-cpu-baseline --no-extras 2>/dev/null | tail -1 | python -c "import json,sys; print(json.loads(sys.stdin.read())['ms_per_step'])")
  echo "[${lib:-in-tree}] $ms"
done
