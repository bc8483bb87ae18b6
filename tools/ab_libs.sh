#!/bin/bash
# A/B of library builds on the C2 device leg (L2 flushed / not flushed):  tools/ab_libs.sh "lib1 lib2"
LIBS=${1:?usage: tools/ab_libs.sh "lib1 lib2 ..." (shared objects under nav_gym_b200/)}
for lib in $LIBS; do
  for fl in "" "--no-flush"; do
  NAVGYM_LIB=/root/repo/nav_gym_b200/$lib python bench.py --steps 400 --warmup 50 --no-configs --no-e2e --no-cpu-baseline $fl | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('$lib $fl ms %.4f' % d['ms_per_step'])"
  done
done
