#!/bin/bash
# A/B of the pedestrian-lidar kernel builds on the crowd configuration: tools/ab_agent_scan.sh "lib1 lib2"
LIBS=${1:?usage: tools/ab_agent_scan.sh "lib1 lib2 ..." (shared objects under nav_gym_b200/)}
for lib in $LIBS; do
  echo "== $lib"
  NAVGYM_LIB=/root/repo/nav_gym_b200/$lib python tools/bench_configs.py crowd
done
