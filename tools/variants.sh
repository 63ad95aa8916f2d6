#!/bin/bash
# build K4 variants on the GPU box (only hl_astar.cu is recompiled, ~20 s) and time each:
#   tools/variants.sh "<flags1>" "<flags2>" ...      e.g.  tools/variants.sh "" "-DAQ_FAR=3" "-DAQ_SLOTS=4 -DAQ_GD_UNROLL=2"
cd "$(dirname "$0")/.."
P=headland_trajectory_planning_b200
build() {
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC --fmad=true $1 -c $P/csrc/hl_astar.cu -o $P/csrc/hl_astar.o > /dev/null 2>&1 || return 1
  nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $P/libheadland_b200.so $P/csrc/*.o -lcudart
}
for f in "$@"; do
  build "$f" || { echo "build failed: $f"; continue; }
  echo "=== $f"
  REPS=${REPS:-6} timeout 180 python tools/profile_k4.py 4096 2>&1 | tail -2 | cut -c1-420
done
build ""
