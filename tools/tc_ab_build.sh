#!/bin/bash
# builds the experiment variants of the library (run here; the .so files travel with gpurun)
set -e
cd "$(dirname "$0")/.."
F="-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=hidden --shared"
S=$(python -c "from nisqa_b200 import build as b; print(' '.join('nisqa_b200/csrc/' + f for f in b.SOURCES))")
mkdir -p nisqa_b200/exp
nvcc $F -DNISQA_TC_TIMING $S -o nisqa_b200/exp/libnisqa_timing.so -ldl &
for v in "$@"; do     # extra variants: name=-DFLAG[,-DFLAG2]
  nvcc $F $(echo "${v#*=}" | tr ',' ' ') $S -o nisqa_b200/exp/libnisqa_${v%%=*}.so -ldl &
done
wait
ls -la nisqa_b200/exp
