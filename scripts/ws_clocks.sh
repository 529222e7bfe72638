#!/bin/bash
# Per-phase clocks of the K2q dynamics and policy loops (measurement build: rollout.cu compiled with -DRL_WS_CLOCKS into
# build/clk/librelearn_b200.so, swapped in for the duration of this script).  The env count sets K2q's shape: 2 policy
# warps per CTA at E = 1024, 7 at E = 4096.  usage: bash scripts/ws_clocks.sh <tag> [env counts]
# Build it first (here, after __graft_entry__.build()):
#   mkdir -p build/clk && nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -DRL_WS_CLOCKS \
#       -c relearn_b200/csrc/rollout.cu -o build/clk/rollout.o
#   ls build/*.o | grep -v build/rollout.o | xargs nvcc --shared -o build/clk/librelearn_b200.so build/clk/rollout.o -ldl
R=${1:-r2u}
SIZES=${2:-1024 4096}
O=gpurun_out
mkdir -p $O
cp relearn_b200/librelearn_b200.so /tmp/librelearn_b200.keep
cp build/clk/librelearn_b200.so relearn_b200/librelearn_b200.so
for E in $SIZES; do
  echo "== E=$E"
  timeout -k 5 40 python scripts/sweep_rollout.py $E 160 2>&1 | tail -5
done > $O/${R}_ws_clocks.txt 2>&1
cp /tmp/librelearn_b200.keep relearn_b200/librelearn_b200.so
cat $O/${R}_ws_clocks.txt
