#!/bin/bash
# Builds align2d.cu variants on the GPU box and times the Align2D stage of one 4096-pair step.
for v in "-DDSDTM_A2D_MINB=2" "-DDSDTM_A2D_MINB=3" "-DDSDTM_A2D_MINB=4"; do
  echo "=== $v"
  touch dsdtm_b200/csrc/align2d.cu
  DSDTM_NVCC_FLAGS="$v" python dsdtm_b200/build.py 2>&1 | grep -E " error |align2d_kernel" -A3 | grep -E "error|Used"
  timeout 120 python scripts/prof_step.py --pairs 4096 --steps 5 --direct 2>&1 | tail -2 | head -1 | cut -c100-160
done
