#!/bin/bash
# One `ncu --set full` capture per hot kernel of the encoder chain (B200_PROFILING.md recipe).
# usage (on the GPU box): bash scripts/ncu_full.sh <tag> [kernel-regex ...]   -> gpurun_out/<tag>_<kernel>.ncu-rep
tag=${1:-r01}; shift
kernels=("$@")
[ ${#kernels[@]} -eq 0 ] && kernels=(project_kernel segment_fps_wide_kernel assign_labels_kernel quantize_pack_kernel)
mkdir -p gpurun_out
for k in "${kernels[@]}"; do
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:$k -s 1 -c 1 -f \
    -o gpurun_out/${tag}_$k python scripts/profile_chain.py ${FRAMES:-296} ${REPS:-2} > gpurun_out/${tag}_$k.log 2>&1
  tail -2 gpurun_out/${tag}_$k.log
done
