#!/bin/bash
# scratch: per-kernel timings of one training step for several builds of the library (libroomslam_b200<suffix>.so)
cd "$GRAFT_REPO_ROOT" 2>/dev/null || cd /root/repo
mkdir -p gpurun_out
{
for B in ${AB_SIZES:-1024}; do
  for lib in ${AB_LIBS:-_base "" _vA _vP _vAP}; do
    echo "=== lib '$lib' B $B"
    RS_LIB=$PWD/roomslam_b200/libroomslam_b200$lib.so timeout 300 python tools/step_probe.py $B 2>&1 | grep "rec_\|ms/step" | cut -c1-200
  done
done
} > gpurun_out/ab_variants.txt 2>&1
cat gpurun_out/ab_variants.txt
