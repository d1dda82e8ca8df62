#!/bin/bash
# r06b: register budget of the two-row series kernel: builds with SO3D_SERIES2_MINCTAS=7 (<= 72 registers) and 8 (<= 64)
#   python tests/tools/build_variant.py m7 --kernels-only -DSO3D_SERIES2_MINCTAS=7   (and m8 ... =8)
# next to the shipped build (SO3D_SERIES2_MINCTAS=4: 74 registers, 6 resident CTAs; series_adaptive capped at 3 CTAs per SM)
OUT=${OUT:-out}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r06b_gpu.txt 2>&1
for v in shipped m7 m8; do
  if [ $v = shipped ]; then unset SO3D_LIB_PATH; else export SO3D_LIB_PATH=build/variants/libso3d_$v.so; fi
  python tests/tools/probe_series_lanes.py 24 3 3,6 > $OUT/r06b_probe_$v.jsonl 2>&1
  echo $v; grep summary $OUT/r06b_probe_$v.jsonl
done
cat $OUT/r06b_gpu.txt
