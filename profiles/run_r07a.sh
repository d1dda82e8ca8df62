#!/bin/bash
# r07a: source forms of the two-row series kernel with the kappa-form derivative, against HEAD (w form), all builds in one
# process, alternating; with a resident-CTA sweep.  The builds (tests/tools/build_variant.py, ranked first by
# profiles/sass_series_reads.py):
#   head      the parent commit's library
#   k_oO_bB   python tests/tools/build_variant.py k_oO_bB --kernels-only -DSO3D_SERIES2_ORDER=O -DSO3D_SERIES2_BLOCK=B
OUT=${OUT:-out}
mkdir -p $OUT
T=r07a
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
V=build/variants
timeout 900 python tests/tools/probe_series_forms.py --rounds 5 --ctas 4,5,6,7 head=$V/libso3d_head.so \
  k_o0_b32=$V/libso3d_k_o0_b32.so k_o2_b32=$V/libso3d_k_o2_b32.so k_o3_b32=$V/libso3d_k_o3_b32.so \
  k_o0_b16=$V/libso3d_k_o0_b16.so k_o3_b16=$V/libso3d_k_o3_b16.so k_o0_b64=$V/libso3d_k_o0_b64.so k_o1_b64=$V/libso3d_k_o1_b64.so \
  > $OUT/${T}_series_forms.jsonl 2> $OUT/${T}_probe.err; echo "probe exit $?"
grep -v '"round"' $OUT/${T}_series_forms.jsonl | grep -v ctas
tail -3 $OUT/${T}_probe.err
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv,noheader >> $OUT/${T}_gpu.txt 2>&1
