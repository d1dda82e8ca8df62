#!/bin/bash
# r06a: series evaluator, one row per thread vs two rows per thread (packed FP32), resident-CTA sweep of the two-row kernel;
# then the series / two-row GPU tests (outputs kept as r06a_series_lanes.jsonl, r06a_pytest.log, r06a_gpu.txt)
OUT=${OUT:-out}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv > $OUT/gpu.txt 2>&1
python tests/tools/probe_series_lanes.py 24 3 2,3,4,5 > $OUT/probe.jsonl 2> $OUT/probe.err
tail -40 $OUT/probe.jsonl
python -m pytest -q -m gpu tests/test_gpu_series_lanes.py tests/test_gpu_parity.py -k "series or two_row or 2pow28" > $OUT/pytest1.log 2>&1
tail -15 $OUT/pytest1.log
cat $OUT/gpu.txt
