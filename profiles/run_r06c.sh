#!/bin/bash
# r06c: GPU tests, smoke and the A/B probe of the series modes at HEAD
OUT=${OUT:-out}
mkdir -p $OUT
T=r06c
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
timeout 400 python -m pytest tests -m gpu -q > $OUT/${T}_pytest.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest.log; tail -3 $OUT/${T}_pytest.log
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${T}_smoke.log 2>&1; tail -1 $OUT/${T}_smoke.log
timeout 200 python tests/tools/probe_series_lanes.py 24 3 3 > $OUT/${T}_probe.jsonl 2>&1; grep summary $OUT/${T}_probe.jsonl
