#!/bin/bash
# r08a: the capturable SE(3) arm -- the new GPU tests, the whole GPU suite, smoke(), the bench line and the
# eager-vs-graph / by-value-vs-dseed probe (tests/tools/probe_se3_graph.py), in one call
OUT=${OUT:-out}
mkdir -p $OUT
T=r08a
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
timeout 600 python -m pytest tests/test_gpu_se3_graph.py -m gpu -q -x > $OUT/${T}_pytest_se3_graph.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest_se3_graph.log; tail -15 $OUT/${T}_pytest_se3_graph.log
timeout 900 python -m pytest tests -m gpu -q > $OUT/${T}_pytest.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest.log; tail -3 $OUT/${T}_pytest.log
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${T}_smoke.log 2>&1; echo "smoke exit $?"; tail -1 $OUT/${T}_smoke.log
timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/${T}_bench.json 2> $OUT/${T}_bench.err; echo "bench exit $?"; head -c 300 $OUT/${T}_bench.json; echo
timeout 900 python tests/tools/probe_se3_graph.py --out $OUT/${T}_probe_se3_graph.jsonl > /dev/null 2> $OUT/${T}_probe.err; echo "probe exit $?"; cat $OUT/${T}_probe_se3_graph.jsonl; tail -5 $OUT/${T}_probe.err
