#!/bin/bash
# r09a: the exact (table-free) IGSO(3) sampler -- its GPU tests, the whole GPU suite, smoke(), the bench line and the
# rate probe (tests/tools/probe_igso3_exact.py), in one call
OUT=${OUT:-out}
mkdir -p $OUT
T=r09a
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
timeout 900 python -m pytest tests/test_gpu_igso3_exact.py -m gpu -q -x -s > $OUT/${T}_pytest_igso3_exact.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest_igso3_exact.log; tail -15 $OUT/${T}_pytest_igso3_exact.log
timeout 600 python tests/tools/probe_igso3_exact.py --out $OUT/${T}_probe_igso3_exact.jsonl > /dev/null 2> $OUT/${T}_probe.err; echo "probe exit $?"; cat $OUT/${T}_probe_igso3_exact.jsonl; tail -5 $OUT/${T}_probe.err
timeout 1200 python -m pytest tests -m gpu -q > $OUT/${T}_pytest.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest.log; tail -3 $OUT/${T}_pytest.log
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${T}_smoke.log 2>&1; echo "smoke exit $?"; tail -1 $OUT/${T}_smoke.log
timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/${T}_bench.json 2> $OUT/${T}_bench.err; echo "bench exit $?"; head -c 300 $OUT/${T}_bench.json; echo
