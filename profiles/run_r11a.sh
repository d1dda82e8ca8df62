#!/bin/bash
# r11a: the reparameterised exact IGSO(3) draw -- its GPU tests, the cost probe (tests/tools/probe_igso3_rsample.py), the
# whole GPU suite, smoke() and the bench line, in one call
OUT=${OUT:-out}
mkdir -p $OUT
T=r11a
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
timeout 900 python -m pytest -p no:cacheprovider tests/test_gpu_igso3_rsample.py -m gpu -q -s > $OUT/${T}_pytest_rsample.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest_rsample.log; grep -E "err/tol|SE|mean.grad|passed|failed|Error" $OUT/${T}_pytest_rsample.log | tail -40
timeout 600 python tests/tools/probe_igso3_rsample.py --out $OUT/${T}_probe_igso3_rsample.jsonl > /dev/null 2> $OUT/${T}_probe.err; echo "probe exit $?"; cat $OUT/${T}_probe_igso3_rsample.jsonl; tail -5 $OUT/${T}_probe.err
timeout 1500 python -m pytest -p no:cacheprovider tests -m gpu -q > $OUT/${T}_pytest.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest.log; tail -3 $OUT/${T}_pytest.log
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${T}_smoke.log 2>&1; echo "smoke exit $?" | tee -a $OUT/${T}_smoke.log
timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/${T}_bench.json 2> $OUT/${T}_bench.err; echo "bench exit $?"; head -c 300 $OUT/${T}_bench.json; echo
