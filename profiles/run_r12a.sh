#!/bin/bash
# r12a: the IGSO(3) entropy -- its GPU tests, the cost probe (tests/tools/probe_igso3_entropy.py), the whole GPU suite,
# smoke() and the bench line, in one call
OUT=${OUT:-out}
mkdir -p $OUT
T=r12a
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
timeout 600 python -m pytest -p no:cacheprovider tests/test_gpu_igso3_entropy.py -m gpu -q -s > $OUT/${T}_pytest_entropy.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest_entropy.log; grep -E "err/tol|MC|passed|failed|Error" $OUT/${T}_pytest_entropy.log | tail -40
timeout 300 python tests/tools/probe_igso3_entropy.py --out $OUT/${T}_probe_igso3_entropy.jsonl > /dev/null 2> $OUT/${T}_probe.err; echo "probe exit $?"; cat $OUT/${T}_probe_igso3_entropy.jsonl; tail -5 $OUT/${T}_probe.err
timeout 1500 python -m pytest -p no:cacheprovider tests -m gpu -q > $OUT/${T}_pytest.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest.log; tail -3 $OUT/${T}_pytest.log
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${T}_smoke.log 2>&1; echo "smoke exit $?" | tee -a $OUT/${T}_smoke.log
timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/${T}_bench.json 2> $OUT/${T}_bench.err; echo "bench exit $?"; head -c 300 $OUT/${T}_bench.json; echo
