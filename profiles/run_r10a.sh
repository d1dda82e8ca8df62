#!/bin/bash
# r10a: the forward maps and the reverse step against fp64 by stratum (tests/test_gpu_fwd_strata.py) with this tree's build,
# the parent commit's build and four one-line mutants of so3d_math.cuh (build/variants/, built from scratch copies of the tree
# with tests/tools/build_variant.py), summarised per configuration; the whole GPU suite, smoke(), and the bench line of the
# parent and this build alternated
OUT=${OUT:-out}
mkdir -p $OUT
T=r10a
V=$PWD/build/variants
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
fwd() { tag=$1; shift; env "$@" timeout 600 python -m pytest -p no:cacheprovider tests/test_gpu_fwd_strata.py -m gpu -q -s > $OUT/${T}_fwd_$tag.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_fwd_$tag.log; }
fwd head SO3D_HEAD=1
for m in parent mut_a mut_b mut_c mut_d; do fwd $m SO3D_LIB_PATH=$V/libso3d_$m.so; done
python - $OUT/$T > $OUT/${T}_fwd_summary.txt <<'PY'
import re, sys
pre = sys.argv[1]
for tag in ("head", "parent", "mut_a", "mut_b", "mut_c", "mut_d"):
    lines = open(f"{pre}_fwd_{tag}.log").read().splitlines()
    print(f"== {tag}: {lines[-2].strip()}")
    title, worst = None, {}
    for l in lines:
        m = re.match(r"  (.{24}) (.{22}) max err +(\S+) +max err/tol +(\S+)", l)
        if m:
            r = float(m.group(4))
            w = worst.setdefault(title, [0.0, "", []])
            if r > w[0]: w[0], w[1] = r, f"{m.group(1).strip()} / {m.group(2).strip()}"
            if not r <= 1.0: w[2].append(f"{m.group(1).strip()} / {m.group(2).strip()}")
        elif l and not l.startswith((" ", "E", "F", ".", "=", "_", "tests/", "pytest")) and "::" not in l:
            title = l.strip()
    for t, (r, where, over) in worst.items():
        print(f"  {t}: max err/tol {r:.3g} at {where}" + (f"; over tolerance in {len(over)} rows, e.g. {'; '.join(over[:3])}" if over else ""))
    fails = sorted({l.split(" - ")[0].replace("FAILED ", "") for l in lines if l.startswith("FAILED")})
    if fails: print("  failed: " + ", ".join(f.split("::")[1] for f in fails))
PY
cat $OUT/${T}_fwd_summary.txt | grep "^=="
timeout 1200 python -m pytest -p no:cacheprovider tests -m gpu -q > $OUT/${T}_pytest_full.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest_full.log; tail -2 $OUT/${T}_pytest_full.log | tee $OUT/${T}_pytest.txt
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${T}_smoke.log 2>&1; echo "smoke exit $?" | tee -a $OUT/${T}_smoke.log
for i in 1 2; do
  for b in parent head; do
    if [ $b = parent ]; then export SO3D_LIB_PATH=$V/libso3d_parent.so; else unset SO3D_LIB_PATH; fi
    timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/${T}_bench_${b}_$i.json 2> $OUT/${T}_bench_${b}_$i.err; echo "bench $b $i exit $?"; head -c 160 $OUT/${T}_bench_${b}_$i.json; echo
  done
done
unset SO3D_LIB_PATH
