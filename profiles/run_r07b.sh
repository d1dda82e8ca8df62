#!/bin/bash
# r07b: the whole GPU suite, smoke(), and the bench line of the kappa-form build next to the parent commit's library
# (build/variants/libso3d_head.so, w form) with both dumps compared
OUT=${OUT:-out}
mkdir -p $OUT
T=r07b
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
timeout 500 python -m pytest tests -m gpu -q > $OUT/${T}_pytest.log 2>&1; echo "pytest exit $?" >> $OUT/${T}_pytest.log; tail -3 $OUT/${T}_pytest.log
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${T}_smoke.log 2>&1; echo "smoke exit $?"; tail -1 $OUT/${T}_smoke.log
D=$(mktemp -d)
timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs $D/kappa > $OUT/${T}_bench.json 2> $OUT/${T}_bench.err; echo "bench exit $?"
SO3D_LIB_PATH=build/variants/libso3d_head.so timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 --no-sweep --no-cpu --no-e2e --dump-outputs $D/head > $OUT/${T}_bench_head.json 2>> $OUT/${T}_bench.err; echo "bench head exit $?"
OUT=$OUT python - "$D" <<'PY' | tee $OUT/${T}_compare.txt
import json, os, sys
import numpy as np
d = sys.argv[1]
for name in ("logp", "score"):
    a, b = np.load(f"{d}/head/{name}.npy"), np.load(f"{d}/kappa/{name}.npy")
    a2, b2 = a.reshape(a.shape[0], -1).astype(np.float64), b.reshape(b.shape[0], -1).astype(np.float64)
    same = (a.reshape(a.shape[0], -1).view(np.int32) == b.reshape(b.shape[0], -1).view(np.int32)).all(axis=1)
    if name == "logp":
        ulps = np.abs(a2 - b2)[:, 0] / 2.0 ** -23
    else:
        ulps = np.linalg.norm(a2 - b2, axis=1) / np.maximum(np.linalg.norm(a2, axis=1) * 2.0 ** -23, 1e-300)
    print(name, a.shape, "identical rows", int(same.sum()), "of", len(same), "max diff (2^-23 relative)", round(float(ulps.max()), 3))
for tag in ("bench_head", "bench"):
    r = json.load(open(os.path.join(os.environ["OUT"], f"r07b_{tag}.json")))
    x = r.get("extra") or {}
    print(tag, "ms_per_step", round(r["ms_per_step"], 4), "value", r["value"], "frac", r["roofline"]["frac"], "acc", r["accuracy"]["max_rel_err_f"], r["accuracy"]["max_rel_err_score"],
          "adaptive", round(x["score_evals_per_sec_series_adaptive"]["ms_per_step"], 4), "pure", round(x["score_evals_per_sec_series_pure"]["ms_per_step"], 4),
          "auto", round(x["score_evals_per_sec_auto"]["ms_per_step"], 4), "small16384_us", round(x["series_small_batch"]["rows"]["16384"]["us_per_call"], 2),
          "e2e", (r.get("e2e") or {}).get("value"))
PY
rm -rf "$D"
