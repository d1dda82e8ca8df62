#!/bin/bash
# r06d: bench line with the two-row series kernel (default) and with the one-row one (SO3D_LOGP_LANES=1) in the same call
# (headline only), and their dumped outputs compared bit for bit
OUT=${OUT:-out}
mkdir -p $OUT
T=r06d
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${T}_gpu.txt 2>&1; cat $OUT/${T}_gpu.txt
D=$(mktemp -d)
timeout 480 python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs $D/two_row > $OUT/${T}_bench.json 2> $OUT/${T}_bench.err; echo "bench exit $?"
SO3D_LOGP_LANES=1 timeout 100 python bench.py --gpus 1 --steps 20 --warmup 3 --no-extra --no-e2e --no-cpu --no-eager --dump-outputs $D/one_row > $OUT/${T}_bench_one_row.json 2>> $OUT/${T}_bench.err; echo "bench one-row exit $?"
OUT=$OUT python - "$D" <<'PY' | tee $OUT/${T}_compare.txt
import json, os, sys
import numpy as np
d = sys.argv[1]
for name in ("logp", "score"):
    a, b = np.load(f"{d}/one_row/{name}.npy"), np.load(f"{d}/two_row/{name}.npy")
    print(name, a.shape, "identical" if np.array_equal(a.view(np.int32), b.view(np.int32)) else "DIFFERENT")
for tag in ("bench", "bench_one_row"):
    r = json.load(open(os.path.join(os.environ["OUT"], f"r06d_{tag}.json")))
    x = r.get("extra") or {}
    if not x:
        print(tag, "ms_per_step", round(r["ms_per_step"], 4), "value", r["value"], "acc", r["accuracy"]["max_rel_err_f"], r["accuracy"]["max_rel_err_score"])
        continue
    print(tag, "ms_per_step", round(r["ms_per_step"], 4), "value", r["value"], "frac", r["roofline"]["frac"], "acc", r["accuracy"]["max_rel_err_f"], r["accuracy"]["max_rel_err_score"],
          "adaptive", round(x["score_evals_per_sec_series_adaptive"]["ms_per_step"], 4), "pure", round(x["score_evals_per_sec_series_pure"]["ms_per_step"], 4),
          "auto", round(x["score_evals_per_sec_auto"]["ms_per_step"], 4), "small16384_us", round(x["series_small_batch"]["rows"]["16384"]["us_per_call"], 2),
          "e2e", r["e2e"]["value"], "sweep_series_ms", {k: round(v["series"]["ms"], 3) for k, v in x.get("size_sweep", {}).get("sizes", {}).items()})
PY
rm -rf "$D"
