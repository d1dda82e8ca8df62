"""A/B of the series evaluator: one row per thread (SO3D_LOGP_LANES=1) vs two rows per thread with packed FP32 (default),
with a sweep of the two-row kernel's resident CTAs per SM (SO3D_CTAS_PER_SM):
    python tests/tools/probe_series_lanes.py [log2_rows] [rounds] [ctas,ctas,...]
-> one JSON line per (variant, mode, round), then one summary line per (variant, mode): ms per launch (min / median / spread
over rounds) and whether the outputs equal the one-row kernel's bit for bit.  The variants alternate within every round so
that a drift of the clocks hits all of them alike.  Inputs: the bench's E-set (bench.make_eset), L = 2000."""
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import diffusion_extensions_b200 as dx  # noqa: E402

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 24
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
sweep = [int(c) for c in sys.argv[3].split(",")] if len(sys.argv) > 3 else [2, 3, 4, 5, 6]
n, L, reps = 1 << lg, 2000, 10
dev = torch.device("cuda:0")
dx._lib.load()
R, eps = bench.make_eset(n, dev, 1234)
logp = torch.empty(n, device=dev)
score = torch.empty(n, 3, device=dev)
call, ptr = dx._lib.call, dx._lib.ptr
MODES = (("series", dx._lib.MODE_SERIES), ("series_adaptive", dx._lib.MODE_SERIES_ADAPTIVE), ("series_pure", dx._lib.MODE_SERIES_PURE))
VARIANTS = [("one_row", "1", None), ("two_row", "2", None)] + [(f"two_row_ctas{c}", "2", c) for c in sweep]


def set_variant(lanes, ctas):
    os.environ["SO3D_LOGP_LANES"] = lanes  # both are read by the library on every call
    if ctas is None:
        os.environ.pop("SO3D_CTAS_PER_SM", None)
    else:
        os.environ["SO3D_CTAS_PER_SM"] = str(ctas)


def timed(mode, rows):
    fn = lambda: call("so3d_igso3_logp_score_f32", ptr(R), ptr(eps), 1, ptr(logp), ptr(score), None, rows, mode, L, device=dev)
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


print(json.dumps({"gpu": torch.cuda.get_device_name(dev), "rows": n, "L": L, "reps": reps, "rounds": rounds}), flush=True)
ref = {}
times = {}
for r in range(rounds):
    order = VARIANTS if r % 2 == 0 else VARIANTS[::-1]
    for name, lanes, ctas in order:
        set_variant(lanes, ctas)
        for mname, mode in MODES:
            ms = timed(mode, n)
            if name == "one_row" and mname not in ref:
                ref[mname] = (logp.clone(), score.clone())
            same = None
            if mname in ref:
                same = bool(torch.equal(ref[mname][0], logp) and torch.equal(ref[mname][1], score))
            times.setdefault((name, mname), []).append(ms)
            print(json.dumps({"round": r, "variant": name, "mode": mname, "ms": round(ms, 4), "equal_to_one_row": same}), flush=True)
        # small batch just above the one-warp-per-rotation threshold (bench.py's series_small_batch 16384 row)
        ms = timed(dx._lib.MODE_SERIES, 16384)
        times.setdefault((name, "series_16384"), []).append(ms)
set_variant("2", None)
os.environ.pop("SO3D_LOGP_LANES", None)
for (name, mname), v in times.items():
    med = statistics.median(v)
    one = statistics.median(times[("one_row", mname)])
    print(json.dumps({"summary": name, "mode": mname, "ms_min": round(min(v), 4), "ms_median": round(med, 4),
                      "spread": round((max(v) - min(v)) / med, 4), "speedup_vs_one_row": round(one / med, 4)}), flush=True)
