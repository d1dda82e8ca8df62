"""A/B of source forms of the two-row series kernel, several builds of the library in ONE process:
    python tests/tools/probe_series_forms.py [--rounds R] [--log2-rows N] [--ctas c,c,...] NAME=LIB [NAME=LIB ...]
The first build is the reference.  Every round times every build (the builds alternate, and their order flips every
round, so that a drift of the clocks hits all of them alike) in the series modes at 2^N E-set rows, L = 2000, and the
`series` mode at 16 384 rows (the bench's small batch).  `--ctas` adds, per build, `series` with the resident CTAs per SM
capped (SO3D_CTAS_PER_SM).  Output: one JSON line per timing, then per (build, mode) ms min / median / spread over
rounds and the speedup against the reference, then per build how its `series` outputs differ from the reference's:
bit-identical rows, and the largest difference in units of 2^-23 relative (of f for log f, of the score vector's norm for
the score), split into rows the closed-form guard replaces (omega > 4.2 eps, eps <= 1) and the others.  Builds come from tests/tools/build_variant.py."""
import argparse
import ctypes
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import diffusion_extensions_b200 as dx  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("builds", nargs="+")
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--log2-rows", type=int, default=24)
ap.add_argument("--ctas", default="")
a = ap.parse_args()
n, L, reps = 1 << a.log2_rows, 2000, 10
dev = torch.device("cuda:0")
sig = dx._lib.SIGNATURES["so3d_igso3_logp_score_f32"]
libs = []
for spec in a.builds:
    name, path = spec.split("=", 1)
    lib = ctypes.CDLL(os.path.abspath(path))  # RTLD_LOCAL: each build keeps its own kernels and constant tables
    fn = lib.so3d_igso3_logp_score_f32
    fn.argtypes, fn.restype = sig, ctypes.c_int
    libs.append((name, fn))
R, eps = bench.make_eset(n, dev, 1234)
logp = torch.empty(n, device=dev)
score = torch.empty(n, 3, device=dev)
MODES = (("series", dx._lib.MODE_SERIES), ("series_adaptive", dx._lib.MODE_SERIES_ADAPTIVE), ("series_pure", dx._lib.MODE_SERIES_PURE))
ctas = [int(c) for c in a.ctas.split(",") if c]


def timed(fn, mode, rows):
    stream = torch.cuda.current_stream().cuda_stream
    run = lambda: fn(R.data_ptr(), eps.data_ptr(), 1, logp.data_ptr(), score.data_ptr(), None, rows, mode, L, stream)
    for _ in range(2):
        assert run() == 0
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


print(json.dumps({"gpu": torch.cuda.get_device_name(dev), "rows": n, "L": L, "reps": reps, "rounds": a.rounds,
                  "builds": a.builds}), flush=True)
times, outs = {}, {}
for r in range(a.rounds):
    for name, fn in (libs if r % 2 == 0 else libs[::-1]):
        os.environ.pop("SO3D_CTAS_PER_SM", None)
        for mname, mode in MODES:
            ms = timed(fn, mode, n)
            if mname == "series" and name not in outs:
                outs[name] = (logp.clone(), score.clone())
            times.setdefault((name, mname), []).append(ms)
            print(json.dumps({"round": r, "build": name, "mode": mname, "ms": round(ms, 4)}), flush=True)
        times.setdefault((name, "series_16384"), []).append(timed(fn, dx._lib.MODE_SERIES, 16384))
        for c in ctas:
            os.environ["SO3D_CTAS_PER_SM"] = str(c)  # read by the library on every call
            ms = timed(fn, dx._lib.MODE_SERIES, n)
            times.setdefault((name, f"series_ctas{c}"), []).append(ms)
            print(json.dumps({"round": r, "build": name, "mode": f"series_ctas{c}", "ms": round(ms, 4)}), flush=True)
        os.environ.pop("SO3D_CTAS_PER_SM", None)
ref = libs[0][0]
for (name, mname), v in times.items():
    med, rmed = statistics.median(v), statistics.median(times[(ref, mname)])
    print(json.dumps({"summary": name, "mode": mname, "ms_min": round(min(v), 4), "ms_median": round(med, 4),
                      "spread": round((max(v) - min(v)) / med, 4), "speedup_vs_" + ref: round(rmed / med, 4)}), flush=True)
# output differences against the reference, rows the guard replaces vs the others (rows within 1e-5 of the guard's edge,
# where this omega and the kernel's may fall on different sides, are left out of both)
w = dx.ops.log_vec(R).norm(dim=-1)
guard = (eps <= 1.0) & (w > 4.2 * eps * (1 + 1e-5))
below = (eps > 1.0) | (w < 4.2 * eps * (1 - 1e-5))
lp0, sc0 = outs[ref]
for name, _ in libs[1:]:
    lp, sc = outs[name]
    rep = {"compare": name, "vs": ref, "guarded_rows": int(guard.sum()), "unguarded_rows": int(below.sum())}
    # differences in units of 2^-23 relative: of f for log f, of the score vector's norm for the score
    d_lp = (lp.double() - lp0.double()).abs() / 2.0 ** -23
    d_sc = (sc.double() - sc0.double()).norm(dim=1) / (sc0.double().norm(dim=1) * 2.0 ** -23).clamp_min(1e-300)
    for tag, x, y, d in (("logp", lp, lp0, d_lp), ("score", sc.reshape(n, 3), sc0.reshape(n, 3), d_sc)):
        same = (x.reshape(n, -1).view(torch.int32) == y.reshape(n, -1).view(torch.int32)).all(dim=1)
        rep[tag] = {"identical_guarded": bool(same[guard].all()), "identical_rows": int(same.sum()),
                    "max_rel_ulps_unguarded": round(float(d[below].max()), 3),
                    "max_rel_ulps_guarded": round(float(d[guard].max()), 3) if guard.any() else 0.0}
    print(json.dumps(rep), flush=True)
