"""Rates of the exact IGSO(3) sampler (ops.igso3_sample_exact) and of the table path it replaces for per-row eps, on cuda:0
(prints JSON lines; --out FILE also writes them there):

  * exact sampler at 2^20 and 2^24 rows, shared eps and per-row eps log-uniform over the schedule's range [4.67e-3, 1],
    on the one-row (CTA) and two-row engines (SO3D_ROW_LANES=1 / 2), CUDA events around repeated launches;
  * table path at 2^20 rows of per-row eps: the CDF-table build (ops.igso3_cdf_table) and the sampling from it, timed
    apart.

Each record carries the bound that applies: the exact sampler reads 4 B (per-row eps) and writes 36 B per row, so its
HBM floor is (40 B x rows) / 7.7 TB/s; it runs far above that floor, i.e. it is bound by its arithmetic (the record gives
the share of the HBM floor).  The first line records the card and its power limit.

    python tests/tools/probe_igso3_exact.py [--out profiles/xyz.jsonl]
"""
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch

from diffusion_extensions_b200 import ops

dev = torch.device("cuda:0")
OUT = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
_out = open(OUT, "w") if OUT else None
HBM = 7.7e12


def emit(rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if _out:
        _out.write(line + "\n")
        _out.flush()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(dev)


def time_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    emit({"card": card(), "torch": torch.__version__})
    lo, hi = math.log(4.67e-3), 0.0
    for log2n in (20, 24):
        n = 1 << log2n
        eps_row = torch.exp(torch.empty(n, device=dev).uniform_(lo, hi))
        R = torch.empty(n, 3, 3, device=dev)
        for lanes in ("1", "2"):
            os.environ["SO3D_ROW_LANES"] = lanes
            for kind, eps in (("shared eps 0.1", 0.1), ("shared eps 1.0", 1.0), ("per-row eps", eps_row)):
                reps = 20 if log2n == 20 else 5
                ms = time_ms(lambda: ops.igso3_sample_exact(eps, (n,), seed=1, rng_offset=0), reps)
                bytes_ = n * (36 + (4 if kind == "per-row eps" else 0))
                emit({"what": "exact sampler", "rows": n, "eps": kind, "engine": {"1": "one-row", "2": "two-row"}[lanes],
                      "ms": round(ms, 4), "samples_per_s": n / (ms * 1e-3),
                      "bound": "arithmetic (HBM floor %.4f ms = %.1f%% of the time)" % (bytes_ / HBM * 1e3, 100 * bytes_ / HBM / (ms * 1e-3))})
        os.environ.pop("SO3D_ROW_LANES", None)
        del R
    # table path, 2^20 rows of per-row eps: build (999 fp64 densities + a prefix sum per row) and sampling, apart
    n = 1 << 20
    eps_row = torch.exp(torch.empty(n, device=dev).uniform_(lo, hi))
    build_ms = time_ms(lambda: ops.igso3_cdf_table(eps_row), 3, warm=1)
    table = ops.igso3_cdf_table(eps_row)
    row_idx = torch.arange(n, device=dev)
    samp_ms = time_ms(lambda: ops.igso3_sample(table, (n,), row_idx=row_idx, seed=1, rng_offset=0), 20)
    emit({"what": "table path, per-row eps", "rows": n, "table_bytes": table.numel() * 4, "build_ms": round(build_ms, 3),
          "sample_ms": round(samp_ms, 4), "samples_per_s_incl_build": n / ((build_ms + samp_ms) * 1e-3),
          "bound": "build: fp64 arithmetic (999 fp64 closed-form densities per row); sampling: reads of the table rows"})
    exact_ms = time_ms(lambda: ops.igso3_sample_exact(eps_row, (n,), seed=1, rng_offset=0), 20)
    emit({"what": "exact sampler, same eps", "rows": n, "ms": round(exact_ms, 4), "speedup_vs_table_incl_build": (build_ms + samp_ms) / exact_ms})


if __name__ == "__main__":
    main()
