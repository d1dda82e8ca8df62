"""Cost of the IGSO(3) entropy kernel (ops.igso3_entropy, so3d_igso3_entropy_f32) on cuda:0 (prints JSON lines; --out FILE
also writes them): 2^20 and 2^24 rows, eps shared (one value, 0.1, in every row) or per row log-uniform over the schedule's
range [4.67e-3, 1], with and without the dH/deps output.  CUDA events around repeated launches.

The kernel reads 4 B and writes 4 or 8 B per row; each record gives rows/s and its time over that HBM floor at 7.7 TB/s.  Per
row it evaluates 16 quadrature nodes (a few MUFU operations and ~40-60 FP32 instructions each), so the floor is far below the
time: the kernel is bound by its arithmetic.  The first line records the card and its power limit.

    python tests/tools/probe_igso3_entropy.py [--out profiles/xyz.jsonl]
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
    for n in (1 << 20, 1 << 24):
        per_row = torch.exp(torch.empty(n, device=dev).uniform_(math.log(4.67e-3), 0.0))
        for kind, eps in (("shared eps 0.1", torch.full((n,), 0.1, device=dev)), ("per-row eps", per_row)):
            for grad in (False, True):
                ms = time_ms(lambda: ops.igso3_entropy(eps, want_grad=grad), 20 if n > (1 << 20) else 200)
                bytes_ = n * (4 + 4 + (4 if grad else 0))
                floor = bytes_ / HBM * 1e3
                emit({"rows": n, "eps": kind, "grad": grad, "ms": round(ms, 4), "rows_per_s": float(f"{n / ms * 1e3:.4g}"),
                      "bytes_per_row": bytes_ // n, "hbm_floor_ms": round(floor, 4), "time_over_hbm_floor": round(ms / floor, 1)})


if __name__ == "__main__":
    main()
