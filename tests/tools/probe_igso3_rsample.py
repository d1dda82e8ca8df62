"""Cost of the reparameterised exact IGSO(3) draw on cuda:0 at 2^24 rows (prints JSON lines; --out FILE also writes them):

  * the forward, ops.igso3_sample_exact with the angle and axis outputs rsample keeps for its backward;
  * the backward kernel alone, ops.igso3_rsample_bwd (dw/deps and G N^T per row);
  * IsotropicGaussianSO3.rsample forward plus backward through autograd (eps requires grad), upstream G given;
for shared eps 0.1 and per-row eps log-uniform over the schedule's range [4.67e-3, 1].  CUDA events around repeated launches.

The backward reads G (36 B), the axis (12 B), the angle (4 B) and per-row eps (4 B), and writes g_eps (4 B) and g_mean
(36 B) per row; each backward record gives its time over that HBM floor at 7.7 TB/s.  The first line records the card and
its power limit.

    python tests/tools/probe_igso3_rsample.py [--out profiles/xyz.jsonl]
"""
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch

import diffusion_extensions_b200 as dx
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
    n = 1 << 24
    eps_row = torch.exp(torch.empty(n, device=dev).uniform_(math.log(4.67e-3), 0.0))
    G = torch.randn(n, 3, 3, device=dev)
    for kind, eps in (("shared eps 0.1", torch.tensor(0.1, device=dev)), ("per-row eps", eps_row)):
        per_row = eps.numel() > 1
        fwd = time_ms(lambda: ops.igso3_sample_exact(eps, (n,), seed=1, rng_offset=0, want_angle=True, want_axis=True), 10)
        _, ang, ax = ops.igso3_sample_exact(eps, (n,), seed=1, rng_offset=0, want_angle=True, want_axis=True)
        bwd = time_ms(lambda: ops.igso3_rsample_bwd(eps, ang, ax, G, seed=1, rng_offset=0), 10)
        bytes_ = n * (36 + 12 + 4 + (4 if per_row else 0) + 4 + 36)
        e = eps.clone().requires_grad_()
        d = dx.IsotropicGaussianSO3(e, sampler="exact")

        def step():
            e.grad = None
            d.rsample((n,) if not per_row else ()).backward(G)

        both = time_ms(step, 10)
        emit({"rows": n, "eps": kind, "forward_ms": round(fwd, 4), "backward_kernel_ms": round(bwd, 4),
              "rsample_fwd_bwd_ms": round(both, 4), "backward_over_forward": round(bwd / fwd, 3),
              "backward_bytes_per_row": bytes_ // n, "backward_hbm_floor_ms": round(bytes_ / HBM * 1e3, 4),
              "backward_time_over_hbm_floor": round(bwd / (bytes_ / HBM * 1e3), 2)})


if __name__ == "__main__":
    main()
