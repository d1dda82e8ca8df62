"""SE(3) arm, eager vs CUDA graph, in one process on cuda:0 (prints JSON lines; --out FILE also writes them there):

  * training step  -- SE3Diffusion + a small AffineT denoiser + Adam: eager step vs make_graphed_train_step, at (4,)
    (prot_train.py's batch), (4, 256) and (64, 256) frames; device events around 200 steps;
  * sampling loop  -- 1000 steps of p_sample_loop, eager vs cuda_graph=True, at (4, 256), (20 000,) and (64, 256);
    host clock around whole loops ending in a synchronise;
  * kernel cost    -- by-value vs device-seed kernels (so3d_se3_q_sample[_dseed]_f32, shared-t so3d_se3_p_sample[_dseed]_f32)
    at 2^24 rows (inputs of 2^24 * 48 B, larger than L2), alternating, CUDA events, several rounds.

The first line records the card and its power limit.

    python tests/tools/probe_se3_graph.py [--out profiles/xyz.jsonl]
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch

import diffusion_extensions_b200 as dx
from diffusion_extensions_b200 import ops

dev = torch.device("cuda:0")
OUT = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
_out = open(OUT, "w") if OUT else None


def emit(rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if _out:
        _out.write(line + "\n")
        _out.flush()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(dev)


class Net(torch.nn.Module):
    """A small AffineT denoiser (a per-frame MLP on rotation, translation and step)."""

    def __init__(self, width=64):
        super().__init__()
        self.net = torch.nn.Sequential(torch.nn.Linear(13, width), torch.nn.SiLU(), torch.nn.Linear(width, width), torch.nn.SiLU(),
                                       torch.nn.Linear(width, 6))

    def forward(self, x, t):
        tt = t.reshape(tuple(t.shape) + (1,) * (x.shift.dim() - t.dim())).expand(x.shift.shape[:-1] + (1,)).float() / 1000
        h = self.net(torch.cat([x.rot.flatten(-2), x.shift / 75.0, tt], -1))
        return dx.AffineGrad(h[..., :3], h[..., 3:])


def frames(shape):
    return dx.AffineT(ops.quat_to_rmat(torch.randn(*shape, 4, device=dev)), torch.randn(*shape, 3, device=dev) * 10)


def train_leg(shape, graph, reps=200):
    torch.manual_seed(0)
    net = Net().to(dev)
    proc = dx.SE3Diffusion(net).to(dev)
    proc.tables(); proc.guides()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, capturable=graph)
    x0 = frames(shape)

    def eager():
        opt.zero_grad(set_to_none=True)
        loss = proc(x0)
        loss.backward()
        opt.step()
        return loss

    run = eager
    if graph:
        stepper = proc.make_graphed_train_step(opt, x0)
        run = lambda: stepper(x0)
    for _ in range(20):
        loss = run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(reps):
        loss = run()
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return {"leg": "train_step", "frames": list(shape), "cuda_graph": graph, "ms_per_step": round(e0.elapsed_time(e1) / reps, 4),
            "wall_ms_per_step": round(1e3 * wall / reps, 4), "loss": float(loss)}


def loop_leg(shape, graph, reps=3):
    torch.manual_seed(0)
    net = Net().to(dev).eval()
    proc = dx.SE3Diffusion(net).to(dev)
    proc.p_sample_loop(shape, cuda_graph=graph)                     # warm-up (and capture)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        x = proc.p_sample_loop(shape, cuda_graph=graph)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    ok = bool(torch.isfinite(x.shift).all())
    return {"leg": "p_sample_loop", "steps": proc.num_timesteps, "frames": list(shape), "cuda_graph": graph, "loop_ms": round(1e3 * min(times), 2),
            "loop_ms_all": [round(1e3 * t, 2) for t in times], "finite": ok}


def kernel_leg(rounds=5, reps=20):
    n = 1 << 24
    torch.manual_seed(0)
    proc = dx.SE3Diffusion(None).to(dev)
    fwd, post, _ = proc.tables()
    g = proc.guides()[0]
    x = frames((n,))
    t = torch.randint(0, 1000, (n,), device=dev)
    tp = torch.tensor([500], device=dev)
    pr, ps = torch.randn(n, 3, device=dev) * 0.3, torch.randn(n, 3, device=dev)
    qargs = (proc.sqrt_alphas_cumprod, proc.sqrt_one_minus_alphas_cumprod, fwd, 75.0)
    sched = (proc.sqrt_recip_alphas_cumprod, proc.sqrt_recipm1_alphas_cumprod, proc.posterior_mean_coef1, proc.posterior_mean_coef2)
    sigma = proc._sigma()
    S = 12345
    seed_t = torch.full((1,), S, dtype=torch.int64, device=dev)
    calls = {
        ("q_sample", "by_value"): lambda: ops.se3_q_sample_fused(x.rot, x.shift, t, *qargs, seed=S, rng_offset=0, guide=g),
        ("q_sample", "dseed"): lambda: ops.se3_q_sample_fused(x.rot, x.shift, t, *qargs, seed=seed_t, rng_offset=0, guide=g),
        ("p_sample_shared_t", "by_value"): lambda: ops.se3_p_sample_fused(x.rot, x.shift, pr, ps, tp, *sched, sigma, 75.0, post_cdf=post, seed=S,
                                                                          rng_offset=0),
        ("p_sample_shared_t", "dseed"): lambda: ops.se3_p_sample_fused(x.rot, x.shift, pr, ps, tp, *sched, sigma, 75.0, post_cdf=post, seed=seed_t,
                                                                       rng_offset=0),
    }
    for op in ("q_sample", "p_sample_shared_t"):                      # the two launches agree bit for bit at this size too
        a, b = calls[(op, "by_value")](), calls[(op, "dseed")]()
        va = list(a.values()) if isinstance(a, dict) else list(a)
        vb = list(b.values()) if isinstance(b, dict) else list(b)
        emit({"leg": "kernel_equal", "op": op, "rows": n, "bit_identical": all(torch.equal(u, v) for u, v in zip(va, vb))})
    res = {k: [] for k in calls}
    for f in calls.values():
        f()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, f in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                f()
            e1.record()
            torch.cuda.synchronize()
            res[k].append(e0.elapsed_time(e1) / reps)
    for op in ("q_sample", "p_sample_shared_t"):
        rec = {"leg": "kernel", "op": op, "rows": n, "reps_per_round": reps}
        for kind in ("by_value", "dseed"):
            ms = res[(op, kind)]
            rec[kind] = {"ms_median": round(sorted(ms)[len(ms) // 2], 4), "ms_min": round(min(ms), 4), "ms_max": round(max(ms), 4)}
        rec["dseed_over_by_value"] = round(rec["dseed"]["ms_median"] / rec["by_value"]["ms_median"], 4)
        emit(rec)


emit({"leg": "device", "card": card(), "torch": torch.__version__})
for shape in ((4,), (4, 256), (64, 256)):
    for graph in (False, True):
        emit(train_leg(shape, graph))
for shape in ((4, 256), (20000,), (64, 256)):
    for graph in (False, True):
        emit(loop_leg(shape, graph))
kernel_leg()
