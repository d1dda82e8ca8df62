#!/usr/bin/env python
"""Benchmark of the SO(3) diffusion hot path (BASELINE.json metric: IGSO(3) score evals/sec &
reverse-diffusion particle-steps/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n ROWS] [--L 2000] [--dump-outputs DIR]

Headline workload (BASELINE configs[1]): one *step* = one fused launch evaluating log-density and
score of the IGSO(3) truncated series (exactly L = 2000 terms per evaluation, no early exit) on
n = 2^24 random rotations per GPU with per-row eps (E-set of SURVEY 8d).  `value` is device-timed with
the inputs resident in HBM; `e2e` goes through the public Python API from pinned HOST buffers and
back.  `accuracy` is the measured error of exactly those results against the fp64 oracle.  Secondary numbers
(the other BASELINE configs and kernels) are reported under "extra" with their own rooflines, each with the
reference's CPU path (`cpu_baseline`) and the reference's op sequence as stock PyTorch on the same GPU
(`torch_cuda_eager`) beside it.  Rank 0 prints ONE JSON line.

--impl reference times the torch-CPU port of the reference's algorithm (oracle/ref_port.py; the
pure-Python reference cannot travel to the GPU box) on the host cores for the same metric.

--dump-outputs DIR writes the results of the last timed step on rank 0 as DIR/<name>.npy (logp and score;
--impl reference: logp and logp_grad, its gradient in the rotation matrix), a fixed seeded sample of DUMP_ROWS
rows when there are more.  The inputs are the same on every run, so two builds can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "igso3_score_evals_per_sec"
UNIT = "evals/s"
SEED = 1234

# ---- work of the series kernel per term (DESIGN.md section 4) ------------------------------------
# Executed: 7 FP32 instructions (1 FMUL, 4 FFMA, 2 FADD = 11 flop) + 1 MUFU.EX2 + 1 uniform constant load
# (LDCU.64) = 9 issue slots.  SURVEY 8(d) fixed the algorithmic unit for recurrence-based variants at
# >= 10 FP32 lane-instructions per term (bound 1.86e9 evals/s/GPU at 128 lanes/clk/SM); `roofline.frac` uses
# that unit, and the executed mix is reported next to it.
ALGO_LANE_INSTR_PER_TERM = 10
FP32_INSTR_PER_TERM = 7
MUFU_PER_TERM = 1
UNIFORM_PER_TERM = 1
FLOP_PER_TERM = 11
BYTES_PER_EVAL = 56          # 36 R + 4 eps in, 4 logp + 12 score out
BYTES_PER_PARTICLE_STEP = 84 # 36 x_t + 12 pred in, 36 out
BYTES_PER_QSAMPLE = 92       # 36 x0 + 8 t in, 36 x_t + 12 target out
BYTES_PER_SE3_QSAMPLE = 128  # 36 rot0 + 12 shift0 + 8 t in, 36 rot_t + 12 shift_t + 12 + 12 targets out
BYTES_PER_SE3_PSTEP = 120    # 36 rot + 12 shift + 12 + 12 predictions in, 36 rot + 12 shift out (shared t)
# DRAM traffic of the series kernel per evaluation from the ncu --set full capture (profiles/r02p_series_full.md:
# 169.07 MB read + 43.80 MB written for 4 194 304 evaluations; the rest of the 16 B/eval of results is still in L2
# when the kernel ends) -- equal to the algorithmic 40 B/eval of inputs: nothing is re-read.
NCU_DRAM_BYTES_PER_EVAL = (169.070080e6 + 43.798272e6) / 4194304
MMD_LANE_INSTR_PER_PAIR = 41  # executed FP32-pipe instructions per pair of the all-pairs kernel (SASS count, DESIGN.md 4.6)
CPU_SAMPLE_ROWS = 1 << 18     # rows of the bench's own inputs the CPU legs evaluate per call
SAMPLER_B = 1 << 16           # batch of the q_sample / p_sample CPU and CUDA-eager legs (the reference's (1000, B) fp64 table bounds it)
DUMP_ROWS = 1 << 21           # rows --dump-outputs writes at most: 2^21 x (4 + 12) B = 32 MiB of float32 results


def peaks():
    p = {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)", "sm_max_mhz": 1965.0}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update(hbm_gbs=float(m["hbm_gbs"]), sm_max_mhz=float(m.get("sm_max_mhz", 1965.0)), source="measured (MEASURED_PEAKS.json)")
    except Exception:
        pass
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled from before the warm-up until the end of the run; every sample is
    time-stamped so that the ones that fell INSIDE a timed window can be picked out afterwards."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, period_ms=25):
        self.index, self.rows, self.proc, self.period = index, [], None, int(period_ms)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.period)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=3.0):
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def stop(self):
        if self.proc is not None:
            time.sleep(0.1)
            self.proc.terminate()

    def summary(self, windows):
        """windows: [(name, t0, t1)] in time.time() seconds, narrowest first; the first one holding >= 3 samples is reported."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        isnum = lambda s: s.replace(".", "", 1).isdigit()
        out = None
        for wname, t0, t1 in windows:
            rows = [r for ts, r in self.rows if t0 <= ts <= t1]
            sm = [float(r[0]) for r in rows if r and isnum(r[0])]
            mx = [float(r[1]) for r in rows if len(r) > 1 and isnum(r[1])]
            pw = [float(r[2]) for r in rows if len(r) > 2 and isnum(r[2])]
            reasons = [nm for k, nm in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in rows)]
            cand = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                    "samples": len(sm), "window": wname, "period_ms": self.period, "reasons": reasons}
            if out is None or cand["samples"] > out["samples"]:
                out = cand
            if out["samples"] >= 3:
                break
        return out


def make_eset(n, device, seed):
    """E-set of SURVEY 8(d): eps log-uniform in [6.4e-3, 1], omega = eps*sqrt2*k, k~U[0,4] (<= 3.0)."""
    import diffusion_extensions_b200 as dx

    g = torch.Generator(device=device).manual_seed(seed)
    eps = torch.exp(torch.empty(n, device=device).uniform_(math.log(6.4e-3), 0.0, generator=g))
    k = torch.empty(n, device=device).uniform_(0.0, 4.0, generator=g)
    omega = torch.clamp(eps * math.sqrt(2.0) * k, max=3.0)
    del k
    axis = torch.randn(n, 3, device=device, generator=g)
    R = dx.ops.aa_to_rmat(axis, omega)
    return R, eps


def make_eset_cpu(n, seed):
    """The same law on the host (the reference arm runs without a GPU): R by Rodrigues in torch."""
    from oracle import ref_port as P

    g = torch.Generator().manual_seed(seed)
    eps = torch.exp(torch.empty(n).uniform_(math.log(6.4e-3), 0.0, generator=g))
    k = torch.empty(n).uniform_(0.0, 4.0, generator=g)
    ang = torch.clamp(eps * math.sqrt(2.0) * k, max=3.0)
    axis = torch.randn(n, 3, generator=g)
    axis = axis / axis.norm(dim=-1, keepdim=True)
    K = P.hat(axis)
    R = torch.eye(3) + torch.sin(ang)[:, None, None] * K + (1 - torch.cos(ang))[:, None, None] * (K @ K)
    return R, eps


def time_loop(fn, steps, warmup, dist_on):
    """W untimed + K timed calls, bracketed by barrier + synchronize; device time via CUDA events."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_on:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    if dist_on:
        torch.distributed.barrier()
    ms = ev0.elapsed_time(ev1)
    if dist_on:
        tt = torch.tensor([ms], device="cuda")
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        ms = tt.item()
    return ms


# ---------------------------------------------------------------------------------------------------------------
# the reference's algorithm on the host cores / as stock PyTorch on the GPU (oracle/ref_port.py, the checker's port)
# ---------------------------------------------------------------------------------------------------------------
def _timed_reps(fn, seconds_target, min_reps=1, sync=None):
    fn()  # warm-up (thread pool, allocator, cuSOLVER handles)
    if sync:
        sync()
    t0 = time.perf_counter()
    reps = 0
    while True:
        fn()
        reps += 1
        if sync:
            sync()
        dt = time.perf_counter() - t0
        if reps >= min_reps and dt > seconds_target:
            return reps, dt


def reference_legs(R, eps, x0, device, seconds=(10.0, 5.0, 5.0)):
    """The reference's own op sequence (oracle/ref_port.py) on `device` ('cpu': all host threads; 'cuda': stock PyTorch
    eager on the same B200) for the three workloads of BASELINE.md section 3:
      score     IGSO3(eps).log_prob(R) + autograd (distributions.py:74-77,186-190), per-row eps, the bench's own inputs
      q_sample  SO3Diffusion.q_sample (diffusion.py:339-346), per-row t, B = 65 536 (a (1000, B) fp64 table per call)
      p_sample  SO3Diffusion.p_sample (diffusion.py:315-326), zero denoiser, shared t = 500, B = 65 536."""
    from oracle import ref_port as P

    dev = torch.device(device)
    sync = (lambda: torch.cuda.synchronize(dev)) if dev.type == "cuda" else None
    out = {}
    R, eps, x0 = R.to(dev), eps.to(dev), x0.to(dev)

    def leg(name, fn, rows, secs, unit, what):
        try:
            reps, dt = _timed_reps(fn, secs, sync=sync)
            out[name] = {"value": rows * reps / dt, "unit": unit, "rows_per_call": rows, "calls": reps, "seconds": round(dt, 2), "what": what}
        except Exception as e:  # recorded, not hidden (e.g. a batched LAPACK routine missing on the device)
            out[name] = {"error": repr(e)[:200]}

    leg("score", lambda: P.score_via_autograd(R, eps), R.shape[0], seconds[0], "evals/s",
        "closed-form fp64 log_prob + autograd score, per-row eps (oracle/ref_port.py after distributions.py:53-77,186-190)")
    proc = P.SO3DiffusionPort(lambda x, t: torch.zeros(x.shape[0], 3, device=dev), device=dev)
    B = x0.shape[0]
    g = torch.Generator().manual_seed(SEED)
    t_rows = torch.randint(0, 1000, (B,), generator=g).to(dev)
    t_shared = torch.full((B,), 500, dtype=torch.long, device=dev)
    with torch.no_grad():
        leg("q_sample", lambda: proc.q_sample(x0, t_rows), B, seconds[1], "rotations/s",
            "SO3Diffusion.q_sample, per-row t: (1000,B) fp64 table + compare-and-sum search + matrix_exp/SVD (diffusion.py:339-346)")
        leg("p_sample", lambda: proc.p_sample(x0, t_shared), B, seconds[2], "particle-steps/s",
            "SO3Diffusion.p_sample, zero denoiser, shared t = 500 (diffusion.py:315-326)")
    return out


def cpu_baseline(R, eps):
    """The reference's CPU path (torch port, all host threads) on a bounded sample of the bench's OWN inputs."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n = min(CPU_SAMPLE_ROWS, R.shape[0])
    Rc, ec = R[:n].cpu(), eps[:n].cpu()
    legs = reference_legs(Rc, ec, Rc[:SAMPLER_B], "cpu")
    s = legs["score"]
    return {"value": s.get("value"), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{s.get('calls')} x the first 2^{int(math.log2(n))} rows of the timed inputs, per-row eps, reference closed-form fp64 log_prob + autograd score "
                      f"(oracle/ref_port.py), {s.get('seconds')} s",
            "also": {k: legs[k] for k in ("q_sample", "p_sample")}}


def accuracy_of_timed_results(R, eps, logp, score, rows=1 << 16):
    """Max relative error of the results the timed launches left in `logp` / `score`, against the fp64 oracle series
    (SURVEY A.1) on a strided sample of the timed inputs.  The oracle is the checker here, nothing else."""
    from oracle import so3_oracle as O

    n = R.shape[0]
    idx = torch.arange(0, n, max(1, n // rows), device=R.device)[:rows]
    Rs = R[idx].cpu().numpy().astype(np.float64)
    es = eps[idx].cpu().numpy().astype(np.float64)
    lp = logp[idx].cpu().numpy().astype(np.float64)
    sc = score[idx].cpu().numpy().astype(np.float64)
    axis, ang = O.rmat_to_aa(Rs)
    om = ang[:, 0]
    ft, gt = O.igso3_series(om, es)
    far = (es < 0.4) & (om > 3.0 * es)   # far tail at small eps: the fp64 series itself cancels, the closed form is exact to 1e-9 there
    ft = np.where(far, O.igso3_closed(om, es), ft)
    gt = np.where(far, O.igso3_closed_dlog(om, es), gt)
    ef = np.abs(np.exp(lp - np.log(ft)) - 1)
    g = (sc * axis).sum(-1)
    ok = om > 1e-4
    eg = np.abs(g - gt) / np.maximum(np.abs(gt), 1e-30)
    es3 = np.linalg.norm(sc - gt[:, None] * axis, axis=-1) / np.maximum(np.abs(gt), 1e-30)
    k = om / (math.sqrt(2.0) * es)
    return {"rows": int(len(idx)), "max_rel_err_f": float(ef.max()), "max_rel_err_score": float(eg[ok].max()),
            "max_rel_err_score_vector": float(es3[om > 1e-2].max()), "tolerance": 1e-5, "k_max": float(k.max()),
            "rows_replaced_by_closed_form_frac": float(((om > 4.2 * es) & (es <= 1.0)).mean()),
            "against": "oracle/so3_oracle.py igso3_series (fp64, L = 2000) at the angle of the float32 matrix the kernel saw; score: d log f/d omega "
                       "(omega > 1e-4) and the 3-vector (omega > 1e-2: the axis of a rotation by omega is defined to ~6e-8/omega in fp32)"}


def dump_outputs(out_dir, arrays):
    """Write each row-major array of `arrays` (name -> tensor, rows first) as out_dir/<name>.npy.  Above DUMP_ROWS rows
    the same rows of every array are kept, chosen by a seeded permutation: the same rows for every run with the same --n."""
    n = next(iter(arrays.values())).shape[0]
    idx = None
    if n > DUMP_ROWS:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(SEED))[:DUMP_ROWS].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach()
        if idx is not None:
            a = a[idx.to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_port as P

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n = CPU_SAMPLE_ROWS
    R, eps = make_eset_cpu(n, SEED)
    for _ in range(args.warmup):
        P.score_via_autograd(R, eps)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        logp, logp_grad = P.score_via_autograd(R, eps)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logp": logp, "logp_grad": logp_grad})
    val = n * args.steps / dt
    sample = "each step = 2^18 rotations (bounded sample of the 2^24-row step), E-set law, per-row eps, reference closed-form fp64 log_prob + autograd score"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": "igso3_logp_score E-set, CPU reference port", "rows_per_step": n, "series_terms": None,
                                         "evaluator": "closed form fp64 (the reference has no series)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_RESULT_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on
    stdout when NCCL_DEBUG is set on the box), so file descriptor 1 is pointed at stderr for the whole run and the
    result line goes to a saved copy of the original stdout."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def hbm_roof(rows_per_s_per_gpu, bytes_per_row, pk):
    gbs = rows_per_s_per_gpu * bytes_per_row / 1e9
    return {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "bytes_per_row": bytes_per_row}


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=1 << 24, help="rotations per GPU per step")
    ap.add_argument("--L", type=int, default=2000, help="series truncation")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary kernels")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (profiling runs)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the 2^20..2^28 size sweep of cfg 2")
    ap.add_argument("--no-eager", action="store_true", help="skip the stock-PyTorch-on-the-same-GPU legs")
    ap.add_argument("--no-accuracy", action="store_true", help="skip the fp64-oracle check of the timed results (profiling runs)")
    ap.add_argument("--no-numa-bind", action="store_true", help="multi-GPU runs: leave the ranks' CPU affinity alone (A/B of the e2e leg)")
    ap.add_argument("--e2e-chunk", type=int, default=1 << 21, help="rows per chunk of the host-buffer pipeline")
    ap.add_argument("--sweep-max-log2", type=int, default=28, help="largest size of the cfg 2 sweep (2^k rotations)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        return run_reference(args)

    import diffusion_extensions_b200 as dx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()          # before anything is launched: the first sample needs ~0.3 s to appear
    numa = None
    if dist_on and not args.no_numa_bind:
        # one process per GPU: keep it (and the pinned staging buffers it is about to allocate) on the GPU's NUMA node
        numa = dx.parallel.bind_to_gpu_numa_node(local)
    if dist_on:
        torch.distributed.init_process_group("nccl", device_id=device)
    dx._lib.load()
    n, L = args.n, args.L
    pk = peaks()
    windows = []

    # ---- inputs: this rank's shard of the global batch (rows are independent: no exchange) -----
    R, eps = make_eset(n, device, SEED + rank)
    logp = torch.empty(n, device=device)
    score = torch.empty(n, 3, device=device)
    lib_call, ptr = dx._lib.call, dx._lib.ptr

    def step_series():
        lib_call("so3d_igso3_logp_score_f32", ptr(R), ptr(eps), 1, ptr(logp), ptr(score), None, n, dx._lib.MODE_SERIES, L, device=device)

    t_all0 = time.time()
    for _ in range(args.warmup):
        step_series()
    torch.cuda.synchronize()
    if sampler:
        sampler.wait_first()
    t_w0 = time.time()
    ms = time_loop(step_series, args.steps, 0, dist_on)
    windows.append(("headline timed region", t_w0, time.time()))
    evals_per_s = world * n * args.steps / (ms * 1e-3)
    per_gpu = evals_per_s / world
    # measured error of exactly these results (rank 0; CPU work, outside every timed region)
    accuracy = accuracy_of_timed_results(R, eps, logp, score) if (rank == 0 and not args.no_accuracy) else None
    if rank == 0 and args.dump_outputs:   # now: the legs below reuse logp / score
        dump_outputs(args.dump_outputs, {"logp": logp, "score": score})

    # ---- e2e: public host-buffer API, pinned host inputs -> host results -------------------------
    # dx.ops.HostScorePipeline is the call a user with host-resident batches makes: it overlaps the H2D copy,
    # the kernel and the D2H copy chunk by chunk.  Staging buffers are allocated once outside the timed
    # region; every timed step moves all n x 40 B in and n x 16 B out across PCIe.
    n_e2e = n
    e2e = None
    if not args.no_e2e:
        hR = torch.empty(n_e2e, 3, 3, pin_memory=True).copy_(R[:n_e2e].cpu())
        heps = torch.empty(n_e2e, pin_memory=True).copy_(eps[:n_e2e].cpu())
        hlogp = torch.empty(n_e2e, pin_memory=True)
        hscore = torch.empty(n_e2e, 3, pin_memory=True)
        pipe = dx.ops.HostScorePipeline(device, chunk_rows=args.e2e_chunk, depth=3)

        # a stream of batches: every step moves its own 40 B/row in and 16 B/row out; the pipeline is joined to the
        # timing stream once, after the last step (the next batch's uploads overlap the previous batch's drain)
        e2e_steps = args.steps
        count = {"k": 0}

        def step_e2e():
            count["k"] += 1
            pipe.run(hR, heps, hlogp, hscore, mode="series", L=L, wait=False, join=False)
            if count["k"] in (2, 2 + e2e_steps):      # last warm-up step / last timed step: join before the event is recorded
                pipe.finish()

        ms_e2e = time_loop(step_e2e, e2e_steps, 2, dist_on)
        windows.append(("headline + e2e timed regions", windows[0][1], time.time()))
        # the results really are on the host: spot-check them against the device-resident run
        torch.cuda.synchronize()
        assert torch.equal(hlogp[:4096], logp[:4096].cpu()) and torch.equal(hscore[-4096:], score[-4096:].cpu())
        # what bounds this leg: the pinned H2D copy of the step's inputs alone (and with the D2H of the results running
        # the other way at the same time), measured live on this box with the same buffers, ALL ranks copying at once
        # (time_loop's barrier aligns them and takes the max over ranks): the aggregate figure is the box's ceiling
        dR = torch.empty_like(R[:n_e2e])
        s_up, s_down = torch.cuda.Stream(), torch.cuda.Stream()

        def copy_up():
            dR.copy_(hR, non_blocking=True)
            eps.copy_(heps, non_blocking=True)

        def copy_duplex():
            with torch.cuda.stream(s_up):
                copy_up()
            with torch.cuda.stream(s_down):
                hlogp.copy_(logp, non_blocking=True)
                hscore.copy_(score, non_blocking=True)
            torch.cuda.current_stream().wait_stream(s_up)
            torch.cuda.current_stream().wait_stream(s_down)

        ms_up = time_loop(copy_up, 3, 1, dist_on) / 3
        ms_duplex = time_loop(copy_duplex, 3, 1, dist_on) / 3
        del dR
        step_ms = ms_e2e / e2e_steps
        pcie = {"h2d_alone_gbs": n_e2e * 40 / (ms_up * 1e-3) / 1e9, "h2d_alone_ms": ms_up, "duplex_ms": ms_duplex,
                "aggregate_h2d_alone_gbs": world * n_e2e * 40 / (ms_up * 1e-3) / 1e9,
                "aggregate_duplex_gbs": {"h2d": world * n_e2e * 40 / (ms_duplex * 1e-3) / 1e9, "d2h": world * n_e2e * 16 / (ms_duplex * 1e-3) / 1e9},
                "frac_of_duplex_copy_floor": ms_duplex / step_ms,
                "floor_evals_per_s": world * n_e2e / (max(ms_duplex, ms / args.steps) * 1e-3),
                "note": "floor of a step = max(kernel, duplex copy of the same pinned buffers with all ranks copying at once, max over ranks); "
                        "the copies are PCIe / host-memory bound, the kernel is not"}
        e2e = {"value": world * n_e2e * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT, "pcie_floor": pcie, "h2d_bytes_per_step": n_e2e * 40, "d2h_bytes_per_step": n_e2e * 16,
               "steps": e2e_steps, "ms_per_step": step_ms,
               "api": "ops.HostScorePipeline.run(join=False) x steps + finish() (3-stream chunked overlap, batches streamed back to back)", "chunk_rows": args.e2e_chunk, "numa_bind_rank0": numa,
               "launches": pipe.launches,
               "pcie_gbs": {"h2d": n_e2e * 40 / (step_ms * 1e-3) / 1e9, "d2h": n_e2e * 16 / (step_ms * 1e-3) / 1e9}}
        del hR, heps, hlogp, hscore, pipe

    # ---- secondary kernels ----------------------------------------------------------------------
    extra = {}
    if not args.no_extra:
        def rate(fn, rows, reps=5):
            m = time_loop(fn, reps, 3, dist_on)
            return world * rows * reps / (m * 1e-3), m / reps

        for mode_name, mode in (("auto", dx._lib.MODE_AUTO), ("series_adaptive", dx._lib.MODE_SERIES_ADAPTIVE), ("series_pure", dx._lib.MODE_SERIES_PURE)):
            v, m = rate(lambda: lib_call("so3d_igso3_logp_score_f32", ptr(R), ptr(eps), 1, ptr(logp), ptr(score), None, n, mode, L, device=device), n)
            extra[f"score_evals_per_sec_{mode_name}"] = {"value": v, "ms_per_step": m}
            if mode_name == "auto":
                extra[f"score_evals_per_sec_{mode_name}"]["roofline"] = hbm_roof(v / world, BYTES_PER_EVAL, pk)
        # small batches of the same evaluator (north_star: "warp-shuffle reductions for the per-omega series partial sums"):
        # below ~96 rows per SM the library runs ONE WARP per rotation, the 2000 terms split over the lanes
        if rank == 0:
            sb = {}
            for nb in (256, 4096, 9472, 16384):
                ms_b = time_loop(lambda: lib_call("so3d_igso3_logp_score_f32", ptr(R), ptr(eps), 1, ptr(logp), ptr(score), None, nb, dx._lib.MODE_SERIES, L,
                                                  device=device), 50, 5, False) / 50
                sb[str(nb)] = {"us_per_call": ms_b * 1e3, "evals_per_s": nb / (ms_b * 1e-3)}
            extra["series_small_batch"] = {"rows": sb, "note": "back-to-back launches through the Python binding, device-timed (~13 us of host launch overhead per call "
                                                               "bounds the small sizes; kernel durations are in profiles/*_launches.md); <= 9472 rows (64 per SM): one warp per "
                                                               "rotation (series_warp_kernel), above: one thread per rotation (16384 shown for contrast)"}
        if dist_on:
            torch.distributed.barrier()
        proc = dx.SO3Diffusion(None).to(device)
        proc.row_offset = rank * n
        fwd, post, t_range = proc.tables()
        fwd_guide, post_guide = proc.guides()
        loc_tab = dx.ops.cdf_grid(device)[2]
        pred = torch.zeros(n, 3, device=device)
        xa, xb = R.clone(), torch.empty_like(R)
        t_step = t_range[500:501]
        state = {"off": 0}

        def step_rev():
            state["off"] += 1
            lib_call("so3d_p_sample_f32", ptr(xa), ptr(pred), ptr(t_step), 0, ptr(proc.sqrt_recip_alphas_cumprod), ptr(proc.sqrt_recipm1_alphas_cumprod),
                     ptr(proc.posterior_mean_coef1), ptr(proc.posterior_mean_coef2), 1000, ptr(post), None, ptr(loc_tab), SEED, state["off"],
                     rank * n, ptr(xb), None, n, device=device)

        v, m = rate(step_rev, n, 10)
        extra["reverse_particle_steps_per_sec"] = {"value": v, "ms_per_step": m, "note": "fused p_sample kernel, pred = 0 (denoiser excluded), shared t = 500",
                                                   "roofline": hbm_roof(v / world, BYTES_PER_PARTICLE_STEP, pk)}
        tt = torch.randint(0, 1000, (n,), device=device)
        tgt = torch.empty(n, 3, device=device)

        def step_fwd():
            state["off"] += 1
            lib_call("so3d_q_sample_f32", ptr(xa), ptr(tt), ptr(proc.sqrt_alphas_cumprod), ptr(proc.sqrt_one_minus_alphas_cumprod), 1000, ptr(fwd),
                     ptr(fwd_guide), ptr(loc_tab), SEED, state["off"], rank * n, ptr(xb), ptr(tgt), None, None, n, device=device)

        v, m = rate(step_fwd, n, 10)
        extra["noised_rotations_per_sec"] = {"value": v, "ms_per_step": m, "note": "fused q_sample + skewvec target, per-row t",
                                             "roofline": hbm_roof(v / world, BYTES_PER_QSAMPLE, pk)}

        # north_star's "fused IGSO(3) score + noising": the same launch also evaluates the score of the drawn noise
        # (d log f / d omega along the axis, closed form / series by eps): 36 + 8 B in, 36 + 12 + 12 B out per rotation
        scr = torch.empty(n, 3, device=device)

        def step_fwd_score():
            state["off"] += 1
            lib_call("so3d_q_sample_f32", ptr(xa), ptr(tt), ptr(proc.sqrt_alphas_cumprod), ptr(proc.sqrt_one_minus_alphas_cumprod), 1000, ptr(fwd),
                     ptr(fwd_guide), ptr(loc_tab), SEED, state["off"], rank * n, ptr(xb), ptr(tgt), None, ptr(scr), n, device=device)

        v, m = rate(step_fwd_score, n, 10)
        extra["noised_rotations_with_score_per_sec"] = {"value": v, "ms_per_step": m, "note": "fused q_sample + skewvec target + IGSO(3) score of the noise, per-row t",
                                                        "roofline": hbm_roof(v / world, BYTES_PER_QSAMPLE + 12, pk)}
        del scr

        # BASELINE configs[2]: the whole reverse process, 1000 fused steps over this GPU's share of 2^24 particles
        # (pred = 0: the denoiser is excluded, SURVEY 8d).  Two routes: one launch per step from the host (x ping-pongs
        # between two buffers), and so3d_p_sample_loop_f32 -- ALL steps in one launch, particles resident in shared memory.
        n_loop = max(1, (1 << 24) // world)
        la, lb = R[:n_loop].clone(), torch.empty_like(R[:n_loop])
        pz = pred[:n_loop]

        def reverse_loop():
            a, b = la, lb
            for i in reversed(range(1000)):
                lib_call("so3d_p_sample_f32", ptr(a), ptr(pz), ptr(t_range[i:i + 1]), 0, ptr(proc.sqrt_recip_alphas_cumprod),
                         ptr(proc.sqrt_recipm1_alphas_cumprod), ptr(proc.posterior_mean_coef1), ptr(proc.posterior_mean_coef2), 1000, ptr(post),
                         None, ptr(loc_tab), SEED, 1000 + i, rank * n_loop, ptr(b), None, n_loop, device=device)
                a, b = b, a

        m = time_loop(reverse_loop, 1, 1, dist_on)
        v = world * n_loop * 1000 / (m * 1e-3)
        loop_entry = {"value": v, "unit": "particle-steps/s", "seconds": m * 1e-3, "particles": world * n_loop, "steps": 1000,
                      "note": "BASELINE configs[2]: 1000 fused reverse steps x 2^24 particles (split over the GPUs), pred = 0, one launch per step",
                      "roofline": hbm_roof(v / world, BYTES_PER_PARTICLE_STEP, pk)}
        if hasattr(dx.ops, "p_sample_loop_fused"):
            try:
                def one_launch():
                    dx.ops.p_sample_loop_fused(la, None, 999, 0, proc.sqrt_recip_alphas_cumprod, proc.sqrt_recipm1_alphas_cumprod, proc.posterior_mean_coef1,
                                               proc.posterior_mean_coef2, post, post_guide, seed=SEED, rng_offset=1000, row_offset=rank * n_loop, out=lb)

                m1 = time_loop(one_launch, 1, 1, dist_on)
                v1 = world * n_loop * 1000 / (m1 * 1e-3)
                sm_n = torch.cuda.get_device_properties(device).multi_processor_count
                loop_entry["one_launch"] = {"value": v1, "unit": "particle-steps/s", "seconds": m1 * 1e-3,
                                            "note": "so3d_p_sample_loop_f32: ONE launch for all 1000 steps -- a CTA keeps its chunk of particles resident in shared memory "
                                                    "(x_T read from HBM once, x_0 written once), per step and particle one 16-byte guide record comes from the L2-resident "
                                                    "posterior table; bit-identical to the per-step launches; no HBM traffic to speak of, bound by instruction issue",
                                            "equivalent_hbm_gbs_per_gpu": v1 / world * BYTES_PER_PARTICLE_STEP / 1e9,
                                            "thread_instr_budget_per_particle_step": sm_n * 128 * pk["sm_max_mhz"] * 1e6 / (v1 / world)}
            except Exception as e:
                loop_entry["one_launch"] = {"error": repr(e)[:300]}
        extra["reverse_loop_1000_steps"] = loop_entry
        del la, lb

        # SURVEY 8(f4): one reverse step WITH the reference's RotPredict denoiser (so3_train.py:11-49) inside the kernel
        # (tcgen05 tf32 3-term split), against the two-kernel route (stock PyTorch MLP + fused step).
        torch.manual_seed(SEED)
        net = dx.RotPredict(out_type="skewvec").to(device)
        procn = dx.SO3Diffusion(net).to(device)
        procn.row_offset = rank * n
        procn.tables()
        with torch.no_grad():
            vd, md = rate(lambda: procn.p_sample(xa, t_step), n, 5)
            procn.fuse_denoiser = False
            nu = min(n, 1 << 22)  # the stock route materialises (n, 65) activations: bounded
            vu, mu = rate(lambda: procn.p_sample(xa[:nu], t_step), nu, 3)
        flop_ps = 2 * 65 * (65 * 4 + 3)                       # algorithmic MLP flops per particle-step (fp32 semantics)
        extra["reverse_with_denoiser_particle_steps_per_sec"] = {
            "value": vd, "ms_per_step": md, "note": "RotPredict (65-wide, 5 layers) + reverse step in ONE tcgen05 kernel, shared t = 500",
            "stock_mlp_plus_fused_step": {"value": vu, "ms_per_step": mu, "rows": nu},
            "mlp_tflops_algorithmic": vd / world * flop_ps * 1e-12}
        del net, procn

        # BASELINE configs[4] (prot_train.py on synthetic frames): per-residue SE(3) noising and reverse step on
        # (B, N_res = 256) frame batches -- rot (B,256,3,3) + shift (B,256,3), one step index per complex (B,)
        # broadcast over its residues (diffusion.py:432-522); both halves of every step in one launch.
        try:
            nres = 256
            bsz = max(1, n // nres)
            rows5 = bsz * nres
            se3 = dx.SE3Diffusion(None).to(device)
            se3.row_offset = rank * rows5
            f5, p5, _ = se3.tables()
            g5f, g5p = se3.guides()
            rot0 = R[:rows5].reshape(bsz, nres, 3, 3)
            shift0 = torch.randn(bsz, nres, 3, device=device) * 10.0
            t5 = dx.ops._rows_t(torch.randint(0, 1000, (bsz,), device=device), (bsz, nres), device)   # (B,) broadcast over N_res
            rot_t, shift_t = torch.empty_like(rot0), torch.empty_like(shift0)
            tr5, ts5, so5 = torch.empty_like(shift0), torch.empty_like(shift0), torch.empty_like(shift0)
            sig5 = se3._sigma()

            def step_se3_q():
                state["off"] += 1
                lib_call("so3d_se3_q_sample_f32", ptr(rot0), ptr(shift0), ptr(t5), ptr(se3.sqrt_alphas_cumprod), ptr(se3.sqrt_one_minus_alphas_cumprod), 1000,
                         ptr(f5), ptr(g5f), ptr(loc_tab), float(se3.shift_scale), SEED, state["off"], rank * rows5, ptr(rot_t), ptr(shift_t), ptr(tr5), ptr(ts5),
                         rows5, device=device)

            vq, mq = rate(step_se3_q, rows5, 10)

            def step_se3_p():
                state["off"] += 1
                lib_call("so3d_se3_p_sample_f32", ptr(rot_t), ptr(shift_t), ptr(tr5), ptr(ts5), ptr(t_step), 0, ptr(se3.sqrt_recip_alphas_cumprod),
                         ptr(se3.sqrt_recipm1_alphas_cumprod), ptr(se3.posterior_mean_coef1), ptr(se3.posterior_mean_coef2), ptr(sig5), 1000, ptr(p5), ptr(g5p),
                         ptr(loc_tab), float(se3.shift_scale), SEED, state["off"], rank * rows5, ptr(xb), ptr(so5), rows5, device=device)

            vp, mp = rate(step_se3_p, rows5, 10)
            extra["se3_frames_cfg5"] = {
                "shape": [bsz, nres], "frames_per_gpu": rows5,
                "noising_frames_per_sec": {"value": vq, "ms_per_step": mq, "roofline": hbm_roof(vq / world, BYTES_PER_SE3_QSAMPLE, pk)},
                "reverse_frame_steps_per_sec": {"value": vp, "ms_per_step": mp, "roofline": hbm_roof(vp / world, BYTES_PER_SE3_PSTEP, pk)},
                "note": "SE3Diffusion on (B, N_res=256) synthetic backbone frames: fused q_sample + both grad_mse targets (per-complex t broadcast over residues), "
                        "fused reverse step (shared t = 500, predictions = the targets)"}
            del rot_t, shift_t, tr5, ts5, so5, shift0, t5, se3
        except Exception as e:
            extra["se3_frames_cfg5"] = {"error": repr(e)[:300]}

        # BASELINE configs[3] (bingham_train.py under DDP): Bingham data (fused sampler, bingham_train.py:55,88-90) ->
        # SO3Diffusion('skewvec') + RotPredict + Adam, data-parallel over the ranks.
        try:
            extra["ddp_train_rows_per_sec"] = ddp_train_leg(dx, device, rank, world, dist_on)
        except Exception as e:
            extra["ddp_train_rows_per_sec"] = {"error": repr(e)[:300]}

        # the launch-bound ends of the same paths, as ONE CUDA graph each (device-resident Philox seed):
        # the reference's own sampling size (bingham_test.py:25: 20 000 particles x 1000 steps) and its toy training step
        # (so3_train.py:65-76: batch 256, RotPredict + Adam).  Wall clock, per call, on this rank.
        if rank == 0:
            try:  # secondary, wall-clock legs built on graph capture: a failure here must not cost the headline line
                torch.manual_seed(SEED)
                gnet = dx.RotPredict(out_type="skewvec").to(device)
                gproc = dx.SO3Diffusion(gnet).to(device)
                loops = {}
                for mode, use_graph, one_launch in (("eager", False, False), ("cuda_graph", True, False), ("one_launch", True, True)):
                    gproc.fused_loop = one_launch
                    gproc.p_sample_loop((20000,), cuda_graph=use_graph)          # warm-up / capture
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(3):
                        gproc.p_sample_loop((20000,), cuda_graph=use_graph)
                    torch.cuda.synchronize()
                    loops[mode] = (time.perf_counter() - t0) / 3 * 1e3
                extra["reverse_loop_20000_particles_ms"] = {**loops, "unit": "ms per 1000-step loop (wall clock)",
                                                            "note": "RotPredict + reverse step fused: one launch per step from the host (eager), the same launches as one "
                                                                    "captured CUDA graph, and all 1000 steps inside ONE launch (so3d_rotpredict_p_sample_loop_f32)"}
                gopt = torch.optim.Adam(gnet.parameters(), lr=1e-3, capturable=True)
                xb256 = R[:256].contiguous()
                steps_ms = {}

                def eager_step():
                    gopt.zero_grad(set_to_none=True)
                    gproc(xb256).backward()
                    gopt.step()

                graphed = gproc.make_graphed_train_step(gopt, xb256, sync_grads=False)
                for name, fn in (("eager", eager_step), ("cuda_graph", lambda: graphed(xb256))):
                    for _ in range(10):
                        fn()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(200):
                        fn()
                    torch.cuda.synchronize()
                    steps_ms[name] = (time.perf_counter() - t0) / 200 * 1e3
                extra["train_step_batch256_ms"] = {**steps_ms, "unit": "ms per step (wall clock)",
                                                   "note": "SO3Diffusion('skewvec') + RotPredict + Adam; eager vs SO3Diffusion.make_graphed_train_step"}
                del gnet, gproc, gopt, graphed
            except Exception as e:  # recorded, not hidden
                extra["graph_legs_error"] = repr(e)[:300]
        if dist_on:
            torch.distributed.barrier()

        # SURVEY 8(f1): MMD two-sample statistic at bingham_test.py:29's size (20 000 vs 20 000 rotations), one fused
        # all-pairs launch; multi-GPU: tile pairs dealt over the ranks, three doubles all-reduced.
        nm = 20000
        mx, my = R[:nm].contiguous(), xb[:nm].contiguous()

        def step_mmd():
            sums = dx.ops.pair_kernel_sums(mx, my, "gaussian", shard=rank, nshards=world)
            if dist_on:
                torch.distributed.all_reduce(sums)

        mm = time_loop(step_mmd, 5, 3, dist_on) / 5
        pairs_logical = 3 * nm * nm                      # k(X,X), k(Y,Y), k(X,Y) as the reference evaluates them
        tiles = (nm + 255) // 256
        pairs_computed = (tiles * (tiles + 1) + tiles * tiles) * 65536   # lower-triangular tile pairs for the two self sums
        sm_ = torch.cuda.get_device_properties(device).multi_processor_count
        lane_peak = world * sm_ * 128 * pk["sm_max_mhz"] * 1e6
        extra["mmd_pairs_per_sec"] = {"value": pairs_logical / (mm * 1e-3), "unit": "kernel evaluations/s (as the reference counts them)", "ms_per_mmd": mm,
                                      "n": [nm, nm], "note": "util.MMD with rmat_gaussian_kernel, fused all-pairs kernel (bingham_test.py:29 size)",
                                      "roofline": {"bound": "fp32", "achieved": pairs_computed * MMD_LANE_INSTR_PER_PAIR / (mm * 1e-3) * 1e-12,
                                                   "peak": lane_peak * 1e-12, "unit": "T lane-instr/s",
                                                   "frac": pairs_computed * MMD_LANE_INSTR_PER_PAIR / (mm * 1e-3) / lane_peak}}
        del mx, my, xa, xb, pred, tt, tgt

        # the reference's op sequence as stock PyTorch eager on THIS GPU (SURVEY 2.2: "beat stock PyTorch eager running the
        # reference code on the same B200"); figures also go beside the kernels they match
        if rank == 0 and not args.no_eager:
            try:
                ne = min(n, 1 << 20)
                eager = reference_legs(R[:ne], eps[:ne], R[:SAMPLER_B], device, seconds=(2.0, 2.0, 2.0))
                eager["note"] = ("oracle/ref_port.py (the reference's op sequence: fp64 closed form + autograd, (1000,B) table rebuilt per call, matrix_exp, SVD, "
                                 "masked eigh) on cuda tensors, stock PyTorch eager, wall clock with synchronize; score on 2^20 rows, samplers at B = 65 536")
            except Exception as e:
                eager = {"error": repr(e)[:300]}
            extra["torch_cuda_eager"] = eager
            torch.cuda.empty_cache()
        if dist_on:
            torch.distributed.barrier()

    # ---- BASELINE configs[1] size sweep: 2^20 ... 2^28 rotations on ONE GPU (64-bit offsets above 2^27 rows) -----------
    if world == 1 and not args.no_sweep and not args.no_extra:
        try:
            extra["size_sweep"] = size_sweep(dx, device, R, eps, logp, score, L, pk, args.sweep_max_log2)
        except Exception as e:
            extra["size_sweep"] = {"error": repr(e)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        windows.append(("whole GPU part of the run", t_all0, time.time()))
        cpu = cpu_baseline(R, eps)
        for key, leg in (("reverse_particle_steps_per_sec", "p_sample"), ("noised_rotations_per_sec", "q_sample")):
            if key in extra:
                extra[key]["cpu_baseline"] = cpu["also"].get(leg)
    if rank == 0 and isinstance(extra.get("torch_cuda_eager"), dict):
        for key, leg in (("reverse_particle_steps_per_sec", "p_sample"), ("noised_rotations_per_sec", "q_sample"), ("score_evals_per_sec_auto", "score")):
            if key in extra and leg in extra["torch_cuda_eager"]:
                extra[key]["torch_cuda_eager"] = extra["torch_cuda_eager"][leg]

    if rank == 0:
        clocks = None
        if sampler:
            windows.append(("whole run", t_all0, time.time()))
            sampler.stop()
            clocks = sampler.summary(windows)
        sm = torch.cuda.get_device_properties(device).multi_processor_count
        ghz = pk["sm_max_mhz"] * 1e-3
        issue_peak = sm * 128 * ghz * 1e9                      # FP32 lane-instructions/s (= 4 warp-instr/clk/SM)
        mufu_peak = sm * 16 * ghz * 1e9
        fp32_peak_tflops = sm * 128 * 2 * ghz * 1e-3          # FFMA = 2 flop/lane/clk
        ach = per_gpu * L * ALGO_LANE_INSTR_PER_TERM
        # time per term implied by each resource for the executed mix, in SMSP clocks per warp-term:
        #   issue 9 slots; XU pipe 8 (MUFU at 4 lanes/clk/SMSP); FP32 operand reads 8.8 (measured per-form costs:
        #   1-register 1.0, 2-register 1.09, 3-register 1.5 clk, profiles/microbench/pipes.cu)
        clk_per_term = sm * 4 * ghz * 1e9 * 32 / (per_gpu * L)
        roofline = {
            "bound": "fp32", "achieved": ach * 1e-12, "peak": issue_peak * 1e-12, "unit": "T lane-instr/s", "frac": ach / issue_peak,
            "traffic": NCU_DRAM_BYTES_PER_EVAL * n, "traffic_source": "ncu --set full, profiles/r02p_series_full.md (bytes/eval x rows per launch)",
            "definition": "SURVEY 8(d): FP32-issue bound with 10 lane-instr/term (1.86e9 evals/s/GPU); executed mix below",
            "executed_per_term": {"fp32_instr": FP32_INSTR_PER_TERM, "mufu": MUFU_PER_TERM, "uniform_ldc": UNIFORM_PER_TERM, "flop": FLOP_PER_TERM},
            "clk_per_warp_term": clk_per_term, "clk_floor_issue": 9.0, "clk_floor_xu": 8.0, "clk_floor_fp32_operands": 8.8,
            "frac_of_executed_mix_floor": 9.0 / clk_per_term,
            "executed_tflops": per_gpu * L * FLOP_PER_TERM * 1e-12, "fp32_peak_tflops": fp32_peak_tflops,
            "mufu_frac": per_gpu * L * MUFU_PER_TERM / mufu_peak,
            "naive_3mufu_roofline_evals_per_s": mufu_peak / (3 * L), "frac_of_naive_3mufu_roofline": per_gpu / (mufu_peak / (3 * L)),
            "hbm_gbs": per_gpu * BYTES_PER_EVAL / 1e9,
            "peak_source": f"derived: {sm} SMs x 128 FP32 lanes x {pk['sm_max_mhz']:.0f} MHz ({pk['source']}); HBM {pk['hbm_gbs']} GB/s",
        }
        line = {
            "metric": METRIC, "value": evals_per_s, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "igso3_logp_score series L=2000, E-set (BASELINE configs[1])", "rows_per_gpu_per_step": n, "series_terms": L,
                       "eps": "per-row, log-uniform [6.4e-3,1]", "l2": "inputs (640 MiB/GPU) larger than L2", "parallelism": f"batch-sharded x{world}, no collective in the data path",
                       "series_guard": "every row runs all L terms; rows with omega > 4.2 eps (fp32 series cond > 14) are then replaced by the closed form "
                                       "(accuracy.rows_replaced_by_closed_form_frac)"},
            "roofline": roofline, "accuracy": accuracy, "e2e": e2e, "gpu_launches": args.steps, "clocks": clocks, "extra": extra,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        emit(line)
    if dist_on:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def size_sweep(dx, device, R, eps, logp, score, L, pk, max_log2):
    """evals/s of the series and the auto evaluator at n = 2^20 ... 2^28 rotations (BASELINE configs[1]); at 2^28 the row
    arrays are 9.7 GB in + 4.3 GB out and element offsets exceed 2^31, so a strided sample of the big run (reaching the
    last rows) is compared with the results of the same rows evaluated in a small launch."""
    lib_call, ptr = dx._lib.call, dx._lib.ptr
    out = {"unit": UNIT, "sizes": {}}
    n0 = R.shape[0]
    big = None
    for k in (20, 22, 24, 26, 28):
        if k > max_log2:
            break
        nk = 1 << k
        if nk <= n0:
            Rk, ek, lk, sk = R[:nk], eps[:nk], logp[:nk], score[:nk]
        else:
            big = None
            torch.cuda.empty_cache()
            Rb, eb = make_eset(nk, device, SEED + 77)
            big = (Rb, eb, torch.empty(nk, device=device), torch.empty(nk, 3, device=device))
            Rk, ek, lk, sk = big
        entry = {}
        for name, mode, reps in (("series", dx._lib.MODE_SERIES, 3), ("auto", dx._lib.MODE_AUTO, 5)):
            fn = lambda: lib_call("so3d_igso3_logp_score_f32", ptr(Rk), ptr(ek), 1, ptr(lk), ptr(sk), None, nk, mode, L, device=device)
            ms = time_loop(fn, reps, 2, False) / reps
            entry[name] = {"evals_per_s": nk / (ms * 1e-3), "ms": ms}
        entry["auto"]["hbm_frac"] = entry["auto"]["evals_per_s"] * BYTES_PER_EVAL / 1e9 / pk["hbm_gbs"]
        if nk > n0:   # the last launch was `auto`: compare a strided sample (reaching the last rows) with a small launch of the same rows
            idx = torch.cat([torch.arange(0, nk, nk // 4096, device=device), torch.arange(nk - 4096, nk, device=device)])
            Rs, es = Rk[idx].contiguous(), ek[idx].contiguous()
            ls, ss = torch.empty(idx.numel(), device=device), torch.empty(idx.numel(), 3, device=device)
            lib_call("so3d_igso3_logp_score_f32", ptr(Rs), ptr(es), 1, ptr(ls), ptr(ss), None, idx.numel(), dx._lib.MODE_AUTO, L, device=device)
            entry["sample_bit_identical_to_small_launch"] = bool(torch.equal(ls, lk[idx]) and torch.equal(ss, sk[idx]))
        out["sizes"][f"2^{k}"] = entry
    del big
    torch.cuda.empty_cache()
    return out


def ddp_train_leg(dx, device, rank, world, dist_on):
    """cfg 4: rows/s of data-parallel training on Bingham targets.  Three routes per batch size:
      ddp_eager      stock DistributedDataParallel around RotPredict + parallel.train_step_sharded (fused noising launch,
                     DDP's bucketed all-reduce, one 2-float loss all-reduce);
      no_sync        the same step with the gradient all-reduce and the loss all-reduce switched off -> their time share;
      cuda_graph     SO3Diffusion.make_graphed_train_step with the gradient bucket all-reduced INSIDE the captured graph."""
    import torch.distributed as dist

    cov1 = torch.diag(torch.tensor([1000.0, 0.1, 0.1, 0.1], device=device))      # bingham_train.py:55 "small uncorrelated rotations"
    data = dx.Bingham(torch.zeros(4, device=device), covariance_matrix=cov1)
    out = {"unit": "training rows/s (all ranks)", "data": "Bingham(cov1) -> rotation matrices, fused sampler (so3d_bingham_sample_f32), fresh batch every step",
           "model": "RotPredict(d_model=65, out_type='skewvec'), Adam lr 3e-4 (bingham_train.py:84-95)", "batches": {}}
    for bsz in (256, 1 << 16):
        entry = {}
        torch.manual_seed(SEED)                                                   # identical initial weights on every rank
        net = dx.RotPredict(out_type="skewvec").to(device)
        proc = dx.SO3Diffusion(net).to(device)
        proc.tables()
        data.row_offset = rank * bsz
        ddp = dx.parallel.wrap_denoiser(net, device)
        proc.denoise_fn = ddp
        opt = torch.optim.Adam(ddp.parameters(), lr=3e-4)

        def step_ddp():
            return dx.parallel.train_step_sharded(proc, data.sample_rmat((bsz,)), opt)

        def step_nosync():
            x0 = data.sample_rmat((bsz,))
            opt.zero_grad(set_to_none=True)
            t = torch.randint(0, 1000, (bsz,), device=device)
            fused = proc.noise_and_target(x0, t)
            if dist_on:
                with ddp.no_sync():
                    ((ddp(fused["x_t"], t) - fused["target"]) ** 2).mean().backward()
            else:
                ((ddp(fused["x_t"], t) - fused["target"]) ** 2).mean().backward()
            opt.step()

        reps = 50 if bsz <= 4096 else 10
        ms = time_loop(step_ddp, reps, 5, dist_on) / reps
        ms0 = time_loop(step_nosync, reps, 5, dist_on) / reps
        entry["ddp_eager"] = {"value": world * bsz / (ms * 1e-3), "ms_per_step": ms}
        entry["no_sync"] = {"value": world * bsz / (ms0 * 1e-3), "ms_per_step": ms0}
        entry["allreduce_time_share"] = max(0.0, 1.0 - ms0 / ms)
        # graph-captured data-parallel step: bare module, gradient bucket all-reduced by a captured NCCL launch
        try:
            torch.manual_seed(SEED)
            gnet = dx.RotPredict(out_type="skewvec").to(device)
            gproc = dx.SO3Diffusion(gnet).to(device)
            gproc.row_offset = rank * bsz
            gopt = torch.optim.Adam(gnet.parameters(), lr=3e-4, capturable=True)
            step = gproc.make_graphed_train_step(gopt, data.sample_rmat((bsz,)))

            def step_graph():
                step(data.sample_rmat((bsz,)))

            msg = time_loop(step_graph, reps, 5, dist_on) / reps
            entry["cuda_graph"] = {"value": world * bsz / (msg * 1e-3), "ms_per_step": msg, "grad_allreduce_in_graph": bool(step.sync_grads)}
            if dist_on:  # the ranks' weights must still agree after the captured all-reduces
                w = torch.cat([p.detach().flatten() for p in gnet.parameters()])
                w0 = w.clone()
                dist.broadcast(w0, 0)
                entry["cuda_graph"]["weights_in_sync"] = bool(torch.equal(w, w0))
            del gnet, gproc, gopt, step
        except Exception as e:
            entry["cuda_graph"] = {"error": repr(e)[:300]}
        out["batches"][str(bsz)] = entry
        del net, proc, ddp, opt
    vals = [e[k]["value"] for e in out["batches"].values() for k in ("ddp_eager", "cuda_graph") if isinstance(e.get(k), dict) and "value" in e[k]]
    out["value"] = max(vals) if vals else None
    return out


if __name__ == "__main__":
    main()
