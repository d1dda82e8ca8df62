"""bench.py's contract with the driver, as far as it can be checked without a GPU: the reference arm prints exactly ONE
JSON line on stdout (everything else goes to stderr) with the keys the driver reads, times the oracle port on the host
cores, and exits 0; ranks other than 0 of a multi-rank reference run print nothing."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMP_LIMIT = 64 << 20   # bytes --dump-outputs may write in all


def run_reference(extra_env=None, extra_args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "3",
                           *extra_args], capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)


def load_dump(d):
    out = {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
    assert all(f.endswith(".npy") for f in os.listdir(d))
    assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= DUMP_LIMIT
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    return out


def test_reference_arm_prints_one_json_line():
    p = run_reference()
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "igso3_score_evals_per_sec" and d["unit"] == "evals/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] >= 3 and d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent():
    p = run_reference({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_our_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: on a box without CUDA the product arm must not print a result line."""
    import torch

    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--no-extra", "--no-cpu", "--no-e2e"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert p.returncode != 0 and p.stdout.strip() == ""


def test_steps_below_one_is_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert p.returncode != 0 and p.stdout.strip() == "" and "--steps" in p.stderr


def test_reference_arm_dumps_its_last_step(tmp_path):
    import torch

    import bench
    from oracle import ref_port as P

    p = run_reference(extra_args=("--dump-outputs", str(tmp_path)))
    assert p.returncode == 0, p.stderr[-2000:]
    n = json.loads(p.stdout)["config"]["rows_per_step"]
    got = load_dump(tmp_path)
    assert set(got) == {"logp", "logp_grad"}
    R, eps = bench.make_eset_cpu(n, bench.SEED)
    lp, g = P.score_via_autograd(R, eps)
    assert got["logp"].shape == tuple(lp.shape) and got["logp_grad"].shape == (n, 3, 3)
    # the reference's closed form is NaN on ~12 % of the E-set (its own quirks): those rows must be NaN in the dump too
    assert torch.allclose(torch.from_numpy(got["logp"]), lp, rtol=1e-6, atol=0, equal_nan=True)
    assert torch.allclose(torch.from_numpy(got["logp_grad"]), g, rtol=1e-5, atol=1e-5 * float(g.nan_to_num().abs().max()), equal_nan=True)


@pytest.mark.gpu
def test_dump_is_a_seeded_sample_of_the_timed_results(cuda_device, tmp_path):
    """Above DUMP_ROWS rows --dump-outputs keeps the rows of a permutation seeded with SEED, of inputs that are the same
    on every run; what it writes equals a fresh evaluation of those inputs."""
    import torch

    import bench
    import diffusion_extensions_b200 as dx

    n = bench.DUMP_ROWS + 4099
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--steps", "2", "--no-extra", "--no-cpu", "--no-e2e",
                        "--no-accuracy", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout)
    assert d["steps"] == 2 and d["gpu_launches"] == 2
    got = load_dump(tmp_path)
    assert set(got) == {"logp", "score"}
    R, eps = bench.make_eset(n, cuda_device, bench.SEED)
    logp, score = torch.empty(n, device=cuda_device), torch.empty(n, 3, device=cuda_device)
    ptr = dx._lib.ptr
    dx._lib.call("so3d_igso3_logp_score_f32", ptr(R), ptr(eps), 1, ptr(logp), ptr(score), None, n, dx._lib.MODE_SERIES, d["config"]["series_terms"],
                 device=cuda_device)
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(bench.SEED))[:bench.DUMP_ROWS].sort().values
    assert np.array_equal(got["logp"], logp.cpu()[idx].numpy()) and np.array_equal(got["score"], score.cpu()[idx].numpy())
