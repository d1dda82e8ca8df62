"""GPU tests of the capturable SE(3) arm: the device-seed SE(3) kernels (so3d_se3_q_sample_dseed_f32,
so3d_se3_p_sample_dseed_f32) against their by-value counterparts, and SE3Diffusion / ProjectedSE3Diffusion training steps
and sampling loops captured in CUDA graphs.  Every comparison with the by-value kernels is bit for bit: the device-seed
kernels draw from the same two Philox streams (rotation at (row, rng_offset), translation at (row, rng_offset | 2^63))."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASK64 = 0xFFFFFFFFFFFFFFFF
SEEDS = (0x1234_5678_9ABC_DEF0, 0xF00D_CAFE_0BAD_BEEF)  # the second has the top bit set: a negative int64 on the device


@pytest.fixture(scope="module")
def dx(cuda_device):
    import diffusion_extensions_b200 as pkg

    pkg._lib.load()
    return pkg


def seed_tensor(S, device):
    """One int64 element holding the 64 bits of S."""
    return torch.full((1,), S - (1 << 64) if S >= (1 << 63) else S, dtype=torch.int64, device=device)


def rows_of(dx, shape, device, unaligned=False):
    """Rotations (*shape,3,3) and translations (*shape,3); unaligned=True puts both at a 4-byte offset in their storage."""
    n = 1
    for d in shape:
        n *= d
    rot = dx.ops.quat_to_rmat(torch.randn(*shape, 4, device=device))
    shift = torch.randn(*shape, 3, device=device) * 20
    if unaligned:
        rb, sb = torch.empty(n * 9 + 1, device=device), torch.empty(n * 3 + 1, device=device)
        rb[1:].copy_(rot.reshape(-1))
        sb[1:].copy_(shift.reshape(-1))
        rot, shift = rb[1:].view(*shape, 3, 3), sb[1:].view(*shape, 3)
        assert rot.data_ptr() % 16 and shift.data_ptr() % 16
    return rot, shift


SHAPES = [(1,), (257,), (8, 33), (4099,), "unaligned"]


# ---- 1. device-seed forward noising ---------------------------------------------------------------
@pytest.mark.parametrize("lanes", ["2", "1"])
@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_dseed_noising_equals_by_value(dx, cuda_device, monkeypatch, shape, lanes):
    monkeypatch.setenv("SO3D_SE3_QS_LANES", lanes)                      # read per call: two-row (default) or one-row kernel
    torch.manual_seed(11)
    unaligned = shape == "unaligned"
    shape = (1031,) if unaligned else shape
    proc = dx.SE3Diffusion(None, shift_scale=75.0).to(cuda_device)
    R0, s0 = rows_of(dx, shape, cuda_device, unaligned)
    t = torch.randint(0, 1000, shape[:1], device=cuda_device)
    fwd, _, _ = proc.tables()
    args = (proc.sqrt_alphas_cumprod, proc.sqrt_one_minus_alphas_cumprod, fwd, 75.0)
    g = proc.guides()[0]
    for S in SEEDS:
        a = dx.ops.se3_q_sample_fused(R0, s0, t, *args, seed=seed_tensor(S, cuda_device), rng_offset=7, guide=g)
        b = dx.ops.se3_q_sample_fused(R0, s0, t, *args, seed=S, rng_offset=7, guide=g)
        for k in ("rot", "shift", "target_rot", "target_shift"):
            assert torch.equal(a[k], b[k]), (k, hex(S))
        assert torch.isfinite(a["shift"]).all()
    n = shape[0]
    if len(shape) == 1 and n > 300:                                     # sharding: a slice at row_offset 300
        part = dx.ops.se3_q_sample_fused(R0[300:], s0[300:], t[300:], *args, seed=seed_tensor(SEEDS[0], cuda_device), rng_offset=7,
                                         row_offset=300, guide=g)
        full = dx.ops.se3_q_sample_fused(R0, s0, t, *args, seed=seed_tensor(SEEDS[0], cuda_device), rng_offset=7, guide=g)
        for k in ("rot", "shift", "target_rot", "target_shift"):
            assert torch.equal(part[k], full[k][300:]), k


# ---- 2. device-seed reverse step ----------------------------------------------------------------
def reverse_step_cases(dx, device):
    """Shared-t device-seed reverse step == by-value step at seed = *seed_dev, both halves, for several shapes and steps;
    at t = 0 both halves are the posterior mean.  Also run in a child process with SO3D_SE3_PSTEP_LANES=1."""
    torch.manual_seed(12)
    proc = dx.SE3Diffusion(None, shift_scale=75.0).to(device)
    sched = (proc.sqrt_recip_alphas_cumprod, proc.sqrt_recipm1_alphas_cumprod, proc.posterior_mean_coef1, proc.posterior_mean_coef2)
    _, post, _ = proc.tables()
    sigma = proc._sigma()
    for shape in SHAPES:
        unaligned = shape == "unaligned"
        shape = (1031,) if unaligned else shape
        Rt, st = rows_of(dx, shape, device, unaligned)
        pr, ps = torch.randn(*shape, 3, device=device) * 0.3, torch.randn(*shape, 3, device=device)
        for step in (0, 1, 400, 999):
            t = torch.tensor([step], device=device)
            for S in SEEDS:
                a = dx.ops.se3_p_sample_fused(Rt, st, pr, ps, t, *sched, sigma, 75.0, post_cdf=post, seed=seed_tensor(S, device), rng_offset=5,
                                              row_offset=3)
                b = dx.ops.se3_p_sample_fused(Rt, st, pr, ps, t, *sched, sigma, 75.0, post_cdf=post, seed=S, rng_offset=5, row_offset=3)
                assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), (shape, step, hex(S))
            if step == 0:                                               # no noise on either half
                m = dx.ops.se3_p_sample_fused(Rt, st, pr, ps, t, *sched, sigma, 75.0, post_cdf=None)
                assert torch.equal(a[0], m[0]) and torch.equal(a[1], m[1])
            else:
                assert not torch.equal(a[1], dx.ops.se3_p_sample_fused(Rt, st, pr, ps, t, *sched, sigma, 75.0, post_cdf=None)[1])


def test_dseed_reverse_step_equals_by_value(dx, cuda_device):
    reverse_step_cases(dx, cuda_device)


def test_dseed_reverse_step_one_row_kernel(dx, cuda_device):
    """The one-row kernel (SO3D_SE3_PSTEP_LANES=1) is chosen once per process, so this leg runs in a child process."""
    child = ("import sys, torch; sys.path.insert(0, sys.argv[1]); import diffusion_extensions_b200 as dx; "
             "from tests.test_gpu_se3_graph import reverse_step_cases; reverse_step_cases(dx, torch.device('cuda:0')); print('OK')")
    env = dict(os.environ, SO3D_SE3_PSTEP_LANES="1", PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-c", child, ROOT], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("OK"), p.stdout[-2000:] + p.stderr[-4000:]


# ---- 3. a captured launch follows the seed tensor ----------------------------------------------------
def test_graph_replay_follows_the_seed(dx, cuda_device):
    torch.manual_seed(13)
    n, S = 3001, SEEDS[1]
    proc = dx.SE3Diffusion(None, shift_scale=75.0).to(cuda_device)
    R0, s0 = rows_of(dx, (n,), cuda_device)
    t = torch.randint(0, 1000, (n,), device=cuda_device)
    fwd, post, _ = proc.tables()
    qargs = (proc.sqrt_alphas_cumprod, proc.sqrt_one_minus_alphas_cumprod, fwd, 75.0)
    sched = (proc.sqrt_recip_alphas_cumprod, proc.sqrt_recipm1_alphas_cumprod, proc.posterior_mean_coef1, proc.posterior_mean_coef2)
    pr, ps = torch.randn(n, 3, device=cuda_device) * 0.3, torch.randn(n, 3, device=cuda_device)
    tp = torch.tensor([321], device=cuda_device)
    g = proc.guides()[0]
    seed_t = seed_tensor(S, cuda_device)

    def launches():
        q = dx.ops.se3_q_sample_fused(R0, s0, t, *qargs, seed=seed_t, rng_offset=0, guide=g)
        p = dx.ops.se3_p_sample_fused(R0, s0, pr, ps, tp, *sched, proc._sigma(), 75.0, post_cdf=post, seed=seed_t, rng_offset=9)
        return q, p

    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        launches()
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        seed_t.add_(1)
        q, p = launches()
    outs = []
    for k in (1, 2):
        graph.replay()
        Sk = (S + k) & MASK64
        qr = dx.ops.se3_q_sample_fused(R0, s0, t, *qargs, seed=Sk, rng_offset=0, guide=g)
        pr_rot, pr_shift = dx.ops.se3_p_sample_fused(R0, s0, pr, ps, tp, *sched, proc._sigma(), 75.0, post_cdf=post, seed=Sk, rng_offset=9)
        for key in ("rot", "shift", "target_rot", "target_shift"):
            assert torch.equal(q[key], qr[key]), (k, key)
        assert torch.equal(p[0], pr_rot) and torch.equal(p[1], pr_shift), k
        outs.append(q["target_shift"].clone())
    assert not torch.equal(outs[0], outs[1])
    assert int(seed_t.item()) & MASK64 == (S + 2) & MASK64


# ---- 4. graphed SE(3) training step --------------------------------------------------------------
class Net(torch.nn.Module):
    """The small AffineT denoiser of test_se3_module_end_to_end; records the step-index shapes it is handed."""

    def __init__(self, dx):
        super().__init__()
        self.dx = dx
        self.lin = torch.nn.Linear(13, 6)
        self.seen_t = []

    def forward(self, x, t):
        self.seen_t.append((tuple(t.shape), t.is_contiguous(), t.stride()))
        tt = t.reshape(tuple(t.shape) + (1,) * (x.shift.dim() - t.dim())).expand(x.shift.shape[:-1] + (1,)).float() / 1000
        h = self.lin(torch.cat([x.rot.flatten(-2), x.shift / 75.0, tt], -1))
        return self.dx.AffineGrad(h[..., :3], h[..., 3:])


def test_graphed_se3_train_step(dx, cuda_device):
    torch.manual_seed(14)
    B, Nres = 8, 32
    net = Net(dx).to(cuda_device)
    proc = dx.SE3Diffusion(net).to(cuda_device)
    opt = torch.optim.Adam(net.parameters(), lr=1e-2, capturable=True)
    z90 = torch.tensor([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]], device=cuda_device)
    rot = torch.stack([z90, z90.T]).repeat(B * Nres // 2, 1, 1).reshape(B, Nres, 3, 3)   # a fixed toy target: frames at the origin
    batch = dx.AffineT(rot, torch.zeros(B, Nres, 3, device=cuda_device))
    step = proc.make_graphed_train_step(opt, batch)
    assert isinstance(step.static_x, dx.AffineT)
    s0 = int(proc._device_seed.item())
    losses = torch.stack([step(batch).detach().clone() for _ in range(400)]).cpu()
    assert torch.isfinite(losses).all()
    assert len(set(losses[:20].tolist())) == 20                               # fresh t and noise on every replay
    assert losses[-50:].mean() < 0.8 * losses[:50].mean()                     # and it learns
    assert int(proc._device_seed.item()) == s0 + 400                          # one seed per replay


# ---- 5. graphed SE(3) sampling loop --------------------------------------------------------------
@pytest.mark.parametrize("shape", [(700,), (3, 17)], ids=str)
@pytest.mark.parametrize("projected", [False, True], ids=["SE3Diffusion", "ProjectedSE3Diffusion"])
def test_se3_p_sample_loop_as_cuda_graph(dx, cuda_device, shape, projected):
    T = 40
    torch.manual_seed(15)
    net = Net(dx).to(cuda_device)
    proc = (dx.ProjectedSE3Diffusion if projected else dx.SE3Diffusion)(net, timesteps=T).to(cuda_device)
    sched = (proc.sqrt_recip_alphas_cumprod, proc.sqrt_recipm1_alphas_cumprod, proc.posterior_mean_coef1, proc.posterior_mean_coef2)
    proj = lambda a: dx.AffineT(a.rot, a.shift * 0.5)

    def run(torch_seed, rng_seed, projection=proj):
        torch.manual_seed(torch_seed)
        dx.ops.manual_seed(rng_seed)
        if projected:
            return proc.p_sample_loop(shape, projection, cuda_graph=True)
        return proc.p_sample_loop(shape, cuda_graph=True)

    def eager_with_seed(torch_seed, rng_seed, projection=proj):
        torch.manual_seed(torch_seed)
        dx.ops.manual_seed(rng_seed)
        rot = dx.ops.quat_to_rmat(torch.randn(*shape, 4, device=cuda_device))                      # the loop's init draws
        shift = torch.randn(*shape, 3, device=cuda_device) * (1.0 if projected else proc.shift_scale)
        seed, off = dx.ops.rng.next()                                                               # the graph's seed draw
        mixed = (seed + 0x9E3779B97F4A7C15 * (off + 1)) & MASK64
        _, post, t_range = proc.tables()
        x = dx.AffineT(rot, shift)
        with torch.no_grad():
            for i in reversed(range(T)):
                pred = net(projection(x) if projected else x, torch.full(shape[:1], i, device=cuda_device, dtype=torch.long))
                r, s = dx.ops.se3_p_sample_fused(x.rot, x.shift, pred.rot_g, pred.shift_g, t_range[i:i + 1], *sched, proc._sigma(), proc.shift_scale,
                                                 post_cdf=post, seed=mixed, rng_offset=i)
                x = dx.AffineT(r, s)
        return x

    a = run(5, 31)
    ref = eager_with_seed(5, 31)
    assert torch.equal(a.rot, ref.rot) and torch.equal(a.shift, ref.shift)
    assert a.rot.shape == (*shape, 3, 3) and a.shift.shape == (*shape, 3)
    a2 = run(5, 31)                                                          # replay of the cached graph, same seeds
    torch.manual_seed(5)                                                     # same initial frames, ...
    b = proc.p_sample_loop(shape, proj, cuda_graph=True) if projected else proc.p_sample_loop(shape, cuda_graph=True)  # ... next seed
    assert torch.equal(a2.rot, a.rot) and torch.equal(a2.shift, a.shift)
    assert not torch.equal(b.rot, a.rot) and not torch.equal(b.shift, a.shift)
    assert len(proc._loop_graphs) == 1
    assert all(s == (shape[:1], True, (1,)) for s in net.seen_t)            # the denoiser saw a contiguous (B,) step index
    eye = torch.eye(3, device=cuda_device)
    assert float((b.rot.transpose(-1, -2) @ b.rot - eye).abs().max()) < 5e-6
    assert torch.isfinite(b.shift).all()
    if projected:                                                            # a new projection closure: re-captured
        proj2 = lambda a: dx.AffineT(a.rot, a.shift * 0.25)
        c = run(6, 33, proj2)
        assert len(proc._loop_graphs) == 2
        ref = eager_with_seed(6, 33, proj2)
        assert torch.equal(c.rot, ref.rot) and torch.equal(c.shift, ref.shift)
    n_graphs = len(proc._loop_graphs)
    net.eval()                                                               # train/eval mode is part of the cache key
    c = run(7, 34)
    assert len(proc._loop_graphs) == n_graphs + 1
    ref = eager_with_seed(7, 34)
    assert torch.equal(c.rot, ref.rot) and torch.equal(c.shift, ref.shift)


# ---- 6. errors -----------------------------------------------------------------------------------
def test_device_seed_errors(dx, cuda_device):
    n = 64
    proc = dx.SE3Diffusion(None).to(cuda_device)
    R0, s0 = rows_of(dx, (n,), cuda_device)
    fwd, post, _ = proc.tables()
    qargs = (proc.sqrt_alphas_cumprod, proc.sqrt_one_minus_alphas_cumprod, fwd, 75.0)
    sched = (proc.sqrt_recip_alphas_cumprod, proc.sqrt_recipm1_alphas_cumprod, proc.posterior_mean_coef1, proc.posterior_mean_coef2)
    pr = torch.zeros(n, 3, device=cuda_device)
    t1 = torch.tensor([10], device=cuda_device)
    good = seed_tensor(5, cuda_device)
    bad = [torch.full((1,), 5, dtype=torch.int32, device=cuda_device), torch.full((1,), 5, dtype=torch.int64),
           torch.full((2,), 5, dtype=torch.int64, device=cuda_device)]
    for s in bad:
        with pytest.raises(ValueError):
            dx.ops.se3_q_sample_fused(R0, s0, t1, *qargs, seed=s, rng_offset=0)
        with pytest.raises(ValueError):
            dx.ops.se3_p_sample_fused(R0, s0, pr, pr, t1, *sched, proc._sigma(), 75.0, post_cdf=post, seed=s, rng_offset=0)
    with pytest.raises(ValueError):                                          # per-row t
        dx.ops.se3_p_sample_fused(R0, s0, pr, pr, torch.full((n,), 10, device=cuda_device), *sched, proc._sigma(), 75.0, post_cdf=post, seed=good,
                                  rng_offset=0)
    with pytest.raises(ValueError):                                          # no post_cdf
        dx.ops.se3_p_sample_fused(R0, s0, pr, pr, t1, *sched, proc._sigma(), 75.0, post_cdf=None, seed=good, rng_offset=0)
    with pytest.raises(ValueError):                                          # no explicit rng_offset
        dx.ops.se3_p_sample_fused(R0, s0, pr, pr, t1, *sched, proc._sigma(), 75.0, post_cdf=post, seed=good)
    with pytest.raises(ValueError):
        dx.ops.se3_q_sample_fused(R0, s0, t1, *qargs, seed=good)
    assert int(good.item()) == 5                                             # nothing was launched
