"""GPU tier: the table-free IGSO(3) sampler (ops.igso3_sample_exact, IsotropicGaussianSO3(sampler="exact")).

Accuracy with given u against the fp64 inverse CDF of the angle law (tests/igso3_angle_law.py), the law itself by a
Kolmogorov-Smirnov test of the probability integral transform, the Philox draws it shares with the table sampler,
the outputs and error cases, and the memory of a 2^24-row per-row-eps draw."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest
import torch
from scipy import stats

import diffusion_extensions_b200 as dx
from diffusion_extensions_b200 import ops, util
from tests import igso3_angle_law as A

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PI32 = float(np.float32(math.pi))


def _u_grid():
    """Dense near 0 and near 1 (down to the smallest gaps of a 24-bit uniform), even in the bulk."""
    return np.concatenate([np.logspace(-9, -2, 40), np.linspace(0.01, 0.99, 99), 1 - np.logspace(-2, -7.2, 40)]).astype(np.float32)


EPS_GRID = np.float32(np.exp(np.linspace(math.log(1e-3), math.log(4.0), 15)))


def _check_given_u(eps64, u, w_got, label):
    """|F64(w_got) - u| <= 2e-6 everywhere; |w_got - w64| <= 1e-5 w64 where p64(w) w >= 0.1."""
    w = w_got.astype(np.float64)
    cdf_err = np.abs(A.igso3_angle_cdf_images(w, eps64) - u)
    w64 = A.igso3_angle_icdf(u.astype(np.float64), eps64)
    bulk = A.igso3_angle_pdf(w64, eps64) * w64 >= 0.1
    rel = np.abs(w - w64) / w64
    print(f"{label}: max |F(w) - u| = {cdf_err.max():.2e}, bulk max |dw|/w = {rel[bulk].max():.2e}")
    assert np.all((w >= 0) & (w <= PI32))
    assert cdf_err.max() <= 2e-6
    assert rel[bulk].max() <= 1e-5
    return cdf_err.max()


def test_given_u_accuracy_scalar_eps(cuda_device):
    u = _u_grid()
    ud = torch.tensor(u, device=cuda_device)
    worst = 0.0
    for e in EPS_GRID:
        _, ang = ops.igso3_sample_exact(float(e), (u.size,), u=ud, seed=1, rng_offset=0, want_angle=True)
        worst = max(worst, _check_given_u(np.full(u.size, float(e)), u, ang.cpu().numpy(), f"eps={e:.4g}"))
        # the table sampler on the same u, for comparison (printed, not asserted)
        d = dx.IsotropicGaussianSO3(torch.tensor(e, device=cuda_device))
        _, ang_t = d.sample((u.size,), u=ud, return_angle=True)
        terr = np.abs(A.igso3_angle_cdf_images(ang_t.cpu().numpy().astype(np.float64), float(e)) - u).max()
        print(f"    table sampler on the same u: max |F(w) - u| = {terr:.2e}")
    print("exact sampler, worst |F(w) - u| over eps in [1e-3, 4]:", worst)


def test_given_u_accuracy_per_row_eps(cuda_device):
    u = _u_grid()
    uu, ee = np.meshgrid(u, EPS_GRID, indexing="ij")
    uu, ee = uu.ravel().copy(), ee.ravel().copy()
    _, ang = ops.igso3_sample_exact(torch.tensor(ee, device=cuda_device), (uu.size,), u=torch.tensor(uu, device=cuda_device),
                                    seed=2, rng_offset=0, want_angle=True)
    w = ang.cpu().numpy()
    for e in EPS_GRID:  # the fp64 reference per eps value (one image count each)
        sel = ee == e
        _check_given_u(np.float64(e), uu[sel], w[sel], f"per-row eps={e:.4g}")


LAW_EPS = [0.005, 0.05, 0.5, 1.0, 2.0, "per_row"]


@pytest.mark.parametrize("eps", LAW_EPS)
def test_law_ks_and_isotropy(cuda_device, eps):
    n = 1 << 20
    if eps == "per_row":
        rng = np.random.default_rng(5)
        e64 = np.exp(rng.uniform(math.log(4.67e-3), 0.0, n)).astype(np.float32).astype(np.float64)
        eps_t = torch.tensor(e64, dtype=torch.float32, device=cuda_device)
    else:
        e64 = np.full(n, np.float64(np.float32(eps)))
        eps_t = float(eps)
    # a stream of its own per case (the probability integral transform of an exact sampler returns u itself)
    R, ang, axis = ops.igso3_sample_exact(eps_t, (n,), seed=20261020, rng_offset=7 + LAW_EPS.index(eps), want_angle=True,
                                          want_axis=True)
    w = ang.cpu().numpy().astype(np.float64)
    pit = np.empty(n)
    for chunk in np.array_split(np.arange(n), 16):
        pit[chunk] = A.igso3_angle_cdf_images(w[chunk], e64[chunk])
    res = stats.kstest(pit, "uniform")
    print(f"eps={eps}: KS D = {res.statistic:.2e}, p = {res.pvalue:.3f}")
    assert res.pvalue > 1e-3
    m = axis.double().mean(0).cpu().numpy()
    assert np.abs(m).max() < 5 / math.sqrt(n), m
    # the matrix is the rotation by `ang` about `axis`
    tr = R.double().diagonal(dim1=-2, dim2=-1).sum(-1).cpu().numpy()
    assert np.abs(np.clip((tr - 1) / 2, -1, 1) - np.cos(w)).max() < 2e-6


@pytest.fixture(scope="module")
def philox(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hm") / "host_math.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "host_math", "host_math.cpp")])
    return ctypes.CDLL(so)


def _device_u(philox, seed, row0, offset, n):
    """The uniform the sampling kernels draw: word z of Philox(seed, row0 + i, offset), converted toward zero / 2^32."""
    out = np.empty(4 * n, np.uint32)
    philox.hm_philox(ctypes.c_ulonglong(seed), ctypes.c_ulonglong(row0), ctypes.c_ulonglong(offset),
                     out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), ctypes.c_long(n))
    z = out.reshape(n, 4)[:, 2].astype(np.uint64)
    bits = np.floor(np.log2(np.maximum(z, 1).astype(np.float64))).astype(np.int64) + 1
    shift = np.maximum(bits - 24, 0).astype(np.uint64)
    z = (z >> shift) << shift  # round toward zero to 24 significant bits
    return (z.astype(np.float64) / 2.0 ** 32).astype(np.float32)


def test_same_draws_as_the_table_sampler(cuda_device, philox):
    n, seed, off, row0 = 50_000, 0x1234_5678_9ABC, 3, 1000
    eps = torch.exp(torch.empty(n, device=cuda_device).uniform_(math.log(4.67e-3), 0.0))
    _, ang_x, ax_x = ops.igso3_sample_exact(eps, (n,), seed=seed, rng_offset=off, row_offset=row0, want_angle=True, want_axis=True)
    d = dx.IsotropicGaussianSO3(eps)
    row_idx = torch.arange(n, device=cuda_device)
    _, ang_t, ax_t = ops.igso3_sample(d.table, (n,), row_idx=row_idx, seed=seed, rng_offset=off, row_offset=row0, want_angle=True,
                                      want_axis=True)
    assert torch.equal(ax_x, ax_t)
    # both samplers saw the u of the Philox layout: explicit u reproduces each one's angle bit for bit
    u = torch.tensor(_device_u(philox, seed, row0, off, n), device=cuda_device)
    _, ang_xu = ops.igso3_sample_exact(eps, (n,), u=u, seed=seed, rng_offset=off, row_offset=row0, want_angle=True)
    _, ang_tu = ops.igso3_sample(d.table, (n,), row_idx=row_idx, u=u, seed=seed, rng_offset=off, row_offset=row0, want_angle=True)
    assert torch.equal(ang_xu, ang_x)
    assert torch.equal(ang_tu, ang_t)
    # shards with row_offset concatenate to the unsharded draw
    R_all, ang_all = ops.igso3_sample_exact(eps, (n,), seed=seed, rng_offset=off, want_angle=True)
    cuts = [0, 7, 12_345, 40_000, n]
    parts = [ops.igso3_sample_exact(eps[a:b], (b - a,), seed=seed, rng_offset=off, row_offset=a, want_angle=True) for a, b in zip(cuts, cuts[1:])]
    assert torch.equal(torch.cat([p[0] for p in parts]), R_all)
    assert torch.equal(torch.cat([p[1] for p in parts]), ang_all)


def test_outputs_mean_and_shapes(cuda_device):
    torch.manual_seed(0)
    eps = torch.tensor([0.01, 0.3, 1.5], device=cuda_device)
    d = dx.IsotropicGaussianSO3(eps, sampler="exact")
    R = d.sample((1000, 4))
    assert R.shape == (1000, 4, 3, 3, 3)
    Rd = R.reshape(-1, 3, 3).double()
    eye = torch.eye(3, dtype=torch.float64, device=cuda_device)
    assert (Rd.transpose(-1, -2) @ Rd - eye).abs().max() <= 5e-6
    assert (torch.linalg.det(Rd) - 1).abs().max() <= 5e-6
    assert d._table is None  # sampling never built the table
    assert d.trap.shape == (ops.CDF_POINTS, 3) and d._table is not None  # reading it still does
    # the per-column eps is respected
    _, ang = dx.IsotropicGaussianSO3(eps, sampler="exact").sample((20000,), return_angle=True)
    med = ang.median(0).values.cpu().numpy()
    for j, e in enumerate(eps.tolist()):
        want = A.igso3_angle_icdf(0.5, e)
        assert abs(med[j] - want) < 0.05 * want
    # mean as the left factor: one 3x3 and per-row
    u = torch.rand(6, device=cuda_device)
    axes = torch.randn(6, 3, device=cuda_device)
    base = ops.igso3_sample_exact(0.2, (6,), u=u, axes=axes)
    M = util.exp_vec(torch.randn(6, 3, device=cuda_device))
    got = ops.igso3_sample_exact(0.2, (6,), u=u, axes=axes, mean=M)
    assert (got - M @ base).abs().max() < 2e-6
    got1 = ops.igso3_sample_exact(0.2, (6,), u=u, axes=axes, mean=M[2])
    assert (got1 - M[2] @ base).abs().max() < 2e-6
    dm = dx.IsotropicGaussianSO3(torch.tensor(0.2, device=cuda_device), mean=M, sampler="exact")
    assert dm.sample(u=u, axes=axes).shape == (6, 3, 3)
    assert (dm.sample(u=u, axes=axes) - M @ base).abs().max() < 2e-6


def test_special_inputs_and_errors(cuda_device):
    n = 4
    u = torch.tensor([0.0, 0.5, 0.5, 1e-30], device=cuda_device)
    eps = torch.tensor([0.1, float("nan"), 0.5, 0.1], device=cuda_device)
    M = torch.eye(3, device=cuda_device) * torch.tensor([1.0, -1.0, -1.0], device=cuda_device)
    R, ang = ops.igso3_sample_exact(eps, (n,), u=u, seed=0, rng_offset=0, mean=M, want_angle=True)
    assert ang[0].item() == 0.0 and torch.equal(R[0], M)  # u = 0: the identity, then the mean
    assert math.isnan(ang[1].item()) and torch.isnan(R[1]).any()
    assert 0.0 < ang[3].item() < 1e-3 and math.isfinite(ang[2].item())
    with pytest.raises(ValueError):
        dx.IsotropicGaussianSO3(torch.tensor(0.1, device=cuda_device), sampler="exact", reference_quirks=True)
    with pytest.raises(ValueError):
        dx.IsotropicGaussianSO3(torch.tensor(0.1, device=cuda_device), sampler="lookup")
    with pytest.raises(TypeError):
        ops.igso3_sample_exact(torch.tensor([0.1, 0.2], dtype=torch.float64, device=cuda_device), (2,))
    with pytest.raises(RuntimeError):
        ops.igso3_sample_exact(torch.tensor([0.1, 0.2]), (2,))
    # the default sampler is unchanged: the table path, bit for bit
    d0 = dx.IsotropicGaussianSO3(torch.tensor(0.1, device=cuda_device))
    assert d0.sampler == "table"
    uu = torch.rand(100, device=cuda_device)
    assert torch.equal(d0.sample((100,), u=uu, axes=torch.ones(100, 3, device=cuda_device)),
                       ops.igso3_sample(d0.table, (100,), u=uu, axes=torch.ones(100, 3, device=cuda_device)))


def test_per_row_eps_memory_2p24(cuda_device):
    n = 1 << 24
    eps = torch.exp(torch.empty(n, device=cuda_device).uniform_(math.log(4.67e-3), 0.0))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    R = dx.IsotropicGaussianSO3(eps, sampler="exact").sample()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    out_bytes = R.numel() * 4
    print(f"2^24 per-row eps: peak {peak / 2**20:.1f} MiB above the inputs, outputs {out_bytes / 2**20:.1f} MiB "
          f"(the table would take {n * ops.CDF_POINTS * 4 / 1e9:.1f} GB)")
    assert R.shape == (n, 3, 3)
    assert peak <= out_bytes + (1 << 20)
    assert torch.isfinite(R[:: 1 << 12]).all()
