"""The series evaluator (modes series / series_adaptive / series_pure) runs two rows per thread with packed FP32 by default;
the one-row kernel (SO3D_LOGP_LANES=1) must give the same bits: sizes above the one-warp-per-rotation threshold (64 rows
per SM, read once per process) with ragged last tiles, truncations L with and without a ragged top block, per-row and
shared eps, unaligned input (the non-TMA path), with and without the dlogf output, and the bench's E-set at 2^24 + 7 rows."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

MODES = ("series", "series_adaptive", "series_pure")


@pytest.fixture(scope="module")
def dx(cuda_device):
    import diffusion_extensions_b200 as pkg

    pkg._lib.load()
    return pkg


def bits(t):
    return None if t is None else t.view(torch.int32)  # bit patterns: NaN rows (raw series far out) compare too


def one_vs_two(ops, monkeypatch, R, eps, mode, L, want_dlogf):
    res = {}
    for lanes in ("1", "2"):
        monkeypatch.setenv("SO3D_LOGP_LANES", lanes)
        res[lanes] = ops.igso3_logp_score(R, eps, mode=mode, L=L, want_dlogf=want_dlogf)
    for x, y in zip(res["1"], res["2"]):
        assert (x is None) == (y is None)
        if x is not None:
            assert torch.equal(bits(x), bits(y)), (R.shape[0], mode, L, eps.numel(), want_dlogf)


def rotations(ops, n, g, device):
    """Half E-set-like rows (omega = eps sqrt2 k, k < 5: both sides of the guard at 4.2 eps), half uniform rotations;
    eps log-uniform in [6.4e-3, 1.35] (some rows above eps = 1, where the guard never applies)."""
    eps = torch.exp(torch.empty(n, device=device).uniform_(math.log(6.4e-3), 0.3, generator=g))
    k = torch.empty(n, device=device).uniform_(0.0, 5.0, generator=g)
    om = torch.clamp(eps * math.sqrt(2.0) * k, max=3.1)
    axis = torch.randn(n, 3, device=device, generator=g)
    R = ops.aa_to_rmat(axis, om)
    R[1::2] = ops.quat_to_rmat(torch.randn(n // 2, 4, device=device, generator=g))
    R[3] = torch.eye(3, device=device)
    return R, eps


@pytest.mark.parametrize("n", [9473, 65_569, 256 * 148 * 8 + 45])
def test_two_row_series_equals_one_row(dx, cuda_device, monkeypatch, n):
    ops = dx.ops
    g = torch.Generator(device=cuda_device)
    g.manual_seed(n)
    R, eps = rotations(ops, n, g, cuda_device)
    buf = torch.empty(n * 9 + 1, device=cuda_device)
    Ru = buf[1:].view(n, 3, 3)
    Ru.copy_(R)
    for L in (2000, 2001, 33, 2896):
        for mode in MODES:
            one_vs_two(ops, monkeypatch, R, eps, mode, L, want_dlogf=False)
            one_vs_two(ops, monkeypatch, R, eps[5:6], mode, L, want_dlogf=True)
            one_vs_two(ops, monkeypatch, Ru, eps, mode, L, want_dlogf=True)


def test_two_row_series_equals_one_row_at_bench_size(dx, cuda_device, monkeypatch):
    import bench

    n = (1 << 24) + 7
    R, eps = bench.make_eset(n, cuda_device, bench.SEED)
    for mode in MODES:
        one_vs_two(dx.ops, monkeypatch, R, eps, mode, 2000, want_dlogf=True)
