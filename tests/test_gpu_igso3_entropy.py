"""GPU tier: IsotropicGaussianSO3.entropy / IGSO3xR3.entropy / ops.igso3_entropy (so3d_igso3_entropy_f32) against the fp64
law of tests/igso3_entropy_law.py, within igso3_entropy_law.entropy_tol (c = 8)."""
import math

import numpy as np
import pytest
import torch

from tests import igso3_entropy_law as E

pytestmark = pytest.mark.gpu

GRID = np.float32(np.concatenate([np.logspace(-20, math.log10(6.0), 61), [0.3, 1.0, np.nextafter(np.float32(0.3), np.float32(0))]]))
_TRUTH = {}


def truth(eps):
    """fp64 (H, dH/deps) per element of a float32 array (cached per distinct value)."""
    eps = np.asarray(eps, np.float32)
    for e in np.unique(eps):
        if float(e) not in _TRUTH:
            _TRUTH[float(e)] = E.entropy(float(e))
    H = np.vectorize(lambda e: _TRUTH[float(e)][0])(eps)
    d = np.vectorize(lambda e: _TRUTH[float(e)][1])(eps)
    return np.asarray(H, np.float64), np.asarray(d, np.float64)


def check(eps, H, d, label):
    """Largest err/tol of H and dH/deps over the elements; assert <= 1."""
    eps = eps.detach().cpu().numpy().astype(np.float32).reshape(-1)
    H = H.detach().cpu().double().numpy().reshape(-1)
    d = d.detach().cpu().double().numpy().reshape(-1)
    uniq, inv = np.unique(eps, return_inverse=True)
    th, td = truth(uniq)
    tol = np.array([E.entropy_tol(e, a, b) for e, a, b in zip(uniq, th, td)])
    rh = np.abs(H - th[inv]) / tol[inv, 0]
    rd = np.abs(d - np.sign(eps) * td[inv]) / tol[inv, 1]
    print(f"{label}: max err/tol H {rh.max():.3f} (eps {eps[rh.argmax()]:.3g}), dH/deps {rd.max():.3f} (eps {eps[rd.argmax()]:.3g})")
    assert rh.max() <= 1.0 and rd.max() <= 1.0, label


def dist(eps, **kw):
    from diffusion_extensions_b200.distributions import IsotropicGaussianSO3

    return IsotropicGaussianSO3(eps, **kw)


@pytest.mark.parametrize("shape", [(), (7,), (3, 5), (2 ** 20 + 3,)])
def test_entropy_and_grad_against_fp64(shape):
    g = torch.Generator().manual_seed(11)
    n = int(np.prod(shape)) if shape else 1
    idx = torch.randint(0, len(GRID), (n,), generator=g)
    eps = torch.from_numpy(GRID)[idx].reshape(shape).cuda().requires_grad_(True)
    H = dist(eps).entropy()
    assert H.shape == eps.shape and H.dtype == torch.float32
    H.sum().backward()
    check(eps, H, eps.grad, f"shape {shape}")


def test_whole_grid_and_special_values():
    from diffusion_extensions_b200 import ops

    eps = torch.from_numpy(np.concatenate([GRID, -GRID])).cuda()
    H, d = ops.igso3_entropy(eps, want_grad=True)
    check(eps, H, d, "grid, both signs")
    H0, d0 = ops.igso3_entropy(torch.tensor([0.0, -0.0, float("nan"), float("inf"), 8.0], device="cuda"), want_grad=True)
    H0, d0 = H0.tolist(), d0.tolist()
    assert H0[:2] == [-math.inf] * 2 and d0[:2] == [math.inf] * 2
    assert math.isnan(H0[2]) and math.isnan(d0[2])
    assert H0[3:] == [0.0, 0.0] and d0[3:] == [0.0, 0.0]
    # no gradient output requested: the same H bits
    H1, none = ops.igso3_entropy(eps)
    assert none is None and torch.equal(H1, ops.igso3_entropy(eps, want_grad=True)[0])


def test_scalar_equals_the_same_value_in_a_batch():
    vals = torch.from_numpy(GRID).cuda()
    batch = dist(vals).entropy()
    for i in range(0, len(GRID), 7):
        e = vals[i].clone().requires_grad_(True)
        h = dist(e).entropy()
        assert h.shape == ()
        h.backward()
        eb = vals.clone().requires_grad_(True)
        dist(eb).entropy().sum().backward()
        assert torch.equal(h.detach(), batch[i]) and torch.equal(e.grad, eb.grad[i])


def test_independent_of_mean_mode_sampler_and_quirks_raise():
    eps = torch.tensor([0.05, 0.3, 1.0, 2.0], device="cuda")
    ref = dist(eps).entropy()
    mean = torch.linalg.qr(torch.randn(4, 3, 3, device="cuda"))[0]
    assert torch.equal(dist(eps, mean=mean, mode="series", series_terms=500, sampler="exact").entropy(), ref)
    with pytest.raises(ValueError):
        dist(eps, reference_quirks=True).entropy()


@pytest.mark.parametrize("eps", [0.05, 0.3, 1.0, 2.0])
def test_monte_carlo_matches(eps):
    """-log_prob over 2^22 exact draws estimates H; it lies within 4 standard errors of entropy()."""
    torch.manual_seed(1234)
    d = dist(torch.tensor(eps, device="cuda"), sampler="exact")
    with torch.no_grad():
        lp = d.log_prob(d.sample((2 ** 22,))).double().reshape(-1)
    est, se = -lp.mean().item(), lp.std().item() / math.sqrt(lp.numel())
    H = d.entropy().item()
    z = (est - H) / se
    print(f"eps {eps}: MC {est:.8g} +- {se:.2g}, entropy() {H:.8g}, z {z:+.2f}")
    assert abs(z) < 4.0


def test_igso3xr3_entropy_is_the_sum_of_its_parts():
    from diffusion_extensions_b200.distributions import IGSO3xR3

    eps = torch.tensor([0.1, 0.5, 1.5], device="cuda", requires_grad=True)
    d = IGSO3xR3(eps, shift_scale=2.0)
    H = d.entropy()
    rot = d.igso3.entropy()
    sh = 1.5 * (1 + math.log(2 * math.pi)) + 3 * torch.log(eps * 2.0)
    assert H.shape == eps.shape
    torch.testing.assert_close(H, rot + sh, rtol=0, atol=1e-5)
    H.sum().backward()
    want = torch.tensor([E.entropy(float(e))[1] for e in eps.detach().cpu()], dtype=torch.float32, device="cuda") + 3 / eps.detach()
    torch.testing.assert_close(eps.grad, want, rtol=1e-5, atol=0)


def test_graph_captured_entropy_replays():
    static = torch.tensor([0.01, 0.2, 0.7, 3.0], device="cuda")
    d = dist(static)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        d.entropy()  # warm up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = d.entropy()
    for vals in ([0.01, 0.2, 0.7, 3.0], [1e-10, 0.3, 1.0, 4.0]):
        static.copy_(torch.tensor(vals, device="cuda"))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, dist(static.clone()).entropy())
