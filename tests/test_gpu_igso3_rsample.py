"""GPU tier: the reparameterised exact IGSO(3) draw (IsotropicGaussianSO3.rsample, ops.igso3_rsample_bwd, IGSO3xR3.rsample).

The backward kernel's eps-gradient against the fp64 implicit derivative -(dF/deps)/p of tests/igso3_angle_deps_law.py at the
sampled angle, by stratum; eps.grad / mean.grad for a random upstream G against an fp64 restatement; Monte Carlo identities
of the law (E chi_l(R) = (2l+1) e^{-l(l+1) eps^2}, E R = e^{-2 eps^2} mean) differentiated through the estimator; bit
equality with sample(); shapes, special inputs and errors."""
import math

import numpy as np
import pytest
import torch

import diffusion_extensions_b200 as dx
from diffusion_extensions_b200 import ops
from diffusion_extensions_b200.util import AffineT
from tests import igso3_angle_deps_law as D

pytestmark = pytest.mark.gpu
U24 = 2.0 ** -24


def _hat64(a):
    z = torch.zeros_like(a[..., 0])
    return torch.stack([z, -a[..., 2], a[..., 1], a[..., 2], z, -a[..., 0], -a[..., 1], a[..., 0], z], -1).reshape(*a.shape[:-1], 3, 3)


def _rodrigues64(axis, ang):
    K = _hat64(axis)
    s, c = torch.sin(ang)[..., None, None], torch.cos(ang)[..., None, None]
    return torch.eye(3, dtype=torch.float64) + s * K + (1 - c) * (K @ K)


def _truth(eps, angle, axis, G, mean=None):
    """fp64: (g_eps per row, its tolerance, g_mean = G N^T per row).  g_eps = <mean^T G, hat(a) N> dw/deps."""
    eps = np.broadcast_to(np.asarray(eps, np.float64), angle.shape).reshape(-1)
    w = angle.double().cpu().reshape(-1)
    a = axis.double().cpu().reshape(-1, 3)
    G = G.double().cpu().reshape(-1, 3, 3)
    N = _rodrigues64(a, w)
    GN = G if mean is None else mean.double().cpu().reshape(-1, 3, 3).transpose(-1, -2) @ G
    prod = GN * (_hat64(a) @ N)
    gw = prod.sum((-1, -2)).numpy()
    scale = prod.abs().sum((-1, -2)).numpy()
    ae, wn = np.abs(eps), w.numpy()
    d = np.zeros_like(wn)
    nz = (wn > 0) & (ae > 0)
    d[nz] = D.igso3_angle_deps(wn[nz], ae[nz]) * np.sign(eps[nz])
    tol = np.abs(gw) * D.deps_tol(wn, ae, d) + 8 * U24 * scale * np.abs(d)
    return gw * d, tol, (G @ N.transpose(-1, -2)).numpy()


def _draw(cuda_device, eps, u, mean=None, seed=3):
    eps_t = eps if isinstance(eps, torch.Tensor) else torch.tensor(eps, device=cuda_device)
    shape = tuple(u.shape)
    R, ang, ax = ops.igso3_sample_exact(eps_t if eps_t.numel() == 1 else eps_t.expand(shape), shape, u=u, seed=seed, rng_offset=0,
                                        mean=mean, want_angle=True, want_axis=True)
    return R, ang, ax


STRATA = {
    "tiny w": (np.float32([1e-3, 0.05, 0.3, 1.0, 4.0]), np.concatenate([[1e-9, U24], np.logspace(-8, -4, 9)])),
    "bulk": (np.float32(np.exp(np.linspace(math.log(1e-3), math.log(4.0), 13))), np.linspace(0.01, 0.99, 99)),
    "near pi, large eps": (np.float32([1.0, 1.5, 2.0, 3.0, 4.0]), 1 - np.logspace(-2, -7, 21)),
    "regime switch": (np.float32([np.nextafter(np.float32(0.3), np.float32(0)), 0.3, np.nextafter(np.float32(0.3), np.float32(1))]),
                      np.concatenate([np.logspace(-9, -2, 8), np.linspace(0.02, 0.98, 49), 1 - np.logspace(-2, -7, 11)])),
}


@pytest.mark.parametrize("per_row", [False, True])
def test_eps_gradient_given_u_by_stratum(cuda_device, per_row):
    gen = torch.Generator().manual_seed(7)
    worst = 0.0
    for name, (eps_list, us) in STRATA.items():
        u = torch.tensor(np.asarray(us, np.float32), device=cuda_device)
        rmax = 0.0
        for e in eps_list:
            if per_row:  # per-row eps in this stratum: the same value per row, through the per-row path
                eps = torch.full(u.shape, float(e), device=cuda_device)
            else:
                eps = torch.tensor(float(e), device=cuda_device)
            _, ang, ax = _draw(cuda_device, eps, u)
            G = torch.randn(*u.shape, 3, 3, generator=gen).to(cuda_device)
            g, _ = ops.igso3_rsample_bwd(eps, ang, ax, G, u=u, want_mean_grad=False)
            t, tol, _ = _truth(float(e), ang, ax, G)
            r = np.abs(g.double().cpu().numpy() - t) / tol
            rmax = max(rmax, r.max())
            assert np.all(r <= 1.0), (name, float(e), us[r > 1.0][:5])
        print(f"{name:20s} per_row={per_row}: max err/tol {rmax:.3f}")
        worst = max(worst, rmax)
    print(f"largest err/tol {worst:.3f}")


@pytest.mark.parametrize("batched_mean", [False, True])
def test_full_eps_and_mean_gradients_random_G(cuda_device, batched_mean):
    n = 4096
    gen = torch.Generator().manual_seed(11)
    eps = torch.exp(torch.empty(n).uniform_(math.log(4.67e-3), 0.0, generator=gen)).to(cuda_device).requires_grad_()
    M = ops.exp_vec(torch.randn(n if batched_mean else 1, 3, generator=gen).to(cuda_device))
    if not batched_mean:
        M = M[0]
    M = M.clone().requires_grad_()
    G = torch.randn(n, 3, 3, generator=gen).to(cuda_device)
    d = dx.IsotropicGaussianSO3(eps, mean=M, sampler="exact")
    dx.manual_seed(5)
    R = d.rsample()
    (R * G).sum().backward()
    # the draw's angle and axis, recovered by redrawing at the same seed (bit-equal, see the sample test)
    dx.manual_seed(5)
    _, ang, ax = ops.igso3_sample_exact(eps.detach(), (n,), mean=M.detach(), want_angle=True, want_axis=True)
    t, tol, gm = _truth(eps.detach().cpu().numpy(), ang, ax, G, M.detach().expand(n, 3, 3))
    r = np.abs(eps.grad.double().cpu().numpy() - t) / tol
    print(f"eps.grad: max err/tol {r.max():.3f}")
    assert np.all(r <= 1.0)
    rows_abs = np.abs(gm).sum() if not batched_mean else None
    gm = gm if batched_mean else gm.sum(0)
    err = np.abs(M.grad.double().cpu().numpy() - gm).max()
    bound = 1e-6 * max(1.0, np.abs(gm).max()) if batched_mean else 1e-6 * rows_abs
    print(f"mean.grad: max err {err:.2e} (bound {bound:.2e})")
    assert err <= bound


@pytest.mark.parametrize("eps", [0.02, 0.1, 0.3, 1.0, 2.0])
def test_monte_carlo_identities(cuda_device, eps):
    """d/deps of the sample means of chi_1 = tr R and chi_2 = 1 + 2 cos w + 2 cos 2w, and d/dmean of the sample mean of
    <M, R>, against the derivatives of E chi_l = (2l+1) e^{-l(l+1) eps^2} and E R = e^{-2 eps^2} mean, within 5 standard
    errors estimated from the per-row gradients (n = 2^22)."""
    n = 1 << 22
    dx.manual_seed(17)
    e = torch.full((n,), eps, device=cuda_device, requires_grad=True)
    Mean = ops.exp_vec(torch.tensor([[0.3, -0.2, 0.5]], device=cuda_device))[0].requires_grad_()
    R = dx.IsotropicGaussianSO3(e, mean=Mean).rsample()
    N = Mean.detach().T @ R  # the draw without its mean: chi_l depends on it only
    c = ((N[:, 0, 0] + N[:, 1, 1] + N[:, 2, 2]) - 1) / 2
    chi1 = 2 * c + 1
    chi2 = 4 * c * c + 2 * c - 1
    Mt = torch.tensor([[0.5, -1.0, 0.2], [0.3, 0.8, -0.4], [1.1, 0.1, 0.6]], device=cuda_device)
    for name, stat, l in (("chi_1", chi1, 1), ("chi_2", chi2, 2)):
        (g,) = torch.autograd.grad(stat.sum(), e, retain_graph=True)
        g = g.double()
        est, se = g.mean().item(), g.std().item() / math.sqrt(n)
        ref = -2 * eps * l * (l + 1) * (2 * l + 1) * math.exp(-l * (l + 1) * eps * eps)
        print(f"eps {eps}: d/deps E {name} = {est:.6g} +- {se:.2g} (closed form {ref:.6g}, {abs(est - ref) / se:.2f} SE)")
        assert abs(est - ref) <= 5 * se
    # d/dmean of mean_i <Mt, R_i> = mean_i Mt N_i^T -> e^{-2 eps^2} Mt
    (gM,) = torch.autograd.grad((R * Mt).sum() / n, Mean)
    rows = (Mt @ N.transpose(-1, -2)).double()
    est, se = rows.mean(0), rows.std(0) / math.sqrt(n)
    assert torch.allclose(gM.double(), est, rtol=1e-4, atol=1e-6)
    ref = math.exp(-2 * eps * eps) * Mt.double()
    z = ((est - ref).abs() / se).max().item()
    print(f"eps {eps}: d/dmean E<M, R>: max {z:.2f} SE from e^(-2 eps^2) M")
    assert z <= 5


@pytest.mark.parametrize("per_row", [False, True])
@pytest.mark.parametrize("with_mean", [False, True])
def test_rsample_equals_sample_bit_for_bit(cuda_device, per_row, with_mean):
    eps = torch.rand(3, 5, device=cuda_device) + 0.01 if per_row else torch.tensor(0.4, device=cuda_device)
    # a batched mean that broadcasts against (*sample_shape, *eps.shape) for both sample shapes below
    mean = ops.exp_vec(torch.randn(*((3, 5) if per_row else (7,)), 3, device=cuda_device)) if with_mean else None
    d = dx.IsotropicGaussianSO3(eps, mean=mean, sampler="exact")
    for shape in ((), (7,)):
        dx.manual_seed(23)
        a = d.sample(shape)
        dx.manual_seed(23)
        b = d.rsample(shape)
        assert torch.equal(a, b)
        # one launch, one rng.next(): what follows draws the same either way
        dx.manual_seed(29)
        d.rsample(shape)
        c1 = d.sample(shape)
        dx.manual_seed(29)
        d.sample(shape)
        c2 = d.sample(shape)
        assert torch.equal(c1, c2)


def test_shapes_and_broadcast_reductions(cuda_device):
    gen = torch.Generator().manual_seed(3)
    eps = (torch.rand(4, generator=gen) * 0.5 + 0.05).to(cuda_device).requires_grad_()
    mean = ops.exp_vec(torch.randn(3, 1, 3, generator=gen).to(cuda_device)).requires_grad_()
    d = dx.IsotropicGaussianSO3(eps, mean=mean)  # table sampler: rsample is exact regardless
    dx.manual_seed(31)
    R = d.rsample()
    assert R.shape == (3, 4, 3, 3) and d.has_rsample and dx.IGSO3xR3.has_rsample
    G = torch.randn(3, 4, 3, 3, generator=gen).to(cuda_device)
    (R * G).sum().backward()
    assert eps.grad.shape == (4,) and mean.grad.shape == (3, 1, 3, 3)
    dx.manual_seed(31)
    _, ang, ax = ops.igso3_sample_exact(eps.detach().expand(3, 4), (3, 4), mean=mean.detach(), want_angle=True, want_axis=True)
    g, gm = ops.igso3_rsample_bwd(eps.detach().expand(3, 4), ang, ax, G, mean=mean.detach())
    assert torch.allclose(eps.grad, g.sum(0), rtol=1e-6, atol=1e-6)
    assert torch.allclose(mean.grad, gm.sum(1, keepdim=True), rtol=1e-6, atol=1e-6)
    # scalar eps, sample_shape, shared mean
    e0 = torch.tensor(0.2, device=cuda_device, requires_grad=True)
    m0 = ops.exp_vec(torch.tensor([0.1, 0.2, 0.3], device=cuda_device)).requires_grad_()
    R = dx.IsotropicGaussianSO3(e0, mean=m0).rsample((2, 5))
    assert R.shape == (2, 5, 3, 3)
    R.sum().backward()
    assert e0.grad.shape == () and m0.grad.shape == (3, 3) and torch.isfinite(e0.grad) and torch.isfinite(m0.grad).all()
    # u / axes given: constants of the draw
    u = torch.rand(6, device=cuda_device).requires_grad_()
    R = dx.IsotropicGaussianSO3(e0.detach().requires_grad_()).rsample((6,), u=u, axes=torch.randn(6, 3, device=cuda_device))
    R.sum().backward()
    assert u.grad is None


def test_special_inputs(cuda_device):
    u = torch.tensor([0.0, 0.3, 0.7, 0.5], device=cuda_device)
    axes = torch.tensor([[0.0, 0.0, 1.0], [1.0, 2.0, 2.0], [0.0, 1.0, 0.0], [1.0, 0.0, 0.0]], device=cuda_device)
    G = torch.randn(4, 3, 3, device=cuda_device)
    eps = torch.tensor([0.2, 0.0, -0.2, float("nan")], device=cuda_device, requires_grad=True)
    mean = ops.exp_vec(torch.tensor([0.4, 0.0, -0.1], device=cuda_device)).requires_grad_()
    R = dx.IsotropicGaussianSO3(eps, mean=mean).rsample(u=u, axes=axes)
    (R * G).sum().backward()
    g = eps.grad.cpu()
    assert torch.equal(R[0], mean.detach()) and g[0] == 0.0  # u = 0: identity (the mean), gradient 0
    # eps = 0: the eps -> 0+ limit 2 x0(u) times <mean^T G, hat(a)>
    x0 = ops.igso3_sample_exact(1e-6, (1,), u=u[1:2], seed=0, rng_offset=0, want_angle=True)[1].item() / 2e-6
    a = axes[1] / axes[1].norm()
    gw = ((mean.detach().T @ G[1]) * _hat64(a.double().cpu()).float().to(cuda_device)).sum().item()
    assert abs(g[1].item() - gw * 2 * x0) <= 1e-5 * abs(gw * 2 * x0) + 1e-6
    assert torch.isfinite(g[:3]).all() and torch.isnan(g[3])
    # negative eps: the law of |eps|, the gradient negated
    e2 = torch.tensor([0.2, -0.2], device=cuda_device, requires_grad=True)
    R2 = dx.IsotropicGaussianSO3(e2).rsample(u=u[2:3].expand(2).contiguous(), axes=axes[2:3].expand(2, 3).contiguous())
    (R2 * G[2]).sum().backward()
    assert torch.equal(R2[0], R2[1]) and e2.grad[0].item() == -e2.grad[1].item() != 0.0


def test_errors_and_double_backward(cuda_device):
    with pytest.raises(ValueError):
        dx.IsotropicGaussianSO3(torch.tensor(0.1, device=cuda_device), reference_quirks=True).rsample()
    e = torch.tensor(0.3, device=cuda_device, requires_grad=True)
    R = dx.IsotropicGaussianSO3(e).rsample((8,))
    (g,) = torch.autograd.grad(R.sum(), e, create_graph=True)
    with pytest.raises(RuntimeError):
        g.backward()


def test_backward_is_deterministic(cuda_device):
    n = 1 << 20
    eps = torch.exp(torch.empty(n, device=cuda_device).uniform_(math.log(4.67e-3), 0.0))
    u = torch.rand(n, device=cuda_device)
    mean = ops.exp_vec(torch.randn(n, 3, device=cuda_device))
    _, ang, ax = ops.igso3_sample_exact(eps, (n,), u=u, mean=mean, want_angle=True, want_axis=True)
    G = torch.randn(n, 3, 3, device=cuda_device)
    a = ops.igso3_rsample_bwd(eps, ang, ax, G, u=u, mean=mean)
    b = ops.igso3_rsample_bwd(eps, ang, ax, G, u=u, mean=mean)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_igso3xr3_rsample_gradients(cuda_device):
    n = 2048
    eps = torch.tensor(0.4, device=cuda_device, requires_grad=True)
    rot = ops.exp_vec(torch.randn(n, 3, device=cuda_device)).requires_grad_()
    shift = torch.randn(n, 3, device=cuda_device).requires_grad_()
    d = dx.IGSO3xR3(eps, mean=AffineT(rot=rot, shift=shift), shift_scale=2.0)
    dx.manual_seed(41)
    x = d.rsample()
    Gr, Gs = torch.randn(n, 3, 3, device=cuda_device), torch.randn(n, 3, device=cuda_device)
    (g_rot_eps,) = torch.autograd.grad((x.rot * Gr).sum(), eps, retain_graph=True)
    (g_shift_eps, g_shift) = torch.autograd.grad((x.shift * Gs).sum(), (eps, shift), retain_graph=True)
    ((x.rot * Gr).sum() + (x.shift * Gs).sum()).backward()
    # rotation: the same draw's angle / axis at the same seed
    dx.manual_seed(41)
    _, ang, ax = ops.igso3_sample_exact(eps.detach(), (n,), mean=rot.detach(), want_angle=True, want_axis=True)
    t, tol, gm = _truth(0.4, ang, ax, Gr, rot.detach())
    assert abs(g_rot_eps.item() - t.sum()) <= tol.sum() + 1e-5 * np.abs(t).sum()
    assert np.abs(rot.grad.double().cpu().numpy() - gm).max() <= 1e-5
    # shift: d shift / d eps = (shift - loc) / eps, d shift / d loc = I
    ref = ((x.shift.detach() - shift.detach()) / 0.4 * Gs).sum().item()
    assert abs(g_shift_eps.item() - ref) <= 1e-4 * (abs(ref) + 1)
    assert torch.equal(g_shift, Gs) and torch.allclose(shift.grad, Gs)
    assert abs(eps.grad.item() - (g_rot_eps + g_shift_eps).item()) <= 1e-5 * (abs(eps.grad.item()) + 1)
