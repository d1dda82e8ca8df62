"""Gradients of the SO(3) kernels and of the differentiable util / distribution paths against float64 torch autograd on
the CPU, applied to restatements of the reference's ops (util.py:164-205, 349-361; distributions.py:74-77).

Inputs are sampled by stratum (rotation angle, |w|, scalar size), and every check reports its maximum error per stratum so
that a failure names its region.  Two things are checked per kernel:
  * the ambient gradient (all 9 matrix entries), relative to the per-row scale max(|ref|_row, 1);
  * the tangent gradient tau = vee_adj(R^T Gamma), the part a caller that keeps R on SO(3) consumes, against the derivative
    along R exp(hat(xi)) of the fp64 restatement at the rotation the fp32 matrix represents.
Tolerances are 1e-5 .. 2e-5 where the problem is well conditioned; where they grow, the formula says why (2^-24 / sin(theta)
above pi/2 only, 2^-24 |w| for long rotation vectors).  Run with -s to see the per-stratum table.
"""
import math
import zlib

import numpy as np
import pytest
import torch

from oracle import so3_oracle as O
from tests.strata import Report, THETA_STRATA, U24, angle_of, pi_amp, rot_stratum, unit_axes

pytestmark = pytest.mark.gpu

F64 = torch.float64


@pytest.fixture(scope="module")
def dx(cuda_device):
    import diffusion_extensions_b200 as pkg

    pkg._lib.load()
    return pkg


def dev(a, device):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(device)


def host(t):
    return t.detach().cpu().numpy().astype(np.float64)


# ---------------------------------------------------------------------------------------------
# float64 restatements of the reference's ops (torch, CPU)
# ---------------------------------------------------------------------------------------------
def ref_log(r):  # util.py:164-176
    a = r - r.transpose(-1, -2)
    v = torch.stack((a[..., 2, 1], -a[..., 2, 0], a[..., 1, 0]), -1)
    s = v.norm(dim=-1) / 2
    c = (torch.einsum("...ii", r) - 1) / 2
    return (torch.atan2(s, c) / (2 * s))[..., None, None] * a


def hat_t(v):
    z = torch.zeros_like(v[..., 0])
    return torch.stack((z, -v[..., 2], v[..., 1], v[..., 2], z, -v[..., 0], -v[..., 1], v[..., 0], z), -1).reshape(v.shape[:-1] + (3, 3))


def ref_aa_to_rmat(axis, ang):  # util.py:195-205 without the SVD projection (a no-op on an exact rotation)
    return torch.matrix_exp(hat_t(axis / axis.norm(dim=-1, keepdim=True)) * ang[..., None])


def ref_scale(r, s):  # util.py:349-361
    return torch.matrix_exp(ref_log(r) * s[..., None, None])


def vee_adj(m):  # <G, hat(u)> = u . vee_adj(G)
    return np.stack((m[..., 2, 1] - m[..., 1, 2], m[..., 0, 2] - m[..., 2, 0], m[..., 1, 0] - m[..., 0, 1]), -1)


def grad64(f, *xs):
    xs = [torch.tensor(np.asarray(x, dtype=np.float64), requires_grad=True) for x in xs]
    gs = torch.autograd.grad(f(*xs), xs)
    return [g.numpy() for g in gs]


def tangent64(f, R):
    """d/dxi f(Rm exp(hat(xi))) at xi = 0, Rm the fp64 rotation with the oracle's axis-angle of the fp32 matrix R."""
    Rm = torch.tensor(O.exp_vec(O.log_vec(R.astype(np.float64))))
    xi = torch.zeros(R.shape[0], 3, dtype=F64, requires_grad=True)
    (g,) = torch.autograd.grad(f(Rm @ torch.matrix_exp(hat_t(xi))), xi)
    return g.numpy()


def row_max(a):
    return np.abs(a).reshape(a.shape[0], -1).max(-1)


# ---------------------------------------------------------------------------------------------
# so3d_log_bwd_f32
# ---------------------------------------------------------------------------------------------
def test_log_bwd_strata(dx, cuda_device):
    """Ambient gradient of <G, log_rmat(R)> vs fp64 autograd of the reference formula at the fp32 matrix, and its tangent
    part vs the derivative of the fp64 log along R exp(hat(xi)).  Near pi the reference formula's tangent part is off by
    ~2^-24/sin^2(theta) on an fp32 matrix; the kernel replaces it there (c < -0.9) with Jr^-T(theta n) vee_adj(G), good to
    ~2^-24/sin(theta), which is what both tolerances allow."""
    rng = np.random.default_rng(101)
    rep = Report("log_rmat backward (so3d_log_bwd_f32)")
    n = 2000
    for name, lo, hi in THETA_STRATA:
        R = rot_stratum(rng, n, lo, hi)
        G = rng.standard_normal((n, 3, 3)).astype(np.float32)
        Rd = dev(R, cuda_device).requires_grad_(True)
        (got,) = torch.autograd.grad((dx.util.log_rmat(Rd) * dev(G, cuda_device)).sum(), Rd)
        got = host(got)
        assert np.isfinite(got).all(), name
        u = vee_adj(G.astype(np.float64))
        tau = vee_adj(np.swapaxes(R.astype(np.float64), -1, -2) @ got)
        if name == "theta=0":
            # the formula's limit: Gamma = (G - G^T)/2, tau = vee_adj(G)
            ref = (G.astype(np.float64) - np.swapaxes(G, -1, -2)) / 2
            rep.add(name, "ambient", row_max(got - ref), 1e-6)
            rep.add(name, "tangent", row_max(tau - u), 1e-6)
            continue
        if name == "theta=pi":
            continue  # log is discontinuous at pi: only finiteness (asserted above) is defined
        G64 = torch.tensor(G, dtype=F64)
        (amb,) = grad64(lambda r: (ref_log(r) * G64).sum(), R)
        amp = pi_amp(angle_of(R))
        rep.add(name, "ambient", row_max(got - amb) / np.maximum(row_max(amb), 1.0), 2e-5 + 4 * U24 * amp)
        tref = tangent64(lambda r: (ref_log(r) * G64).sum(), R)
        rep.add(name, "tangent", np.linalg.norm(tau - tref, axis=-1) / np.maximum(np.linalg.norm(tref, axis=-1), 1.0),
                2e-5 + 8 * U24 * amp)
    rep.check()


# ---------------------------------------------------------------------------------------------
# so3d_expvec_bwd_f32
# ---------------------------------------------------------------------------------------------
W_STRATA = [("|w|=0", 0.0, 0.0), ("[1e-8,1e-4]", 1e-8, 1e-4), ("1e-2+-1%", 0.99e-2, 1.01e-2), ("[1e-2,pi]", 1e-2, math.pi),
            ("[pi,4pi]", math.pi, 4 * math.pi), ("[4pi,500]", 4 * math.pi, 500.0)]


def test_exp_vec_bwd_strata(dx, cuda_device):
    """Gradient of <G, exp(hat(w))> w.r.t. w vs fp64 autograd of torch.matrix_exp.  Lengths above pi are legitimate
    (so3_scale's backward forms w = s log R); there the fp32 angle carries 2^-24 |w| absolute error."""
    rng = np.random.default_rng(102)
    rep = Report("exp_vec backward (so3d_expvec_bwd_f32)")
    n = 2000
    for name, lo, hi in W_STRATA:
        if lo == hi:
            p = np.full(n, lo)
        elif hi <= 1e-2 or lo >= 4 * math.pi:
            p = np.exp(rng.uniform(math.log(lo), math.log(hi), n))
        else:
            p = rng.uniform(lo, hi, n)
        w = (unit_axes(rng, n) * p[:, None]).astype(np.float32)
        G = rng.standard_normal((n, 3, 3)).astype(np.float32)
        wd = dev(w, cuda_device).requires_grad_(True)
        (got,) = torch.autograd.grad((dx.util.exp_vec(wd) * dev(G, cuda_device)).sum(), wd)
        G64 = torch.tensor(G, dtype=F64)
        (ref,) = grad64(lambda v: (torch.matrix_exp(hat_t(v)) * G64).sum(), w)
        err = row_max(host(got) - ref) / np.maximum(row_max(ref), 1.0)
        rep.add(name, "grad w", err, 2e-5 + 4 * U24 * np.linalg.norm(w.astype(np.float64), axis=-1))
    rep.check()


# ---------------------------------------------------------------------------------------------
# so3d_aa_to_rmat_bwd_f32
# ---------------------------------------------------------------------------------------------
def test_aa_to_rmat_bwd_strata(dx, cuda_device):
    """Gradient of <G, aa_to_rmat(axis, ang)> w.r.t. the un-normalised axis and the angle vs fp64 autograd of
    matrix_exp(hat(axis/|axis|) ang).  Angles in [-6, 12] with tiny ones; axis norms 1e-3 .. 1e3 (the axis gradient scales
    as 1/|axis|, so it is compared after multiplying by |axis|).  A zero axis gives NaN without trapping, like the
    reference."""
    rng = np.random.default_rng(103)
    rep = Report("aa_to_rmat backward (so3d_aa_to_rmat_bwd_f32)")
    n = 2000
    strata = [("ang [-6,12]", lambda: rng.uniform(-6, 12, n)), ("|ang| [1e-7,1e-3]", lambda: rng.choice([-1, 1], n) * np.exp(rng.uniform(math.log(1e-7), math.log(1e-3), n))),
              ("ang=0", lambda: np.zeros(n))]
    for name, angf in strata:
        ang = angf().astype(np.float32)[:, None]
        nrm = np.exp(rng.uniform(math.log(1e-3), math.log(1e3), n))
        axes = (unit_axes(rng, n) * nrm[:, None]).astype(np.float32)
        G = rng.standard_normal((n, 3, 3)).astype(np.float32)
        ad, and_ = dev(axes, cuda_device).requires_grad_(True), dev(ang, cuda_device).requires_grad_(True)
        got_a, got_an = torch.autograd.grad((dx.util.aa_to_rmat(ad, and_) * dev(G, cuda_device)).sum(), (ad, and_))
        G64 = torch.tensor(G, dtype=F64)
        ref_a, ref_an = grad64(lambda a, t: (ref_aa_to_rmat(a, t) * G64).sum(), axes, ang)
        L = np.linalg.norm(axes.astype(np.float64), axis=-1)
        ea = row_max((host(got_a) - ref_a) * L[:, None]) / np.maximum(row_max(ref_a * L[:, None]), 1.0)
        rep.add(name, "grad axis * |axis|", ea, 2e-5 + 4 * U24 * np.abs(ang[:, 0]))
        et = np.abs(host(got_an)[:, 0] - ref_an[:, 0]) / np.maximum(np.abs(ref_an[:, 0]), 1.0)
        rep.add(name, "grad angle", et, 2e-5 + 4 * U24 * np.abs(ang[:, 0]))
    rep.check()
    z = torch.zeros(4, 3, device=cuda_device, requires_grad=True)
    t = torch.full((4, 1), 0.5, device=cuda_device, requires_grad=True)
    out = dx.util.aa_to_rmat(z, t)
    assert torch.isnan(out).all()
    ga, gt = torch.autograd.grad(out.sum(), (z, t))
    torch.cuda.synchronize()
    assert torch.isnan(ga).all() and torch.isnan(gt).all()


# ---------------------------------------------------------------------------------------------
# so3d_scale_bwd_f32
# ---------------------------------------------------------------------------------------------
SCALARS = [1e-4, 0.37, 1.0, 3.0, 100.0, 20291.0]


def test_so3_scale_bwd_strata(dx, cuda_device):
    """Gradient of <G, so3_scale(R, s)> w.r.t. R and s vs fp64 autograd of matrix_exp(s ref_log(R)), for the schedule's
    scalar range (up to 20291, SURVEY A.6), per row and shared.  The gradient w.r.t. R is checked as its tangent part
    vee_adj(R^T Gamma) and its normal part sym(R^T Gamma), which together make up all 9 entries.  Errors are relative to
    each row's natural scale: s |G| for R (or |ref| where the normal entries grow like 1/sin(theta) near pi), |log R| |G|
    for s.  The fp32 rotation vector w = s log R carries 2^-24 |w| absolute error; near pi, log's backward carries
    2^-24/sin(theta) in its tangent part (test_log_bwd_strata), while its normal part is the reference formula's own,
    conditioned like 2^-24/sin^2(theta)."""
    rng = np.random.default_rng(104)
    rep = Report("so3_scale backward (so3d_scale_bwd_f32)")
    n = 1000
    for lo, hi, tag in ((1e-3, 2.8, "theta [1e-3,2.8]"), (2.8, 3.1, "theta [2.8,3.1]"), (3.1, math.pi - 1e-3, "theta [3.1,pi-1e-3]")):
        R = rot_stratum(rng, n, lo, hi)
        G = rng.standard_normal((n, 3, 3)).astype(np.float32)
        G64 = torch.tensor(G, dtype=F64)
        th = angle_of(R)
        amp = pi_amp(th)
        Gn = np.linalg.norm(G.reshape(n, 9).astype(np.float64), axis=-1)
        Rt = np.swapaxes(R.astype(np.float64), -1, -2)
        for sv in SCALARS:
            for shared in (False, True):
                s = np.full(n, sv, np.float32)
                Rd = dev(R, cuda_device).requires_grad_(True)
                sd = (torch.tensor(sv, device=cuda_device) if shared else dev(s, cuda_device)).requires_grad_(True)
                got_r, got_s = torch.autograd.grad((dx.util.so3_scale(Rd, sd) * dev(G, cuda_device)).sum(), (Rd, sd))
                got_r = host(got_r)
                ref_r, ref_s = grad64(lambda r, ss: (ref_scale(r, ss) * G64).sum(), R, s)
                wl = np.float64(sv) * th
                label = f"{tag} s={sv:g}{' shared' if shared else ''}"
                tol = 2e-5 + 8 * U24 * (wl + amp)
                sym = lambda m: (m + np.swapaxes(m, -1, -2)) / 2
                en = row_max(sym(Rt @ got_r) - sym(Rt @ ref_r)) / np.maximum(row_max(ref_r), sv * Gn)
                rep.add(label, "normal R", en, 2e-5 + 8 * U24 * (wl + amp ** 2))
                tref = tangent64(lambda r: (torch.matrix_exp(ref_log(r) * torch.tensor(s, dtype=F64)[:, None, None]) * G64).sum(), R)
                tau = vee_adj(Rt @ got_r)
                rep.add(label, "tangent R", np.linalg.norm(tau - tref, axis=-1) / (sv * Gn), tol)
                gsc = th * Gn
                if shared:
                    # the reduced value against the fp64 sum, within the per-row tolerances summed at their scales
                    rep.add(label, "g_s (sum)", abs(got_s.item() - ref_s.sum()) / gsc.sum(), (tol * gsc).sum() / gsc.sum())
                else:
                    rep.add(label, "g_s", np.abs(host(got_s) - ref_s) / gsc, tol)
    rep.check()


def scale_gs64(R, s, G):
    """fp64 per-row d/ds <G, exp(s hat(phi))> = phi . vee_adj(exp(s hat(phi))^T G), phi = log R (Jr(s phi) phi = phi)."""
    phi = O.log_vec(R.astype(np.float64))
    E = O.exp_vec(phi * np.asarray(s, np.float64)[..., None])
    return (phi * vee_adj(np.swapaxes(E, -1, -2) @ G.astype(np.float64))).sum(-1)


def test_so3_scale_bwd_deep_and_shared_reduction(dx, cuda_device):
    """2^22 + 3 rows: the persistent engine runs many tiles deep, checked on a strided sample against fp64 autograd; and a
    shared scalar's gradient reduced over 2^20 rows equals the fp64 sum of the fp64 per-row values."""
    n = (1 << 22) + 3
    g = torch.Generator(device=cuda_device); g.manual_seed(105)
    R = dx.ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
    G = torch.randn(n, 3, 3, device=cuda_device, generator=g)
    s = torch.rand(n, device=cuda_device, generator=g) * 3
    Rd, sd = R.clone().requires_grad_(True), s.clone().requires_grad_(True)
    got_r, got_s = torch.autograd.grad((dx.util.so3_scale(Rd, sd) * G).sum(), (Rd, sd))
    idx = torch.cat((torch.arange(0, n, 4099, device=cuda_device), torch.arange(n - 70, n, device=cuda_device)))
    Rs, Gs, ss = host(R[idx]).astype(np.float32), host(G[idx]), host(s[idx]).astype(np.float32)
    th = O.rmat_to_aa(Rs.astype(np.float64))[1][:, 0]
    keep = th < 3.0   # near pi: test_so3_scale_bwd_strata
    G64 = torch.tensor(Gs[keep])
    ref_r, ref_s = grad64(lambda r, sc: (ref_scale(r, sc) * G64).sum(), Rs[keep], ss[keep])
    Gn = np.linalg.norm(Gs[keep].reshape(-1, 9), axis=-1)
    er = row_max(host(got_r[idx])[keep] - ref_r) / np.maximum(row_max(ref_r), ss[keep] * Gn)
    es = np.abs(host(got_s[idx])[keep] - ref_s) / (th[keep] * Gn)
    rep = Report("so3_scale backward, 2^22 + 3 rows (strided sample) and a shared scalar over 2^20 rows")
    rep.add(f"{keep.sum()} sampled rows", "ambient R", er, 2e-5 + 8 * U24 * (ss[keep] * th[keep] + pi_amp(th[keep]) ** 2))
    rep.add(f"{keep.sum()} sampled rows", "g_s", es, 2e-5)
    m = 1 << 20
    for sv in (0.37, 3.0):
        s0 = torch.tensor(sv, device=cuda_device, requires_grad=True)
        (g0,) = torch.autograd.grad((dx.util.so3_scale(R[:m], s0) * G[:m]).sum(), s0)
        per = scale_gs64(host(R[:m]), sv, host(G[:m]))
        gsc = angle_of(host(R[:m])) * np.linalg.norm(host(G[:m]).reshape(m, 9), axis=-1)
        rep.add(f"2^20 rows s={sv}", "g_s (sum)", abs(g0.item() - per.sum()) / gsc.sum(), 1e-5)
    rep.check()


# ---------------------------------------------------------------------------------------------
# so3d_igso3_logp_bwd_f32: IsotropicGaussianSO3.log_prob
# ---------------------------------------------------------------------------------------------
def logp_rows(rng, n):
    """eps log-uniform in [6.4e-3, 2]; angles over all of [0, pi]: k = omega/(sqrt(2) eps) <= 4 (where the density lives),
    uniform on [0, pi], and exact identity / pi rows."""
    eps = np.exp(rng.uniform(math.log(6.4e-3), math.log(2.0), n))
    om = np.where(rng.uniform(size=n) < 0.5, np.minimum(eps * math.sqrt(2.0) * rng.uniform(0, 4, n), math.pi), rng.uniform(0, math.pi, n))
    om[:16] = 0.0
    om[16:32] = math.pi
    R = O.rodrigues(unit_axes(rng, n), om).astype(np.float32)
    R[:16] = np.eye(3, dtype=np.float32)
    return R, eps.astype(np.float32)


def dlog_truth(om, eps, L=None):
    """fp64 d log f / d omega: the L-term series, or (L None) the converged density (closed form in the far tail at small
    eps, where the fp64 series cancels)."""
    ft, gt = O.igso3_series(om, eps, L or 2000)
    if L is None:
        small = (eps < 0.4) & (om > 3.0 * eps)
        gt = np.where(small, O.igso3_closed_dlog(om, eps), gt)
    return gt


LOGP_CASES = [  # (mode, L, n, shared eps, eps range; the 3-image closed form holds 1e-5 up to eps = 1)
    ("closed", 2000, 20000, False, (6.4e-3, 1.0)), ("closed", 2000, 20000, True, (6.4e-3, 1.0)), ("auto", 2000, 20000, False, None),
    ("auto", 2000, 3000, True, None), ("series", 2000, 20000, False, None), ("series", 2000, 4096, False, None),
    ("series_adaptive", 2000, 20000, False, None), ("series_pure", 2000, 20000, False, "guard"),
    ("series", 1, 3000, False, (0.75, 2.0)), ("series", 1, 20000, False, (0.75, 2.0)), ("series", 33, 3000, False, (0.75, 2.0)), ("series", 2001, 20000, True, None),
]


@pytest.mark.parametrize("mode,L,n,shared,erange", LOGP_CASES)
def test_log_prob_grad_modes(dx, cuda_device, mode, L, n, shared, erange):
    """Tangent of the log_prob gradient, tau = vee_adj(R^T Gamma), equals gout dlogf axis = gout x score: against the fp64
    score at 1e-5 on the domain where the forward score holds 1e-5 (k <= 4, 1e-4 < omega <= 3), plus, above pi/2 only,
    2^-24/sin(theta) for the axis of an fp32 matrix.  Elsewhere on [0, pi] the score is a cancelling sum of terms of size omega/(2 eps^2), which
    sets the scale.  Identity rows give exactly 0, theta = pi rows a finite gradient, L = 1 (f constant) exactly 0 everywhere.
    n <= 4096 takes the one-warp-per-row series kernel for the forward."""
    rng = np.random.default_rng(zlib.crc32(repr((mode, L, n, shared)).encode()))
    R, eps = logp_rows(rng, n)
    if erange == "guard":
        eps = np.exp(rng.uniform(math.log(6.4e-3), math.log(2.0), n)).astype(np.float32)
        om_cap = np.minimum(4.1 * eps.astype(np.float64), math.pi)
        axis = unit_axes(rng, n)
        R = O.rodrigues(axis, rng.uniform(0, 1, n) * om_cap).astype(np.float32)
    elif erange is not None:
        eps = np.exp(rng.uniform(math.log(erange[0]), math.log(erange[1]), n)).astype(np.float32)
    if shared:
        eps = np.full(n, eps[100], np.float32)
    gout = rng.uniform(-2, 2, n).astype(np.float32)
    ed = torch.tensor(float(eps[0]), device=cuda_device) if shared else dev(eps, cuda_device)
    d = dx.IsotropicGaussianSO3(ed, mode=mode, series_terms=L)
    Rd = dev(R, cuda_device).requires_grad_(True)
    lp = d.log_prob(Rd)
    (got,) = torch.autograd.grad(lp, Rd, dev(gout[:, None], cuda_device))
    got = host(got)
    assert np.isfinite(got).all()
    R64 = R.astype(np.float64)
    axis, ang = O.rmat_to_aa(R64)
    om, e64 = ang[:, 0], eps.astype(np.float64)
    gt = dlog_truth(om, e64, None if (L == 2000 or L == 2001) else L)
    tau = vee_adj(np.swapaxes(R64, -1, -2) @ got)
    tref = (gout.astype(np.float64) * gt)[:, None] * axis
    ident = om == 0
    assert np.array_equal(got[ident], np.zeros_like(got[ident]))
    if L == 1:   # f = 1 (the l = 0 term alone): the gradient is exactly 0
        assert np.array_equal(got, np.zeros_like(got))
        return
    amp = pi_amp(om)
    k = om / (math.sqrt(2.0) * e64)
    core = (k <= 4) & (om > 1e-4) & (om <= 3.0)
    inner = ~ident & (om < math.pi - 1e-6)
    err = np.linalg.norm(tau - tref, axis=-1)
    rep = Report(f"log_prob backward, mode={mode} L={L} n={n}{' shared eps' if shared else ''}")
    rel = err / np.maximum(np.abs(gout * gt), 1e-30)
    rep.add("k<=4, 1e-4<omega<=3", "tangent (rel |ref|)", rel[core], 1e-5 + 8 * U24 * amp[core])
    big = np.abs(gout) * np.maximum.reduce([np.abs(gt), om / (2 * e64 ** 2), np.ones(n)])
    rep.add("(0, pi)", "tangent (rel scale)", (err / big)[inner], 1e-5 + 8 * U24 * amp[inner])
    amb = O.log_prob_ambient_grad(R64, gout.astype(np.float64) * gt)
    rep.add("k<=4, 1e-4<omega<=3", "ambient", (row_max(got - amb) / row_max(amb))[core], 1e-5 + 8 * U24 * amp[core])
    rep.check()


def test_log_prob_grad_errors_and_se3(dx, cuda_device):
    """An eps that requires grad raises (the gradient w.r.t. eps is not implemented) instead of returning a result without
    it; IGSO3xR3.log_prob's rotation gradient is the IGSO(3) one."""
    R, eps = logp_rows(np.random.default_rng(106), 64)
    Rd = dev(R, cuda_device)
    e = dev(eps, cuda_device).requires_grad_(True)
    for rg in (False, True):
        with pytest.raises(NotImplementedError):
            dx.IsotropicGaussianSO3(e).log_prob(Rd.clone().requires_grad_(rg))
    with torch.no_grad():
        assert dx.IsotropicGaussianSO3(e).log_prob(Rd).shape == (64, 1)
    assert dx.IsotropicGaussianSO3(e.detach()).log_prob(Rd).shape == (64, 1)
    # IGSO3xR3: one small case
    U = dx.util
    e0 = dev(eps[:8], cuda_device)
    dist = dx.IGSO3xR3(e0, shift_scale=2.0)
    rot = Rd[:8].clone().requires_grad_(True)
    shift = torch.randn(8, 3, device=cuda_device, requires_grad=True)
    lp = dist.log_prob(U.AffineT(rot, shift))
    g_rot, g_shift = torch.autograd.grad(lp.sum(), (rot, shift))
    (ref_rot,) = torch.autograd.grad(dx.IsotropicGaussianSO3(e0).log_prob(rot).sum() * 3, rot)
    assert torch.allclose(g_rot, ref_rot, rtol=1e-6, atol=0)
    want_shift = -shift.detach() / (e0[:, None] * 2.0) ** 2
    assert torch.allclose(g_shift, want_shift, rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------
# composite util paths with requires_grad
# ---------------------------------------------------------------------------------------------
def rots_with_identity(rng, n, max_angle=3.0):
    R = O.rodrigues(unit_axes(rng, n), rng.uniform(0, max_angle, n)).astype(np.float32)
    R[:8] = np.eye(3, dtype=np.float32)
    # +-90 degree z rotations (0/+-1 entries, A^T A exactly I)
    R[8:12] = np.array([[[0, -1, 0], [1, 0, 0], [0, 0, 1]], [[0, 1, 0], [-1, 0, 0], [0, 0, 1]]] * 2, np.float32)
    return R


def test_util_composite_grads(dx, cuda_device):
    """rmat_to_aa, log_vec, rmat_dist, so3_lerp (w in {0, 0.3, 1}, and A == B), se3_lerp and se3_scale with requires_grad:
    the forward equals the no-grad kernel's within 1e-6 (identity rows included: axis (0,0,1), no NaN), and the gradient
    equals fp64 autograd of the same composition of reference restatements."""
    U = dx.util
    rng = np.random.default_rng(107)
    n = 1000
    A = rots_with_identity(rng, n)
    B = O.rodrigues(unit_axes(rng, n), rng.uniform(0, 3.0, n)).astype(np.float32)
    B = (A.astype(np.float64) @ B.astype(np.float64)).astype(np.float32)
    B[:12] = A[:12]   # A^T B = I on those rows
    G9 = rng.standard_normal((n, 3, 3))
    G3 = rng.standard_normal((n, 3))
    G1 = rng.standard_normal((n, 1))
    rep = Report("util composite paths with requires_grad")

    def run(fn, *xs):
        ts = [dev(x, cuda_device).requires_grad_(True) for x in xs]
        out = fn(*ts)
        return out, ts

    def cmp(name, got, ref, scale_floor=1.0, tol=2e-5):
        got = host(got)
        assert np.isfinite(got).all(), name
        rep.add(name, "grad", row_max(got - ref) / np.maximum(row_max(ref), scale_floor), tol)

    def fwd_same(name, a, b):
        a, b = host(a), host(b)
        assert np.isfinite(a).all(), name
        rep.add(name, "fwd grad == no-grad", np.abs(a - b).max(), 1e-6)

    def ref_aa(r):  # fp64 restatement of rmat_to_aa (util.py:208-219) with the kernel's identity axis
        sv = torch.stack((ref_log(r)[..., 2, 1], -ref_log(r)[..., 2, 0], ref_log(r)[..., 1, 0]), -1)
        ang = sv.norm(dim=-1, keepdim=True)
        nz = ang > 0
        return torch.where(nz, sv / torch.where(nz, ang, torch.ones_like(ang)), sv.new_tensor([0.0, 0.0, 1.0])), ang

    nonid = slice(8, None)   # the fp64 formula is 0/0 at an exact identity; those rows are checked for finiteness
    Ag = A[nonid]
    # rmat_to_aa
    (ax, an), (Ad,) = run(U.rmat_to_aa, A)
    ax0, an0 = U.rmat_to_aa(dev(A, cuda_device))
    fwd_same("rmat_to_aa axis", ax, ax0); fwd_same("rmat_to_aa angle", an, an0)
    assert np.array_equal(host(ax[:8]), np.tile([0.0, 0.0, 1.0], (8, 1)))
    (g,) = torch.autograd.grad((ax * dev(G3, cuda_device)).sum() + (an * dev(G1, cuda_device)).sum(), Ad)
    (ref,) = grad64(lambda r: (ref_aa(r)[0] * torch.tensor(G3[nonid])).sum() + (ref_aa(r)[1] * torch.tensor(G1[nonid])).sum(), Ag)
    cmp("rmat_to_aa", g[nonid], ref)
    # log_vec
    lv, (Ad,) = run(U.log_vec, A)
    fwd_same("log_vec", lv, U.log_vec(dev(A, cuda_device)))
    (g,) = torch.autograd.grad((lv * dev(G3, cuda_device)).sum(), Ad)
    (ref,) = grad64(lambda r: (torch.stack((ref_log(r)[..., 2, 1], -ref_log(r)[..., 2, 0], ref_log(r)[..., 1, 0]), -1) * torch.tensor(G3[nonid])).sum(), Ag)
    cmp("log_vec", g[nonid], ref)
    # rmat_dist (A != B rows only: the Frobenius norm is not differentiable at 0)
    sel = slice(12, None)
    dd, (Ad, Bd) = run(U.rmat_dist, A[sel], B[sel])
    fwd_same("rmat_dist", dd, U.rmat_dist(dev(A[sel], cuda_device), dev(B[sel], cuda_device)))
    ga, gb = torch.autograd.grad((dd * dev(G1[sel, 0], cuda_device)).sum(), (Ad, Bd))
    ra, rb = grad64(lambda a, b: (ref_log(a.transpose(-1, -2) @ b).norm(dim=(-1, -2)) * torch.tensor(G1[sel, 0])).sum(), A[sel], B[sel])
    cmp("rmat_dist dA", ga, ra); cmp("rmat_dist dB", gb, rb)
    # so3_lerp / se3_lerp
    def ref_lerp(a, b, ww):
        axis, ang = ref_aa(a.transpose(-1, -2) @ b)
        return a @ ref_aa_to_rmat(axis, ww * ang)

    for wv in (0.0, 0.3, 1.0):
        w = np.full((n, 1), wv, np.float32)
        out, (Ad, Bd, wd) = run(U.so3_lerp, A, B, w)
        fwd_same(f"so3_lerp w={wv}", out, U.so3_lerp(dev(A, cuda_device), dev(B, cuda_device), dev(w, cuda_device)))
        ga, gb, gw = torch.autograd.grad((out * dev(G9, cuda_device)).sum(), (Ad, Bd, wd))
        for t in (ga, gb, gw):
            assert torch.isfinite(t).all()
        assert torch.all(gw[:12] == 0)   # A == B rows (identity, +-90 degree z rotations): the angle is 0
        ra, rb, rw = grad64(lambda a, b, ww: (ref_lerp(a, b, ww) * torch.tensor(G9[12:])).sum(), A[12:], B[12:], w[12:])
        cmp(f"so3_lerp w={wv} dA", ga[12:], ra); cmp(f"so3_lerp w={wv} dB", gb[12:], rb); cmp(f"so3_lerp w={wv} dw", gw[12:], rw)
    w = np.full((n, 1), 0.3, np.float32)
    shA, shB = rng.standard_normal((n, 3)).astype(np.float32), rng.standard_normal((n, 3)).astype(np.float32)
    Ad, Bd, wd = dev(A, cuda_device).requires_grad_(True), dev(B, cuda_device).requires_grad_(True), dev(w, cuda_device).requires_grad_(True)
    sAd = dev(shA, cuda_device).requires_grad_(True)
    res = U.se3_lerp(U.AffineT(Ad, sAd), U.AffineT(Bd, dev(shB, cuda_device)), wd)
    res0 = U.se3_lerp(U.AffineT(dev(A, cuda_device), dev(shA, cuda_device)), U.AffineT(dev(B, cuda_device), dev(shB, cuda_device)), dev(w, cuda_device))
    fwd_same("se3_lerp rot", res.rot, res0.rot); fwd_same("se3_lerp shift", res.shift, res0.shift)
    ga, gw, gsa = torch.autograd.grad((res.rot * dev(G9, cuda_device)).sum() + (res.shift * dev(G3, cuda_device)).sum(), (Ad, wd, sAd))
    ra, rw, rsa = grad64(lambda a, ww, sa: (ref_lerp(a, torch.tensor(B[12:], dtype=F64), ww) * torch.tensor(G9[12:])).sum()
                         + (torch.lerp(sa, torch.tensor(shB[12:], dtype=F64), ww) * torch.tensor(G3[12:])).sum(), A[12:], w[12:], shA[12:])
    cmp("se3_lerp dA", ga[12:], ra); cmp("se3_lerp dw", gw[12:], rw); cmp("se3_lerp dshift_a", gsa[12:], rsa)
    # se3_scale
    s = rng.uniform(0.1, 3.0, n).astype(np.float32)
    Ad, sd = dev(A, cuda_device).requires_grad_(True), dev(s, cuda_device).requires_grad_(True)
    sh = torch.randn(n, 3, device=cuda_device, requires_grad=True)
    res = U.se3_scale(U.AffineT(Ad, sh), sd)
    ref_nograd = U.se3_scale(U.AffineT(dev(A, cuda_device), sh.detach()), dev(s, cuda_device))
    fwd_same("se3_scale rot", res.rot, ref_nograd.rot); fwd_same("se3_scale shift", res.shift, ref_nograd.shift)
    ga, gs, gsh = torch.autograd.grad((res.rot * dev(G9, cuda_device)).sum() + (res.shift * dev(G3, cuda_device)).sum(), (Ad, sd, sh))
    ra, rs = grad64(lambda a, ss: (ref_scale(a, ss) * torch.tensor(G9[nonid])).sum() + (torch.tensor(host(sh)[nonid]) * ss[:, None] * torch.tensor(G3[nonid])).sum(),
                    Ag, s[nonid])
    cmp("se3_scale dR", ga[nonid], ra); cmp("se3_scale ds", gs[nonid, None], rs[:, None])
    cmp("se3_scale dshift", gsh, G3 * s[:, None].astype(np.float64))
    rep.check()
