"""GPU parity tests: the sm_100a kernels, called through the Python drop-in API (which goes through
the C ABI of libso3d.so), against the fp64 oracle and the golden vectors produced by the reference.

Tolerances follow the north star: density / score / exp / log <= 1e-5 relative (fp32 vs fp64
truth), inverse-CDF angles <= 1e-5 rad given the same uniforms.
"""
import math

import numpy as np
import pytest
import torch

from oracle import so3_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dx(cuda_device):
    import diffusion_extensions_b200 as pkg

    pkg._lib.load()
    return pkg


def dev(a, device):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(device)


def host(t):
    return t.detach().cpu().numpy().astype(np.float64)


def rand_rots(n, seed, max_angle=math.pi):
    rng = np.random.default_rng(seed)
    R, axis, ang = O.random_rotations(n, rng, max_angle)
    return R.astype(np.float32), axis, ang


SIZES = [1, 7, 255, 256, 257, 4099]


# ---------------------------------------------------------------------------------------------
# L0 against golden (reference outputs) and oracle
# ---------------------------------------------------------------------------------------------
def test_l0_against_reference_golden(dx, cuda_device, golden):
    g = golden("util_l0")
    U = dx.util
    d = lambda k: dev(g[k], cuda_device)
    assert np.max(np.abs(host(U.log_rmat(d("Rall"))) - g["log_all"])) < 3e-6
    axis, ang = U.rmat_to_aa(d("R"))
    assert ang.shape == (192, 1)
    assert np.max(np.abs(host(ang) - g["angle"])) < 3e-6
    assert np.max(np.abs(host(axis) - g["axis"])) < 5e-6
    assert np.max(np.abs(host(U.aa_to_rmat(d("axes_in"), d("ang_in"))) - g["aa_rmat"])) < 2e-6
    assert np.max(np.abs(host(U.so3_scale(d("R"), d("scalars"))) - g["scaled"])) < 5e-6
    assert np.max(np.abs(host(U.quat_to_rmat(d("quat"))) - g["quat_rmat"])) < 1e-6
    assert np.max(np.abs(host(U.so3_lerp(d("R"), d("R2"), d("lerp_w"))) - g["lerp"])) < 2e-5
    assert np.max(np.abs(host(U.rmat_dist(d("R"), d("R2"))) - g["dist"])) < 5e-6
    assert np.max(np.abs(host(U.exp_vec(d("vec"))) - g["expvec"])) < 2e-6
    assert np.array_equal(host(U.vec2skew(d("vec"))), g["skew"].astype(np.float64))
    assert np.array_equal(host(U.skew2vec(d("skew"))), g["vee"].astype(np.float64))
    # util.py:500,507-512 known answers
    assert torch.all(U.log_rmat(torch.eye(3, device=cuda_device)[None]) == 0)
    piz = host(U.log_rmat(torch.diag(torch.tensor([-1.0, -1.0, 1.0], device=cuda_device))[None]))
    assert np.allclose(np.abs(piz), np.abs(g["pi_z"]), atol=1e-6)


@pytest.mark.parametrize("n", SIZES)
def test_l0_against_oracle_ragged_sizes(dx, cuda_device, n):
    U = dx.util
    R, _, _ = rand_rots(n, n)
    R2, _, _ = rand_rots(n, n + 1)
    rng = np.random.default_rng(n)
    Rd, R2d = dev(R, cuda_device), dev(R2, cuda_device)
    lv = host(dx.ops.log_vec(Rd))
    ang_t = O.rmat_to_aa(R)[1][:, 0]
    ok = ang_t < 3.1
    assert np.max(np.abs(lv - O.log_vec(R))[ok], initial=0) < 3e-6
    axis, ang = U.rmat_to_aa(Rd)
    back = O.rodrigues(host(axis), host(ang)[:, 0])
    assert np.max(np.abs(back - R)) < 2e-6   # log then exp round trip, valid up to pi
    s = np.exp(rng.uniform(math.log(1e-4), math.log(3.0), n)).astype(np.float32)
    assert np.max(np.abs(host(U.so3_scale(Rd, dev(s, cuda_device))) - O.so3_scale(R, s))) < 3e-6
    assert np.max(np.abs(host(U.so3_scale(Rd, 0.37)) - O.so3_scale(R, np.full(n, np.float32(0.37))))) < 3e-6
    for ta in (False, True):
        for tb in (False, True):
            want = (np.swapaxes(R, -1, -2) if ta else R).astype(np.float64) @ (np.swapaxes(R2, -1, -2) if tb else R2).astype(np.float64)
            assert np.max(np.abs(host(U.compose(Rd, R2d, ta, tb)) - want)) < 1e-6
    one = dev(R2[0], cuda_device)
    assert np.max(np.abs(host(U.compose(one, Rd)) - R2[0].astype(np.float64) @ R.astype(np.float64))) < 1e-6
    assert np.max(np.abs(host(U.compose(Rd, one, trans_b=True)) - R.astype(np.float64) @ R2[0].astype(np.float64).T)) < 1e-6
    q = rng.standard_normal((n, 4)).astype(np.float32)
    assert np.max(np.abs(host(U.quat_to_rmat(dev(q, cuda_device))) - O.quat_to_rmat(q))) < 1e-6
    q2 = host(U.rmat_to_quat(Rd))
    assert np.max(np.abs(O.quat_to_rmat(q2) - R)) < 2e-6 and np.all(q2[:, 0] >= 0)
    w = rng.uniform(0, 1, (n, 1)).astype(np.float32)
    lerp_ok = O.rmat_to_aa(np.swapaxes(R, -1, -2).astype(np.float64) @ R2.astype(np.float64))[1][:, 0] < 3.1
    assert np.max(np.abs(host(U.so3_lerp(Rd, R2d, dev(w, cuda_device))) - O.so3_lerp(R, R2, w))[lerp_ok], initial=0) < 5e-6
    assert np.max(np.abs(host(U.rmat_dist(Rd, R2d)) - O.rmat_dist(R, R2))) < 5e-6


def test_unaligned_views_and_empty(dx, cuda_device):
    """Pointers that are only 4-byte aligned (a row-offset view) take the scalar path; n = 0 is a no-op."""
    U = dx.util
    R, _, _ = rand_rots(1025, 5)
    big = dev(R, cuda_device)
    view = big[1:]  # 36-byte offset: not 16-byte aligned
    assert view.data_ptr() % 16 != 0
    assert np.max(np.abs(host(dx.ops.log_vec(view)) - host(dx.ops.log_vec(view.clone())))) == 0
    assert np.max(np.abs(host(U.so3_scale(view, 0.5)) - host(U.so3_scale(view.clone(), 0.5)))) == 0
    empty = torch.empty(0, 3, 3, device=cuda_device)
    assert U.log_rmat(empty).shape == (0, 3, 3)
    assert U.rmat_to_aa(empty)[1].shape == (0, 1)
    # leading batch dims
    R4 = big[:1024].reshape(4, 16, 16, 3, 3)
    assert U.log_rmat(R4).shape == (4, 16, 16, 3, 3)
    assert torch.equal(U.log_rmat(R4).reshape(-1, 3, 3), U.log_rmat(big[:1024]))


def test_log_edge_cases(dx, cuda_device):
    rng = np.random.default_rng(3)
    ax = rng.standard_normal((64, 3)); ax /= np.linalg.norm(ax, axis=-1, keepdims=True)
    Rpi = O.rodrigues(ax, np.full(64, math.pi)).astype(np.float32)
    Rtiny = O.rodrigues(ax, np.full(64, 1e-5)).astype(np.float32)
    R = np.concatenate([np.eye(3, dtype=np.float32)[None], Rpi, Rtiny])
    axis, ang = dx.util.rmat_to_aa(dev(R, cuda_device))
    axis, ang = host(axis), host(ang)[:, 0]
    assert ang[0] == 0 and np.array_equal(axis[0], [0, 0, 1])          # Q10: no NaN at the identity
    assert np.max(np.abs(ang[1:65] - math.pi)) < 1e-6
    assert np.min(np.abs((axis[1:65] * ax).sum(-1))) > 1 - 1e-6        # Q4: correct axis at exactly pi
    assert np.max(np.abs(ang[65:] - 1e-5)) < 1e-9
    nan_in = torch.full((3, 3, 3), float("nan"), device=cuda_device)
    assert torch.isnan(dx.util.log_rmat(nan_in)).any()                # NaN in -> NaN out, no trap


def test_so3_scale_large_scalars(dx, cuda_device):
    """Schedule scalars reach 20291 (SURVEY A.6); the reference loses orthogonality there (Q5),
    Rodrigues does not.  Accuracy vs fp64 truth degrades only as |s * theta| * 2^-24."""
    R, _, _ = rand_rots(4096, 17, 3.0)
    for s in (100.0, 20291.0):
        out = host(dx.util.so3_scale(dev(R, cuda_device), s))
        orth = np.max(np.abs(out @ np.swapaxes(out, -1, -2) - np.eye(3)))
        assert orth < 2e-6
        th32 = O.rmat_to_aa(R)[1][:, 0].astype(np.float32)
        want = O.rodrigues(O.rmat_to_aa(R)[0], (np.float32(s) * th32).astype(np.float64))  # same fp32 product s*theta
        # the kernel's fp32 theta and the oracle's differ by an ulp or two (2.4e-7 at pi), amplified by s
        assert np.max(np.abs(out - want)) < 2e-6 + 6e-7 * s


# ---------------------------------------------------------------------------------------------
# L1: IGSO(3)
# ---------------------------------------------------------------------------------------------
def eset(n, seed, kmax=4.0):
    rng = np.random.default_rng(seed)
    eps = np.exp(rng.uniform(math.log(6.4e-3), 0.0, n)).astype(np.float32)
    k = rng.uniform(0, kmax, n)
    om = np.minimum(eps * math.sqrt(2.0) * k, 3.0).astype(np.float32)
    axis = rng.standard_normal((n, 3)); axis /= np.linalg.norm(axis, axis=-1, keepdims=True)
    R = O.rodrigues(axis, om.astype(np.float64)).astype(np.float32)
    return R, eps


def truth_from_R(R, eps):
    """fp64 truth evaluated at the angle of the float32 matrix the kernel actually sees."""
    axis, ang = O.rmat_to_aa(R.astype(np.float64))
    om, e64 = ang[:, 0], eps.astype(np.float64)
    ft, gt = O.igso3_series(om, e64)
    small = (e64 < 0.4) & (om > 3.0 * e64)   # far tail at small eps: fp64 series cancels, closed form is exact to 1e-9
    ft = np.where(small, O.igso3_closed(om, e64), ft)
    gt = np.where(small, O.igso3_closed_dlog(om, e64), gt)
    return om, axis, ft, gt


def test_density_against_reference_golden(dx, cuda_device, golden):
    g = golden("igso3")
    om = dev(g["omega"], cuda_device)
    for e, ref in zip(g["eps_list"], g["density"]):
        d = dx.IsotropicGaussianSO3(torch.tensor(float(e), device=cuda_device), mode="closed")
        got = host(d._eps_ft(om))
        # reference: NaN at omega == 0 for eps < 0.167 (Q3) and zeroed beyond 709 eps^2/pi (D5)
        ok = np.isfinite(ref) & (g["omega"] <= 0.99 * 709.0 * float(e) ** 2 / math.pi)
        assert np.max(np.abs(got[ok] - ref[ok]) / np.maximum(ref[ok], 1e-30)) < 1e-5, e
        for mode in ("auto", "series"):
            d2 = dx.IsotropicGaussianSO3(torch.tensor(float(e), device=cuda_device), mode=mode)
            got2 = host(d2._eps_ft(om))
            well = ok & (g["omega"] <= 3.5 * float(e))
            assert np.max(np.abs(got2[well] - ref[well]) / ref[well]) < 1e-5, (e, mode)


def test_log_prob_and_grad_against_reference_golden(dx, cuda_device, golden):
    g = golden("igso3")
    for k, e in enumerate(g["eps_list"]):
        d = dx.IsotropicGaussianSO3(torch.tensor(float(e), device=cuda_device), mode="closed")
        R = dev(g["lp_R"][k], cuda_device).requires_grad_(True)
        lp = d.log_prob(R)
        assert lp.shape == (96, 1)
        ref = g["logp"][k]
        assert np.max(np.abs(host(lp) - ref)) < 2e-5 + 1e-6 * np.max(np.abs(ref))
        (gr,) = torch.autograd.grad(lp.sum(), R)
        refg = g["logp_grad"][k]
        scale = np.max(np.abs(refg), axis=(-1, -2), keepdims=True)
        # autograd through the reference's fp32 log_rmat carries ~1e-3 relative noise at small angles
        assert np.max(np.abs(host(gr) - refg) / scale) < 3e-3, e
        # and tightly against the fp64 ambient gradient (SURVEY A.5)
        R64 = g["lp_R"][k].astype(np.float64)
        gd = O.igso3_closed_dlog(O.rmat_to_aa(R64)[1][:, 0], float(e))
        amb = O.log_prob_ambient_grad(R64, gd)
        assert np.max(np.abs(host(gr) - amb) / np.max(np.abs(amb), axis=(-1, -2), keepdims=True)) < 2e-4


@pytest.mark.parametrize("mode", ["auto", "closed"])
def test_logp_score_eset(dx, cuda_device, mode):
    """North-star gate: density and score <= 1e-5 relative vs the fp64 series on the E-set."""
    n = 1 << 16
    R, eps = eset(n, 11)
    om, axis, ft, gt = truth_from_R(R, eps)
    d = dx.IsotropicGaussianSO3(dev(eps, cuda_device), mode=mode)
    logp, score = d.log_prob_and_score(dev(R, cuda_device))
    logp, score = host(logp)[:, 0], host(score)
    assert np.max(np.abs(np.exp(logp - np.log(ft)) - 1)) < 1e-5
    want = gt[:, None] * axis
    err = np.linalg.norm(score - want, axis=-1) / np.maximum(np.abs(gt), 1e-30)
    # the direction of a rotation by omega is only defined to ~6e-8/omega in fp32: exclude omega < 1e-2
    ok = om > 1e-2
    assert np.max(err[ok]) < 1e-5
    g_kernel = (score * axis).sum(-1)
    assert np.max((np.abs(g_kernel - gt) / np.maximum(np.abs(gt), 1e-30))[om > 1e-4]) < 1e-5


def test_logp_score_series_L2000(dx, cuda_device):
    """The benchmarked kernel (mode "series", L = 2000): density AND score <= 1e-5 relative on the whole E-set
    (k <= 4).  Every row runs its 2000 terms; rows whose alternating sum is ill-conditioned in fp32 (omega > 4.2 eps)
    are replaced by the closed form (csrc/so3d_math.cuh kSeriesGuard).  "series_pure" is the raw fp32 series: 1e-5
    below the guard, growing like ~4 u cond beyond (measured bounds)."""
    n = 1 << 16
    R, eps = eset(n, 13)
    om, axis, ft, gt = truth_from_R(R, eps)
    k = om / (math.sqrt(2.0) * eps)
    d = dx.IsotropicGaussianSO3(dev(eps, cuda_device), mode="series", series_terms=2000)
    logp, score = d.log_prob_and_score(dev(R, cuda_device))
    ef = np.abs(np.exp(host(logp)[:, 0] - np.log(ft)) - 1)
    g_kernel = (host(score) * axis).sum(-1)
    eg = np.abs(g_kernel - gt) / np.maximum(np.abs(gt), 1e-30)
    assert ef.max() < 1e-5 and eg[om > 1e-4].max() < 1e-5
    want = gt[:, None] * axis
    es = np.linalg.norm(host(score) - want, axis=-1) / np.maximum(np.abs(gt), 1e-30)
    assert es[om > 1e-2].max() < 1e-5       # (the direction of a rotation by omega is only defined to ~6e-8/omega in fp32)
    # adaptive truncation is bit-identical (skipped weights are exactly zero)
    d2 = dx.IsotropicGaussianSO3(dev(eps, cuda_device), mode="series_adaptive", series_terms=2000)
    logp2, score2 = d2.log_prob_and_score(dev(R, cuda_device))
    assert torch.equal(logp, logp2) and torch.equal(score, score2)
    # the raw series: identical below the guard, measured growth beyond it
    d3 = dx.IsotropicGaussianSO3(dev(eps, cuda_device), mode="series_pure", series_terms=2000)
    logp3, score3 = d3.log_prob_and_score(dev(R, cuda_device))
    below = torch.as_tensor(om <= 4.19 * eps, device=cuda_device)
    assert torch.equal(logp[below], logp3[below]) and torch.equal(score[below], score3[below])
    ef3 = np.abs(np.exp(host(logp3)[:, 0] - np.log(ft)) - 1)
    eg3 = np.abs((host(score3) * axis).sum(-1) - gt) / np.maximum(np.abs(gt), 1e-30)
    assert ef3[k <= 3.5].max() < 3e-5 and ef3.max() < 2e-4 and eg3[om > 1e-4].max() < 2e-4
    assert ef3.max() > 1e-5                  # the reason the guard exists


def test_logp_score_series_small_batch_warp_split(dx, cuda_device):
    """Small batches of the series evaluator run one WARP per rotation (the L terms split over the lanes, partial results
    combined with warp shuffles): same 1e-5 bound against the fp64 series on the whole E-set, within a few 1e-6 of the
    one-thread-per-rotation kernel (the same rows evaluated inside a large batch), ragged sizes, per-row and shared eps."""
    big_n = 1 << 16
    R, eps = eset(big_n, 29)
    om, axis, ft, gt = truth_from_R(R, eps)
    Rd, ed = dev(R, cuda_device), dev(eps, cuda_device)
    lp_big, sc_big, _ = dx.ops.igso3_logp_score(Rd, ed, mode="series", L=2000)          # one thread per rotation
    for n in (1, 33, 4096, 10000):
        lp, sc, _ = dx.ops.igso3_logp_score(Rd[:n].contiguous(), ed[:n].contiguous(), mode="series", L=2000)   # one warp per rotation
        ef = np.abs(np.exp(host(lp) - np.log(ft[:n])) - 1)
        gk = (host(sc) * axis[:n]).sum(-1)
        eg = np.abs(gk - gt[:n]) / np.maximum(np.abs(gt[:n]), 1e-30)
        assert ef.max() < 1e-5 and eg[om[:n] > 1e-4].max(initial=0.0) < 1e-5, n
        assert np.max(np.abs(np.exp(host(lp) - host(lp_big[:n])) - 1)) < 8e-6, n
    # shared eps, and the raw sum
    e0 = torch.tensor(0.9, device=cuda_device)     # (every E-set angle is inside 4.2 eps for this eps: the raw sum stays positive)
    a, _, _ = dx.ops.igso3_logp_score(Rd[:500].contiguous(), e0, mode="series_pure", L=2000)
    b, _, _ = dx.ops.igso3_logp_score(Rd[:500].contiguous(), e0.expand(500).contiguous(), mode="series_pure", L=2000)
    assert torch.isfinite(a).all() and torch.equal(a, b)


def test_scalar_vs_per_row_eps(dx, cuda_device):
    R, _ = eset(5000, 19)
    Rd = dev(R, cuda_device)
    e = torch.tensor(0.3, device=cuda_device)
    a = dx.IsotropicGaussianSO3(e).log_prob(Rd)
    b = dx.IsotropicGaussianSO3(e.expand(5000).contiguous()).log_prob(Rd)
    assert torch.equal(a, b)


def test_cdf_table_against_reference_golden(dx, cuda_device, golden):
    g = golden("igso3")
    loc, haar, trap_loc = dx.ops.cdf_grid(cuda_device)
    assert np.array_equal(loc.cpu().numpy(), g["grid_loc"]) and np.array_equal(haar.cpu().numpy(), g["grid_haar"])
    d = dx.IsotropicGaussianSO3(dev(g["eps_list"], cuda_device))
    assert d.trap.shape == (999, 5) and d.trap_loc.shape == (999, 1)
    assert np.max(np.abs(d.table.cpu().numpy() - g["trap"])) <= 2.4e-7   # <= 2 ulp at 1.0
    assert np.array_equal(d.trap_loc[:, 0].cpu().numpy(), g["trap_loc"])
    ds = dx.IsotropicGaussianSO3(torch.tensor(0.5, device=cuda_device))
    assert ds.trap.shape == (999, 1)
    # reference quirk D5 at the schedule's smallest eps, and the batched (999, B) constructor
    dq = dx.IsotropicGaussianSO3(torch.tensor(float(g["q_eps"]), device=cuda_device), reference_quirks=True)
    assert np.max(np.abs(dq.table.cpu().numpy()[0] - g["q_trap"])) <= 2.4e-7
    db = dx.IsotropicGaussianSO3(dev(g["b_eps"], cuda_device), reference_quirks=True)
    assert np.max(np.abs(db.trap.cpu().numpy() - g["b_trap"])) <= 2.4e-7
    # the oracle's table from the same grid
    want, _ = O.igso3_cdf_table(g["eps_list"], g["grid_loc"], g["grid_haar"])
    assert np.max(np.abs(d.table.cpu().numpy() - want)) <= 2.4e-7
    # monotone, ends at exactly 1
    tb = d.table.cpu().numpy()
    assert np.all(np.diff(tb, axis=1) >= 0) and np.all(tb[:, -1] == 1.0)


def test_sampler_given_reference_draws(dx, cuda_device, golden):
    """Same (axes, u) as the reference's CPU generator produced -> same rotations (1e-5 rad)."""
    g = golden("igso3")
    for k, e in enumerate(g["eps_list"]):
        d = dx.IsotropicGaussianSO3(torch.tensor(float(e), device=cuda_device))
        R, ang = d.sample((256,), u=dev(g["u_draw"][k], cuda_device), axes=dev(g["axes_draw"][k], cuda_device), return_angle=True)
        assert R.shape == (256, 3, 3)
        ref_ang = O.rmat_to_aa(g["samples"][k])[1][:, 0]
        assert np.max(np.abs(host(ang) - ref_ang)) < 1e-5, e
        assert np.max(np.abs(host(R) - g["samples"][k])) < 5e-6
    # batched eps: row 0 matches the reference, other rows match the corrected oracle (Q1)
    d = dx.IsotropicGaussianSO3(dev(g["b_eps"], cuda_device), reference_quirks=True)
    R, ang = d.sample(u=dev(g["b_u"], cuda_device), axes=dev(g["b_axes"], cuda_device), return_angle=True)
    assert R.shape == (6, 3, 3)
    assert np.max(np.abs(host(R)[0] - g["b_samples"][0])) < 5e-6
    want = O.igso3_angle_from_uniform(g["b_u"], g["b_trap"].T, g["trap_loc"])
    assert np.max(np.abs(host(ang) - want)) < 1e-6
    # mean is applied on the left (distributions.py:50)
    m, _, _ = rand_rots(1, 99)
    dm = dx.IsotropicGaussianSO3(torch.tensor(0.2, device=cuda_device), mean=dev(m[0], cuda_device))
    Rm = dm.sample((256,), u=dev(g["u_draw"][2], cuda_device), axes=dev(g["axes_draw"][2], cuda_device))
    assert np.max(np.abs(host(Rm) - m[0].astype(np.float64) @ g["samples"][2].astype(np.float64))) < 5e-6


def test_sampler_device_rng_statistics(dx, cuda_device):
    """Device Philox path: reproducible under manual_seed, sharding invariant, and distributed as
    IGSO3(eps): angle CDF matches the table (KS), axes uniform on the sphere."""
    n = 1 << 18
    eps = 0.25
    d = dx.IsotropicGaussianSO3(torch.tensor(eps, device=cuda_device))
    dx.manual_seed(7)
    R1, a1 = d.sample((n,), return_angle=True)
    dx.manual_seed(7)
    R2, a2 = d.sample((n,), return_angle=True)
    assert torch.equal(R1, R2)
    R3 = d.sample((n,))
    assert not torch.equal(R1, R3)                      # the stream advances between calls
    # two half-size shards with global row offsets reproduce the full batch
    dx.manual_seed(7)
    Ra = d.sample((n // 2,), row_offset=0)
    dx.ops.rng.offset = 0
    Rb = d.sample((n // 2,), row_offset=n // 2)
    assert torch.equal(torch.cat([Ra, Rb]), R1)
    ang = np.sort(host(a1))
    tb = d.table[0].cpu().numpy().astype(np.float64)
    loc = d.trap_loc[:, 0].cpu().numpy().astype(np.float64)
    cdf_at = np.interp(ang, loc, tb)
    ks = np.max(np.abs(cdf_at - (np.arange(n) + 0.5) / n))
    assert ks < 2.0 / math.sqrt(n)
    axis = host(dx.util.rmat_to_aa(R1)[0])
    assert np.max(np.abs(axis.mean(0))) < 5.0 / math.sqrt(n)
    out = host(R1)
    assert np.max(np.abs(out @ np.swapaxes(out, -1, -2) - np.eye(3))) < 1e-6


# ---------------------------------------------------------------------------------------------
# L2: SO3Diffusion
# ---------------------------------------------------------------------------------------------
def test_schedule_and_state_dict(dx, cuda_device, golden):
    s = golden("schedule")
    p = dx.SO3Diffusion(None)
    sd = p.state_dict()
    assert set(sd.keys()) == set(s.keys())
    for k in s:
        assert np.array_equal(sd[k].numpy(), s[k]), k
    p.load_state_dict({k: torch.tensor(v) for k, v in s.items()})


def test_diffusion_algebra_against_reference_golden(dx, cuda_device, golden):
    g = golden("diffusion")
    p = dx.SO3Diffusion(None).to(cuda_device)
    d = lambda k: dev(g[k], cuda_device)
    t = torch.tensor(g["t"], device=cuda_device)
    x_t = p.q_sample(d("x0"), t, noise=d("noise"))
    assert np.max(np.abs(host(x_t) - g["x_t"])) < 5e-6
    tgt = dx.ops.log_vec(d("noise")) / dev(g["eps_t"], cuda_device)[:, None]
    assert np.max(np.abs(host(tgt) - g["target"]) / np.maximum(np.abs(g["target"]), 1.0)) < 2e-5
    tr = torch.tensor(g["t_rev"], device=cuda_device)
    ok = O.rmat_to_aa(g["x_t"])[1][:, 0] < 3.0  # the reference's fp32 log degrades towards pi
    xr = p.predict_start_from_noise(d("x_t"), tr, d("pred"))
    assert np.max(np.abs(host(xr) - g["x_recon"])[ok]) < 2e-5
    ok2 = ok & (O.rmat_to_aa(g["x_recon"])[1][:, 0] < 3.0)
    pm, pv, plv = p.q_posterior(d("x_recon"), d("x_t"), tr)
    assert np.max(np.abs(host(pm) - g["post_mean"])[ok2]) < 2e-5
    assert np.array_equal(pv.cpu().numpy()[:, 0] if pv.dim() > 1 else pv.cpu().numpy(), g["post_var"])
    p.denoise_fn = lambda x, tt: d("pred")
    mm, _, _ = p.p_mean_variance(d("x_t"), tr)
    assert np.max(np.abs(host(mm) - g["mean_pm"])[ok2]) < 3e-5
    # and tightly against the fp64 oracle everywhere (including near pi and large schedule scalars)
    s = golden("schedule")
    want = O.p_sample_mean(g["x_t"], g["pred"], s["sqrt_recip_alphas_cumprod"][g["t_rev"]], s["sqrt_recipm1_alphas_cumprod"][g["t_rev"]],
                           s["posterior_mean_coef1"][g["t_rev"]], s["posterior_mean_coef2"][g["t_rev"]])
    assert np.max(O.geodesic_angle(host(mm), want)) < 2e-5


def test_p_sample_shared_t_against_reference_golden(dx, cuda_device, golden):
    """Full reverse step at shared t with the reference's own draws injected: the fused kernel's
    mean composed with the sampler given (u, axes) equals the reference's p_sample output."""
    g = golden("diffusion")
    p = dx.SO3Diffusion(None, reference_quirks=True).to(cuda_device)
    d = lambda k: dev(g[k], cuda_device)
    p.denoise_fn = lambda x, tt: d("pred")
    _, post, _ = p.tables()
    for k, step in enumerate(g["ps_steps"]):
        t1 = torch.tensor([int(step)], device=cuda_device)
        mean, _, _ = p.p_mean_variance(d("x_t"), t1)
        if step == 0:
            out = mean
            assert torch.equal(p.p_sample(d("x_t"), t1), mean)          # no noise at t == 0
            assert torch.equal(p.p_sample(d("x_t"), t1.expand(128)), mean)
        else:
            noise = dx.ops.igso3_sample(post, (128,), row=int(step), u=dev(g["ps_u"][k], cuda_device), axes=dev(g["ps_axes"][k], cuda_device))
            out = dx.util.compose(mean, noise)
        ref = g["ps_out"][k]
        ok = (O.rmat_to_aa(g["x_t"])[1][:, 0] < 3.0)
        if step > 600:
            continue  # reference so3_scale(x, 1/sqrt(abar)) is itself off by > 1e-3 there (Q5); oracle test covers it
        assert np.max(O.geodesic_angle(host(out), ref)[ok]) < 5e-5, step


def test_fused_q_sample_consistency(dx, cuda_device):
    """The fused training kernel: x_t = so3_scale(x0, a_t) @ noise with noise ~ IGSO3(eps_t), and
    target = vee(log noise)/eps_t, checked against the oracle applied to the kernel's own noise."""
    n = 20000
    p = dx.SO3Diffusion(None).to(cuda_device)
    x0, _, _ = rand_rots(n, 31)
    rng = np.random.default_rng(5)
    t = rng.integers(0, 1000, n)
    t[:4] = [0, 1, 998, 999]
    dx.manual_seed(3)
    out = p.noise_and_target(dev(x0, cuda_device), torch.tensor(t, device=cuda_device), want_noise=True, want_score=True)
    noise, x_t, target, score = host(out["noise"]), host(out["x_t"]), host(out["target"]), host(out["score"])
    s = O.schedule_buffers(1000)
    want_xt = O.q_sample(x0, s["sqrt_alphas_cumprod"][t], noise)
    assert np.max(O.geodesic_angle(x_t, want_xt)) < 3e-6
    eps = s["sqrt_one_minus_alphas_cumprod"][t].astype(np.float64)
    want_tgt = O.skewvec_target(noise, eps)
    assert np.max(np.abs(target - want_tgt) / np.maximum(np.abs(want_tgt), 1.0)) < 2e-5
    # score of the noise under IGSO3(eps_t): g(omega) * axis
    axis, ang = O.rmat_to_aa(noise)
    ft, gt = O.igso3_series(ang[:, 0], eps)
    well = (ang[:, 0] <= 3.0 * eps) & (ang[:, 0] > 1e-3)
    err = np.linalg.norm(score - gt[:, None] * axis, axis=-1) / np.abs(gt)
    assert np.max(err[well]) < 2e-4   # axis recovered from an fp32 matrix with tiny angle: 6e-8/omega
    # reproducible, and identical without the optional outputs
    dx.manual_seed(3)
    out2 = p.noise_and_target(dev(x0, cuda_device), torch.tensor(t, device=cuda_device))
    assert torch.equal(out2["x_t"], out["x_t"]) and torch.equal(out2["target"], out["target"])
    # angle distribution at a fixed t follows the forward table
    tt = torch.full((1 << 17,), 300, device=cuda_device)
    xx = torch.eye(3, device=cuda_device).expand(1 << 17, 3, 3).contiguous()
    o3 = p.noise_and_target(xx, tt, want_noise=True)
    ang = np.sort(O.rmat_to_aa(host(o3["noise"]))[1][:, 0])
    fwd = p.tables()[0][300].cpu().numpy().astype(np.float64)
    loc = dx.ops.cdf_grid(cuda_device)[2].cpu().numpy().astype(np.float64)
    ks = np.max(np.abs(np.interp(ang, loc, fwd) - (np.arange(ang.size) + 0.5) / ang.size))
    assert ks < 2.5 / math.sqrt(ang.size)


def test_two_row_engine_equals_one_row_for_the_maps(dx, cuda_device, monkeypatch):
    """Every map / backward / sampler op can run on the two-row warp-autonomous engine (one row() call per row, the engine's
    work per 64 rows; the default where it measured faster: log_vec, rmat_dist, closed-form score).  SO3D_ROW_LANES=1 / 2 force
    the one-row / two-row kernel for every op, and both must give the same bits: ragged and single-row sizes, aligned and
    unaligned inputs, per-row and broadcast scalars."""
    ops = dx.ops
    p = dx.SO3Diffusion(None).to(cuda_device)
    fwd, _, _ = p.tables()
    fg, _ = p.guides()
    g = torch.Generator(device=cuda_device); g.manual_seed(81)

    def flat(o):
        if isinstance(o, dict):
            return [v for v in o.values() if v is not None]
        if isinstance(o, (tuple, list)):
            return [v for v in o if v is not None]
        return [o]

    for n in (1, 31, 64, 255, 257, 4099, 256 * 148 * 6 + 13):
        buf = torch.empty(n * 9 + 1, device=cuda_device)
        R = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
        R2 = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
        Ru = buf[1:].view(n, 3, 3); Ru.copy_(R)
        v = torch.randn(n, 3, device=cuda_device, generator=g) * 0.7
        G = torch.randn(n, 3, 3, device=cuda_device, generator=g)
        sc = torch.rand(n, device=cuda_device, generator=g) + 0.5
        q = torch.randn(n, 4, device=cuda_device, generator=g)
        tt = torch.randint(0, 1000, (n,), device=cuda_device, generator=g)
        ang = torch.rand(n, device=cuda_device, generator=g) * 3
        cases = {
            "log_rmat": lambda: ops.log_rmat(R), "log_rmat_unaligned": lambda: ops.log_rmat(Ru), "log_vec": lambda: ops.log_vec(R),
            "rmat_to_aa": lambda: ops.rmat_to_aa(R), "aa_to_rmat": lambda: ops.aa_to_rmat(v, ang), "exp_vec": lambda: ops.exp_vec(v),
            "so3_scale": lambda: ops.so3_scale(R, sc), "so3_scale_bcast": lambda: ops.so3_scale(R, sc[:1]), "quat_to_rmat": lambda: ops.quat_to_rmat(q),
            "rmat_to_quat": lambda: ops.rmat_to_quat(R), "compose": lambda: ops.compose(R, R2), "compose_tn": lambda: ops.compose(R, R2, trans_a=True),
            "compose_shared": lambda: ops.compose(R[:1], R2) if n > 1 else ops.compose(R, R2), "rmat_dist": lambda: ops.rmat_dist(R, R2),
            "so3_lerp": lambda: ops.so3_lerp(R, R2, sc - 0.5), "sample_shared": lambda: ops.igso3_sample(fwd, (n,), row=300, seed=3, rng_offset=1),
            "sample_rows": lambda: ops.igso3_sample(fwd, (n,), row_idx=tt, seed=3, rng_offset=1, guide=fg, want_angle=True),
            "q_sample_given": lambda: ops.q_sample_given(R, tt, p.sqrt_alphas_cumprod, R2),
            "bingham": lambda: ops.bingham_sample(torch.eye(4, device=cuda_device), (n,), seed=2, rng_offset=0, want_rmat=True),
            "se3_p_sample_rows": lambda: ops.se3_p_sample_fused(R, v, v * 0.3, v * 0.1, tt, p.sqrt_recip_alphas_cumprod, p.sqrt_recipm1_alphas_cumprod,
                                                                p.posterior_mean_coef1, p.posterior_mean_coef2,
                                                                (0.5 * p.posterior_log_variance_clipped).exp().contiguous(), 75.0,
                                                                post_cdf=p.tables()[1], seed=6, rng_offset=2, post_guide=p.guides()[1]) if n > 1 else R,
        }
        for name, fn in cases.items():
            res = {}
            for lanes in ("1", "2"):
                monkeypatch.setenv("SO3D_ROW_LANES", lanes)
                res[lanes] = flat(fn())
            assert len(res["1"]) == len(res["2"]) >= 1
            for x, y in zip(res["1"], res["2"]):
                assert torch.equal(x, y), (n, name)
    # backward passes (autograd functions of util): same gradients
    n = 3001
    R = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
    v0 = torch.randn(n, 3, device=cuda_device, generator=g) * 0.7
    sc0 = torch.rand(n, device=cuda_device, generator=g) + 0.5
    w = torch.randn(n, 3, 3, device=cuda_device, generator=g)
    ev = torch.rand(n, device=cuda_device, generator=g) + 0.05
    buf = torch.empty(n * 9 + 1, device=cuda_device)
    grads = {}
    for lanes in ("1", "2"):
        monkeypatch.setenv("SO3D_ROW_LANES", lanes)
        Rr = R.clone().requires_grad_(True); vv = v0.clone().requires_grad_(True); ss = sc0.clone().requires_grad_(True)
        ee = (v0 * 3).clone().requires_grad_(True)
        Ru = buf[1:].view(n, 3, 3); Ru.copy_(R); Ru.requires_grad_(True)   # 4-byte aligned view: the scalar load path
        loss = (dx.util.log_rmat(Rr) * w).sum() + (dx.util.so3_scale(Rr, ss) * w).sum() + (dx.util.aa_to_rmat(vv, ss[:, None]) * w).sum()
        loss = loss + (dx.util.exp_vec(ee) * w).sum() + (dx.util.log_rmat(Ru) * w).sum()
        loss = loss + (dx.IsotropicGaussianSO3(ev, mode="closed").log_prob(Rr) * ss[:, None]).sum()
        loss.backward()
        grads[lanes] = (Rr.grad.clone(), vv.grad.clone(), ss.grad.clone(), ee.grad.clone(), Ru.grad.clone())
        Ru.requires_grad_(False)
    for x, y in zip(grads["1"], grads["2"]):
        assert torch.equal(x, y)


def test_two_row_closed_form_score_equals_one_row(dx, cuda_device, monkeypatch):
    """Closed-form / auto log-density + score: the two-row kernel (default) and the one-row kernel (SO3D_LOGP_LANES=1) give
    the same bits -- ragged sizes, scalar and per-row eps, with and without the dlogf output, unaligned input (writes beyond n:
    compute-sanitizer memcheck over tests/tools/sanitize_target.py)."""
    ops = dx.ops
    g = torch.Generator(device=cuda_device); g.manual_seed(80)
    for n in (1, 33, 64, 255, 256, 257, 5000, 256 * 148 * 8 + 45, 400_003):
        buf = torch.empty(n * 9 + 1, device=cuda_device)
        R = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
        Ru = buf[1:].view(n, 3, 3); Ru.copy_(R)
        eps = torch.exp(torch.empty(n, device=cuda_device).uniform_(-5.0, 0.3, generator=g))
        if n > 40:
            R[3] = torch.eye(3, device=cuda_device)
        for mode in ("closed", "auto"):
            for RR, ee in ((R, eps), (Ru, eps), (R, eps[:1])):
                res = {}
                for lanes in ("1", "2"):
                    monkeypatch.setenv("SO3D_LOGP_LANES", lanes)
                    out = ops.igso3_logp_score(RR, ee, mode=mode, want_dlogf=(mode == "closed"))
                    res[lanes] = out
                a, b = res["1"], res["2"]
                a = a if isinstance(a, (tuple, list)) else (a,)
                b = b if isinstance(b, (tuple, list)) else (b,)
                for x, y in zip(a, b):
                    if x is not None:
                        assert torch.equal(x, y), (n, mode)


def test_two_row_noising_equals_one_row(dx, cuda_device, monkeypatch):
    """Forward noising runs two rows per thread (packed FP32, warp-autonomous two-row engine) by default; the one-row
    kernel (SO3D_QS_LANES=1) must give the same bits: full and ragged tiles, a single row, the score output, a shard
    offset, unaligned (non-TMA) arrays and out-of-range step indices."""
    p = dx.SO3Diffusion(None).to(cuda_device)
    fwd, _, _ = p.tables()
    fg, _ = p.guides()
    ops = dx.ops
    g = torch.Generator(device=cuda_device); g.manual_seed(77)
    for n in (1, 31, 64, 255, 256, 257, 1000, 256 * 148 * 4 + 77, 300_001):
        x0 = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
        t = torch.randint(0, 1000, (n,), device=cuda_device, generator=g)
        if n > 40:
            t[:4] = torch.tensor([0, 999, -5, 1234], device=cuda_device)   # clamped like the one-row kernel
            x0[5] = torch.eye(3, device=cuda_device)
        for kw in ({}, {"want_score": True}, {"want_target": False}, {"row_offset": 12345}):
            res = {}
            for lanes in ("1", "2"):
                monkeypatch.setenv("SO3D_QS_LANES", lanes)
                res[lanes] = ops.q_sample_fused(x0, t, p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd, seed=9, rng_offset=3, guide=fg, **kw)
            for k in res["1"]:
                if res["1"][k] is not None:
                    assert torch.equal(res["1"][k], res["2"][k]), (n, kw, k)
    # unaligned views (4-byte aligned only): both kernels fall back to plain loads / stores
    n = 1000
    buf = torch.empty(n * 9 + 1, device=cuda_device)
    x0u = buf[1:].view(n, 3, 3)
    x0u.copy_(ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g)))
    t = torch.randint(0, 1000, (n,), device=cuda_device, generator=g)
    res = {}
    for lanes in ("1", "2"):
        monkeypatch.setenv("SO3D_QS_LANES", lanes)
        res[lanes] = ops.q_sample_fused(x0u, t, p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd, seed=9, rng_offset=3, guide=fg, want_score=True)
    for k in res["1"]:
        if res["1"][k] is not None:
            assert torch.equal(res["1"][k], res["2"][k]), k
    # without the guide table (full binary search per row)
    for lanes in ("1", "2"):
        monkeypatch.setenv("SO3D_QS_LANES", lanes)
        res[lanes] = ops.q_sample_fused(x0u, t, p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd, seed=9, rng_offset=3)
    assert torch.equal(res["1"]["x_t"], res["2"]["x_t"]) and torch.equal(res["1"]["target"], res["2"]["target"])


def test_two_row_kernels_equal_one_row_at_bench_size(dx, cuda_device, monkeypatch):
    """BASELINE-size check of the cross-kernel identities: 2^24 + 7 rows (ragged last tile, every CTA of the persistent grids
    many tiles deep) through forward noising with the score, the per-row-t reverse step and the closed-form score, one-row
    vs two-row kernels, compared bit for bit."""
    n = (1 << 24) + 7
    p = dx.SO3Diffusion(None).to(cuda_device)
    fwd, post, _ = p.tables()
    fg, pg = p.guides()
    ops = dx.ops
    g = torch.Generator(device=cuda_device); g.manual_seed(82)
    x = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
    t = torch.randint(0, 1000, (n,), device=cuda_device, generator=g)
    pred = torch.randn(n, 3, device=cuda_device, generator=g) * 0.3
    eps = torch.exp(torch.empty(n, device=cuda_device).uniform_(-5.0, 0.2, generator=g))
    sched = (p.sqrt_recip_alphas_cumprod, p.sqrt_recipm1_alphas_cumprod, p.posterior_mean_coef1, p.posterior_mean_coef2)

    def run(lanes):
        for k in ("SO3D_QS_LANES", "SO3D_PS_LANES", "SO3D_LOGP_LANES"):
            monkeypatch.setenv(k, lanes)
        q = ops.q_sample_fused(x, t, p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd, seed=11, rng_offset=5, guide=fg, want_score=True)
        r = ops.p_sample_fused(x, pred, t, *sched, post_cdf=post, seed=11, rng_offset=6, post_guide=pg)
        l, s_, _ = ops.igso3_logp_score(x, eps, mode="auto")
        return [q["x_t"], q["target"], q["score"], r, l, s_]

    a = run("1")
    b = run("2")
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    del a, b


def test_two_row_reverse_step_rows_equals_one_row(dx, cuda_device, monkeypatch):
    """The per-row-t reverse step runs two rows per thread by default; the one-row kernel (SO3D_PS_LANES=1) gives the same
    bits: ragged sizes, rows at t = 0 next to noisy rows, without the guide, without noise, unaligned arrays, a shard offset."""
    p = dx.SO3Diffusion(None).to(cuda_device)
    _, post, _ = p.tables()
    _, pg = p.guides()
    ops = dx.ops
    sched = (p.sqrt_recip_alphas_cumprod, p.sqrt_recipm1_alphas_cumprod, p.posterior_mean_coef1, p.posterior_mean_coef2)
    g = torch.Generator(device=cuda_device); g.manual_seed(78)

    def both(x, pred, t, **kw):
        res = {}
        for lanes in ("1", "2"):
            monkeypatch.setenv("SO3D_PS_LANES", lanes)
            res[lanes] = ops.p_sample_fused(x, pred, t, *sched, seed=5, rng_offset=7, **kw)
        return res["1"], res["2"]

    for n in (1, 33, 64, 255, 256, 257, 4097, 256 * 148 * 4 + 99, 200_003):
        x = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
        pred = torch.randn(n, 3, device=cuda_device, generator=g) * 0.4
        t = torch.randint(0, 1000, (n,), device=cuda_device, generator=g)
        t[::3] = 0                                         # mean-only rows interleaved with noisy ones (both lanes of a thread differ)
        if n > 40:
            t[1:5] = torch.tensor([999, -3, 5000, 1], device=cuda_device)
            x[7] = torch.eye(3, device=cuda_device)
        for kw in ({"post_cdf": post, "post_guide": pg}, {"post_cdf": post}, {}, {"post_cdf": post, "post_guide": pg, "row_offset": 999}):
            a, b = both(x, pred, t, **kw)
            assert torch.equal(a, b), (n, list(kw))
    n = 3000
    buf = torch.empty(n * 9 + 1, device=cuda_device)
    xu = buf[1:].view(n, 3, 3)
    xu.copy_(ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g)))
    pred = torch.randn(n, 3, device=cuda_device, generator=g) * 0.4
    t = torch.randint(0, 1000, (n,), device=cuda_device, generator=g)
    a, b = both(xu, pred, t, post_cdf=post, post_guide=pg)
    assert torch.equal(a, b)


def test_two_row_se3_noising_equals_one_row(dx, cuda_device, monkeypatch):
    """SE(3) noising: the two-row kernel (default) and the one-row kernel (SO3D_SE3_QS_LANES=1) give the same bits."""
    p = dx.SO3Diffusion(None).to(cuda_device)
    fwd, _, _ = p.tables()
    fg, _ = p.guides()
    ops = dx.ops
    g = torch.Generator(device=cuda_device); g.manual_seed(79)
    for n in (1, 40, 256, 300, 256 * 148 * 4 + 5, 150_001):
        rot = ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=g))
        shift = torch.randn(n, 3, device=cuda_device, generator=g) * 10
        t = torch.randint(0, 1000, (n,), device=cuda_device, generator=g)
        for kw in ({"guide": fg}, {}, {"guide": fg, "row_offset": 4242}):
            res = {}
            for lanes in ("1", "2"):
                monkeypatch.setenv("SO3D_SE3_QS_LANES", lanes)
                res[lanes] = ops.se3_q_sample_fused(rot, shift, t, p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd, 75.0, seed=4, rng_offset=2, **kw)
            a, b = res["1"], res["2"]
            a = list(a.values()) if isinstance(a, dict) else list(a)
            b = list(b.values()) if isinstance(b, dict) else list(b)
            assert len(a) == len(b) >= 2
            for u, v in zip(a, b):
                if u is not None:
                    assert torch.equal(u, v), (n, list(kw))


def test_fused_p_sample_against_oracle(dx, cuda_device):
    """Fused reverse step with per-row t vs the oracle mean; the noise factor is recovered as
    mean^T out and must be a rotation whose angle follows the posterior table."""
    n = 8192
    p = dx.SO3Diffusion(None).to(cuda_device)
    s = O.schedule_buffers(1000)
    x, _, _ = rand_rots(n, 41, 3.0)
    rng = np.random.default_rng(6)
    pred = (rng.standard_normal((n, 3)) * 0.5).astype(np.float32)
    t = rng.integers(0, 400, n)
    t[:8] = 0
    p.denoise_fn = lambda xx, tt: dev(pred, cuda_device)
    td = torch.tensor(t, device=cuda_device)
    mean = host(p.p_mean_variance(dev(x, cuda_device), td)[0])
    want = O.p_sample_mean(x, pred, s["sqrt_recip_alphas_cumprod"][t], s["sqrt_recipm1_alphas_cumprod"][t],
                           s["posterior_mean_coef1"][t], s["posterior_mean_coef2"][t])
    assert np.max(O.geodesic_angle(mean, want)) < 1e-5
    dx.manual_seed(11)
    out = host(p.p_sample(dev(x, cuda_device), td))
    assert np.max(np.abs(out[:8] - mean[:8])) == 0           # t == 0 rows: mean only
    nz = np.swapaxes(mean, -1, -2) @ out
    assert np.max(np.abs(nz @ np.swapaxes(nz, -1, -2) - np.eye(3))) < 5e-6
    # shared-t fast path equals the per-row path
    t5 = torch.full((n,), 250, device=cuda_device)
    dx.manual_seed(12)
    a = p.p_sample(dev(x, cuda_device), t5)
    dx.manual_seed(12)
    b = p.p_sample(dev(x, cuda_device), t5[:1])
    assert torch.equal(a, b)
    ang = np.sort(O.rmat_to_aa(np.swapaxes(host(p.p_mean_variance(dev(x, cuda_device), t5)[0]), -1, -2) @ host(a))[1][:, 0])
    post = p.tables()[1][250].cpu().numpy().astype(np.float64)
    loc = dx.ops.cdf_grid(cuda_device)[2].cpu().numpy().astype(np.float64)
    ks = np.max(np.abs(np.interp(ang, loc, post) - (np.arange(n) + 0.5) / n))
    assert ks < 2.5 / math.sqrt(n)


def test_training_step_and_sampling_loop(dx, cuda_device):
    """config[0]: the toy so3_train.py setup (two-point target +-90 deg about z, batch 256) steps
    through SO3Diffusion.forward + backward + Adam, and a short reverse chain stays on SO(3)."""
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(10, 64), torch.nn.SiLU(), torch.nn.Linear(64, 3)).to(cuda_device)

    def denoise(x, t):
        return net(torch.cat([x.flatten(-2), (t.float() / 1000)[:, None]], -1))

    proc = dx.SO3Diffusion(denoise, timesteps=100).to(cuda_device)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    z90 = torch.tensor([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]], device=cuda_device)
    data = torch.stack([z90, z90.t()]).repeat(128, 1, 1)
    losses = []
    for _ in range(30):
        loss = proc(data)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(math.isfinite(v) for v in losses)
    assert np.mean(losses[-5:]) < np.mean(losses[:5])
    x = proc.p_sample_loop((64,))  # batch shape, like bingham_test.py:25
    assert x.shape == (64, 3, 3) and torch.isfinite(x).all()
    xx = host(x)
    assert np.max(np.abs(xx @ np.swapaxes(xx, -1, -2) - np.eye(3))) < 1e-4
    # prevstep loss (diffusion.py:358-365) is differentiable through rmat_dist
    proc2 = dx.SO3Diffusion(lambda x, t: dx.util.exp_vec(denoise(x, t)), timesteps=100, loss_type="prevstep").to(cuda_device)
    l2 = proc2(data)
    l2.backward()
    assert math.isfinite(l2.item())
    with pytest.raises(RuntimeError):
        dx.SO3Diffusion(denoise, timesteps=100, loss_type="bogus").to(cuda_device)(data)


def test_error_behaviour(dx, cuda_device):
    with pytest.raises(RuntimeError):
        dx.util.log_rmat(torch.eye(3)[None])            # CPU tensor: no fallback
    with pytest.raises(TypeError):
        dx.util.log_rmat(torch.eye(3, device=cuda_device, dtype=torch.float64)[None])
    with pytest.raises(ValueError):
        dx.util.log_rmat(torch.zeros(4, 3, device=cuda_device))
    with pytest.raises(RuntimeError):
        dx.ops.igso3_logp_score(torch.eye(3, device=cuda_device)[None], 0.5, mode="series", L=5000)  # C ABI argument error


def test_full_size_properties(dx, cuda_device):
    """BASELINE config[1] size (2^24 rotations): size-independent properties instead of a CPU oracle:
    exp(log R) == R, scale(scale(R, s), 1/s) == R, quaternion round trip, score direction == axis."""
    n = 1 << 24
    torch.manual_seed(1)
    R = dx.util.quat_to_rmat(torch.randn(n, 4, device=cuda_device))
    axis, ang = dx.util.rmat_to_aa(R)
    back = dx.util.aa_to_rmat(axis, ang)
    assert (back - R).abs().max().item() < 3e-6
    far = ang[:, 0] < 3.0
    half = dx.util.so3_scale(dx.util.so3_scale(R, 0.5), 2.0)
    assert (half - R)[far].abs().max().item() < 5e-6
    assert (dx.util.quat_to_rmat(dx.util.rmat_to_quat(R)) - R).abs().max().item() < 3e-6
    eps = torch.full((n,), 0.8, device=cuda_device)
    logp, score = dx.IsotropicGaussianSO3(eps).log_prob_and_score(R)
    g = (score * axis).sum(-1)
    assert torch.isfinite(logp).all() and (g <= 1e-6).all()   # density decreases with the angle
    assert ((score - g[:, None] * axis).norm(dim=-1)).max().item() < 1e-6 * g.abs().max().item()


@pytest.mark.parametrize("n", [1, 255, 257, 1300, 70001])
def test_one_launch_reverse_process_equals_step_launches(dx, cuda_device, n):
    """so3d_p_sample_loop_f32 (all steps in one launch, particles resident in shared memory) is bit-identical to the
    per-step launches of so3d_p_sample_f32 with rng_offset = rng_offset0 + t: without a prediction (pred3 == NULL ==
    zero prediction), with a fixed per-particle prediction, through t == 0 (no noise at the last step), in place, and for
    a shard with a global row offset."""
    p = dx.SO3Diffusion(None).to(cuda_device)
    _, post, t_range = p.tables()
    pg = p.guides()[1]
    sched = (p.sqrt_recip_alphas_cumprod, p.sqrt_recipm1_alphas_cumprod, p.posterior_mean_coef1, p.posterior_mean_coef2)
    x0 = dx.ops.quat_to_rmat(torch.randn(n, 4, device=cuda_device, generator=torch.Generator(device=cuda_device).manual_seed(n)))
    zeros = torch.zeros(n, 3, device=cuda_device)
    pred = torch.randn(n, 3, device=cuda_device) * 0.2
    for t_hi, t_lo, pr, row_off in ((999, 992, None, 0), (6, 0, None, 12345), (500, 495, pred, 7), (3, 0, pred, 0)):
        x = x0
        for t in range(t_hi, t_lo - 1, -1):
            x = dx.ops.p_sample_fused(x, zeros if pr is None else pr, t_range[t:t + 1], *sched, post_cdf=post, seed=91, rng_offset=1000 + t,
                                      row_offset=row_off)
        got = dx.ops.p_sample_loop_fused(x0, pr, t_hi, t_lo, *sched, post, pg, seed=91, rng_offset=1000, row_offset=row_off)
        assert torch.equal(got, x), (t_hi, t_lo, pr is None)
    inplace = x0.clone()
    dx.ops.p_sample_loop_fused(inplace, None, 6, 0, *sched, post, pg, seed=91, rng_offset=1000, row_offset=12345, out=inplace)
    want = dx.ops.p_sample_loop_fused(x0, None, 6, 0, *sched, post, pg, seed=91, rng_offset=1000, row_offset=12345)
    assert torch.equal(inplace, want)
    # the module-level entry point (SO3Diffusion.reverse_process) and argument errors
    if n == 257:
        p.row_offset = 5
        dx.manual_seed(3)
        a = p.reverse_process(x0, t_hi=20)
        dx.manual_seed(3)
        b = p.reverse_process(x0, t_hi=20)
        assert torch.equal(a, b) and torch.isfinite(a).all() and not torch.equal(a, x0)
        with pytest.raises(RuntimeError):
            dx.ops.p_sample_loop_fused(x0, None, 1000, 0, *sched, post, pg, seed=1)      # t_hi out of range: C-ABI argument error
        with pytest.raises(ValueError):
            dx.ops.p_sample_loop_fused(x0, None, 5, 0, *sched, post, None, seed=1)


def test_logp_score_at_2pow28_rows_with_64bit_offsets(dx, cuda_device):
    """BASELINE config[1]'s largest size: 2^28 rotations in ONE launch (9.7 GB of matrices: element offsets beyond 2^31,
    byte offsets beyond 2^33).  The E-set is built on the device (itself a 2^28-row aa_to_rmat launch); a strided sample
    of the results -- including the very last rows -- is compared with the fp64 oracle at the north-star tolerance, for
    the HBM-bound `auto` evaluator and for the L = 2000 series."""
    n = 1 << 28
    free, _ = torch.cuda.mem_get_info(cuda_device)
    if free < 60e9:
        pytest.skip("needs ~30 GB of free device memory")
    g = torch.Generator(device=cuda_device).manual_seed(2028)
    eps = torch.exp(torch.empty(n, device=cuda_device).uniform_(math.log(6.4e-3), 0.0, generator=g))
    k = torch.empty(n, device=cuda_device).uniform_(0.0, 4.0, generator=g)
    omega = torch.clamp(eps * math.sqrt(2.0) * k, max=3.0)
    del k
    axis = torch.randn(n, 3, device=cuda_device, generator=g)
    R = dx.ops.aa_to_rmat(axis, omega)
    del axis, omega
    idx = torch.cat([torch.arange(0, n, n // 8192, device=cuda_device), torch.arange(n - 4096, n, device=cuda_device)])
    Rs, es = R[idx].cpu().numpy(), eps[idx].cpu().numpy()
    om, ax, ft, gt = truth_from_R(Rs, es)
    for mode in ("auto", "series"):
        logp, score, _ = dx.ops.igso3_logp_score(R, eps, mode=mode, L=2000)
        lp, sc = host(logp[idx]), host(score[idx])
        del logp, score
        assert np.max(np.abs(np.exp(lp - np.log(ft)) - 1)) < 1e-5, mode
        gk = (sc * ax).sum(-1)
        assert np.max((np.abs(gk - gt) / np.maximum(np.abs(gt), 1e-30))[om > 1e-4]) < 1e-5, mode
    del R, eps
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# sharding invariance, guide tables, host-buffer pipeline
# ---------------------------------------------------------------------------------------------
def test_shard_invariance_of_random_draws(dx, cuda_device):
    """A batch split into shards (each passing its global row offset, as parallel.attach does) draws the
    same noise as the unsplit batch: results are bit-identical for any number of GPUs (SURVEY 8e)."""
    n = 5000
    p = dx.SO3Diffusion(None).to(cuda_device)
    x0 = dev(rand_rots(n, 51)[0], cuda_device)
    t = torch.randint(0, 1000, (n,), device=cuda_device)
    fwd, post, _ = p.tables()
    fg, pg = p.guides()
    args = (p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd)
    full = dx.ops.q_sample_fused(x0, t, *args, seed=77, rng_offset=5, row_offset=0, guide=fg)
    cuts = [0, 1234, 1234 + 256 * 7, n]
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        part = dx.ops.q_sample_fused(x0[lo:hi], t[lo:hi], *args, seed=77, rng_offset=5, row_offset=lo, guide=fg)
        assert torch.equal(part["x_t"], full["x_t"][lo:hi]) and torch.equal(part["target"], full["target"][lo:hi])
    pred = torch.randn(n, 3, device=cuda_device) * 0.3
    sched = (p.sqrt_recip_alphas_cumprod, p.sqrt_recipm1_alphas_cumprod, p.posterior_mean_coef1, p.posterior_mean_coef2)
    t1 = torch.tensor([500], device=cuda_device)
    fullp = dx.ops.p_sample_fused(x0, pred, t1, *sched, post_cdf=post, seed=78, rng_offset=9, row_offset=0)
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        part = dx.ops.p_sample_fused(x0[lo:hi], pred[lo:hi], t1, *sched, post_cdf=post, seed=78, rng_offset=9, row_offset=lo)
        assert torch.equal(part, fullp[lo:hi])


def test_warp_schedule_ragged_and_unaligned_pieces(dx, cuda_device):
    """The ops on the warp-autonomous engine schedule (per-row table look-ups: forward noising, per-row-t reverse step,
    per-row sampler, SE(3) noising) on pieces of every awkward size and alignment -- 1 row, a partial warp, one row past
    a warp / a tile, pieces starting 4-byte-aligned only (bulk copies impossible: per-warp ld/st fallback) -- must equal
    the corresponding rows of one big aligned launch bit for bit (global-row Philox counters)."""
    n = 3000
    p = dx.SE3Diffusion(None).to(cuda_device)
    x0 = dev(rand_rots(n, 61)[0], cuda_device)
    sh = torch.randn(n, 3, device=cuda_device)
    pred = torch.randn(n, 3, device=cuda_device) * 0.3
    t = torch.randint(0, 1000, (n,), device=cuda_device)
    fwd, post, _ = p.tables()
    fg, pg = p.guides()
    sched = (p.sqrt_recip_alphas_cumprod, p.sqrt_recipm1_alphas_cumprod, p.posterior_mean_coef1, p.posterior_mean_coef2)
    qargs = (p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd)
    full_q = dx.ops.q_sample_fused(x0, t, *qargs, seed=5, rng_offset=3, guide=fg, want_noise=True, want_score=True)
    full_p = dx.ops.p_sample_fused(x0, pred, t, *sched, post_cdf=post, seed=6, rng_offset=4, post_guide=pg)
    full_s = dx.ops.igso3_sample(post, (n,), row_idx=t, seed=7, rng_offset=5, guide=pg)
    full_e = dx.ops.se3_q_sample_fused(x0, sh, t, *qargs, 75.0, seed=8, rng_offset=6, guide=fg)
    pieces = [(0, 1), (1, 32), (3, 36), (64, 64 + 255), (401, 401 + 257), (1001, 1001 + 513), (2000, 3000), (2999, 3000)]
    for lo, hi in pieces:
        q = dx.ops.q_sample_fused(x0[lo:hi], t[lo:hi], *qargs, seed=5, rng_offset=3, row_offset=lo, guide=fg, want_noise=True, want_score=True)
        for k in ("x_t", "target", "noise", "score"):
            assert torch.equal(q[k], full_q[k][lo:hi]), (k, lo, hi)
        pp = dx.ops.p_sample_fused(x0[lo:hi], pred[lo:hi], t[lo:hi], *sched, post_cdf=post, seed=6, rng_offset=4, row_offset=lo, post_guide=pg)
        assert torch.equal(pp, full_p[lo:hi]), ("p_sample", lo, hi)
        ss = dx.ops.igso3_sample(post, (hi - lo,), row_idx=t[lo:hi], seed=7, rng_offset=5, row_offset=lo, guide=pg)
        assert torch.equal(ss, full_s[lo:hi]), ("sample", lo, hi)
        e = dx.ops.se3_q_sample_fused(x0[lo:hi], sh[lo:hi], t[lo:hi], *qargs, 75.0, seed=8, rng_offset=6, row_offset=lo, guide=fg)
        for k in ("rot", "shift", "target_rot", "target_shift"):
            assert torch.equal(e[k], full_e[k][lo:hi]), (k, lo, hi)
    # and the rows are what they should be: x_t = so3_scale(x0, sqrt_ac[t]) @ noise (diffusion.py:344-346)
    ref = O.so3_scale(host(x0), host(p.sqrt_alphas_cumprod)[t.cpu().numpy()]) @ host(full_q["noise"]).astype(np.float64)
    assert np.max(np.abs(host(full_q["x_t"]) - ref)) < 5e-6


def test_projected_so3_diffusion(dx, cuda_device):
    """diffusion.py:377-429 ProjectedSO3Diffusion (row a19): the denoiser sees projection(x) -- here a point cloud rotated
    by x, as in the reference's jigsaw / aircraft scripts -- through the same fused kernels.  With the identity
    projection it IS SO3Diffusion (same seed -> same loss, same reverse step); with a real projection the loss is finite,
    differentiable w.r.t. the denoiser, the reverse loop stays on SO(3); an unknown loss_type raises (Q9)."""
    torch.manual_seed(1)
    pts = torch.randn(3, 5, device=cuda_device)
    net = torch.nn.Sequential(torch.nn.Linear(16, 64), torch.nn.SiLU(), torch.nn.Linear(64, 3)).to(cuda_device)
    net9 = torch.nn.Sequential(torch.nn.Linear(10, 64), torch.nn.SiLU(), torch.nn.Linear(64, 3)).to(cuda_device)

    def denoise_cloud(cloud, t):                     # cloud: (B, 3, 5) = x @ pts
        return net(torch.cat([cloud.flatten(-2), (t.float() / 100)[:, None]], -1))

    def denoise_rot(x, t):
        return net9(torch.cat([x.flatten(-2), (t.float() / 100)[:, None]], -1))

    x0 = dev(rand_rots(512, 81)[0], cuda_device)
    plain = dx.SO3Diffusion(denoise_rot, timesteps=100).to(cuda_device)
    proj_id = dx.ProjectedSO3Diffusion(denoise_rot, timesteps=100).to(cuda_device)
    assert set(proj_id.state_dict()) == set(plain.state_dict()) | {"identity"}          # diffusion.py:380
    for seed in (3, 4):
        torch.manual_seed(seed); dx.ops.manual_seed(seed)
        la = plain(x0)
        torch.manual_seed(seed); dx.ops.manual_seed(seed)
        lb = proj_id(x0, lambda x: x)
        assert torch.equal(la, lb)
    t = torch.full((512,), 37, device=cuda_device)
    dx.ops.manual_seed(9)
    sa = plain.p_sample(x0, t)
    dx.ops.manual_seed(9)
    proj_id.projection = lambda x: x
    sb = proj_id.p_sample(x0, t)
    assert torch.equal(sa, sb)
    proc = dx.ProjectedSO3Diffusion(denoise_cloud, timesteps=100).to(cuda_device)
    loss = proc(x0, lambda x: x @ pts)
    loss.backward()
    assert math.isfinite(loss.item()) and all(p.grad is not None and torch.isfinite(p.grad).all() for p in net.parameters())
    xs = proc.p_sample_loop((64,), lambda x: x @ pts)
    xx = host(xs)
    assert xs.shape == (64, 3, 3) and np.max(np.abs(xx @ np.swapaxes(xx, -1, -2) - np.eye(3))) < 1e-4
    assert np.max(np.abs(np.linalg.det(xx) - 1)) < 1e-4
    bad = dx.ProjectedSO3Diffusion(denoise_cloud, timesteps=100, loss_type="l1").to(cuda_device)
    with pytest.raises(RuntimeError):
        bad(x0, lambda x: x @ pts)


def test_device_seed_and_graphed_train_step(dx, cuda_device):
    """Forward noising with the Philox seed in device memory: (1) equal to the by-value launch at the same seed, bit for
    bit; (2) captured in a CUDA graph it follows the seed tensor (replays differ, and each equals the by-value launch at
    that seed); (3) `make_graphed_train_step` trains the toy model of so3_train.py (loss falls, fresh noise per replay)."""
    n = 3001
    p = dx.SO3Diffusion(None).to(cuda_device)
    x0 = dev(rand_rots(n, 71)[0], cuda_device)
    t = torch.randint(0, 1000, (n,), device=cuda_device)
    fwd, _, _ = p.tables()
    fg, _ = p.guides()
    args = (p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, fwd)
    S = 0x1234_5678_9ABC_DEF
    seed_t = torch.full((1,), S, dtype=torch.int64, device=cuda_device)
    a = dx.ops.q_sample_fused(x0, t, *args, seed=seed_t, rng_offset=4, row_offset=17, guide=fg)
    b = dx.ops.q_sample_fused(x0, t, *args, seed=S, rng_offset=4, row_offset=17, guide=fg)
    assert torch.equal(a["x_t"], b["x_t"]) and torch.equal(a["target"], b["target"])
    # captured: bump the seed on the device, launch
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        dx.ops.q_sample_fused(x0, t, *args, seed=seed_t, rng_offset=0, guide=fg)
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        seed_t.add_(1)
        out = dx.ops.q_sample_fused(x0, t, *args, seed=seed_t, rng_offset=0, guide=fg)
    for k in (1, 2):
        g.replay()
        ref = dx.ops.q_sample_fused(x0, t, *args, seed=S + k, rng_offset=0, guide=fg)
        assert torch.equal(out["x_t"], ref["x_t"]) and torch.equal(out["target"], ref["target"])
    # the reference's toy problem (so3_train.py:65-76): two-point target, RotPredict, Adam -- as one graph per step
    torch.manual_seed(0)
    net = dx.RotPredict(out_type="skewvec").to(cuda_device)
    proc = dx.SO3Diffusion(net).to(cuda_device)
    opt = torch.optim.Adam(net.parameters(), lr=3e-3, capturable=True)
    z90 = torch.tensor([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]], device=cuda_device)
    batch = torch.stack([z90, z90.T]).repeat(128, 1, 1)                      # so3_train.py:65-68, batch 256
    step = proc.make_graphed_train_step(opt, batch)
    losses = torch.stack([step(batch).detach().clone() for _ in range(400)]).cpu()
    assert torch.isfinite(losses).all()
    assert len(set(losses[:20].tolist())) == 20                              # fresh t and noise on every replay
    assert losses[-50:].mean() < 0.8 * losses[:50].mean()                    # and it learns
    assert proc._device_seed.item() > 400


def test_guide_table_lookup_is_exact(dx, cuda_device):
    """The guided inverse-CDF search returns exactly the index of the full search: sampling with and
    without the guide table gives bit-identical rotations, for per-row table rows and for the shared row."""
    p = dx.SO3Diffusion(None).to(cuda_device)
    fwd, post, _ = p.tables()
    fg, pg = p.guides()
    g = fg.cpu().numpy()                                   # (T, 2051, 4) int32 records
    trap = fwd.cpu().numpy()
    # the range [a_k, b_k] of u each record serves (include/so3d.h): u < 2^-13 | 64 per octave up to 1/8 | 1/1024 steps on
    # [1/8, 7/8] | the mirror image in 1 - u, counted down from 1
    log_edges = np.concatenate([(np.float32(2.0) ** -o) * (1 + np.arange(64, dtype=np.float32) / 64) for o in range(13, 3, -1)]
                               + [np.float32([0.125])]).astype(np.float32)
    lower_a = np.concatenate([np.float32([0.0]), log_edges[:-1]]); lower_b = log_edges
    mid = np.arange(128, 898, dtype=np.float32) / np.float32(1024)
    a_k = np.concatenate([lower_a, mid[:-1], (np.float32(1) - lower_b).astype(np.float32)])
    b_k = np.concatenate([lower_b, mid[1:], (np.float32(1) - lower_a).astype(np.float32)])
    assert a_k.shape[0] == g.shape[1] == 2051 and np.all(a_k < b_k)
    for row in (0, 17, 500, 999):
        lo = np.searchsorted(trap[row], a_k, side="right")
        hi = np.searchsorted(trap[row], b_k, side="right")
        lohi = g[row, :, 0].astype(np.int64) & 0xFFFFFFFF
        assert np.array_equal(lohi & 0xFFFF, lo) and np.array_equal(lohi >> 16, hi)
        vals = g[row, :, 1:].view(np.float32)
        for j, off in enumerate((-1, 0, 1)):
            assert np.array_equal(vals[:, j], trap[row][np.clip(lo + off, 0, 998)])
    n = 1 << 16
    rows = torch.randint(0, 1000, (n,), device=cuda_device)
    u = torch.rand(n, device=cuda_device)
    u[:4] = torch.tensor([0.0, 1.0 - 2 ** -24, 0.5, 2 ** -24])
    u[4:8192] = u[4:8192] * 2 ** -10                      # the float-format buckets of the lower tail ...
    u[8192:16384] = 1 - u[8192:16384] * 2 ** -10          # ... and of the upper one
    u[16384:16390] = torch.tensor([0.125, 0.875, 2 ** -13, 1 - 2 ** -13, 0.125 - 2 ** -27, 0.875 + 2 ** -24])
    a = dx.ops.igso3_sample(post, (n,), row_idx=rows, u=u, seed=1, rng_offset=0, want_angle=True)
    b = dx.ops.igso3_sample(post, (n,), row_idx=rows, u=u, seed=1, rng_offset=0, want_angle=True, guide=pg)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # shared-row path (guide built in shared memory) against the per-row path pointed at the same row
    c = dx.ops.igso3_sample(post, (n,), row=321, u=u, seed=1, rng_offset=0, want_angle=True)
    d = dx.ops.igso3_sample(post, (n,), row_idx=torch.full((n,), 321, device=cuda_device), u=u, seed=1, rng_offset=0, want_angle=True)
    assert torch.equal(c[1], d[1]) and torch.equal(c[0], d[0])


def test_host_score_pipeline(dx, cuda_device):
    """ops.HostScorePipeline (pinned host in -> host out, H2D / kernel / D2H overlapped) returns exactly
    what the device-resident call returns, for ragged sizes and for repeated runs on the same staging ring."""
    for n, chunk in ((100_003, 1 << 14), (1 << 15, 1 << 15), (5, 1 << 10)):
        R, eps = eset(n, 61)
        hR = torch.from_numpy(R).pin_memory()
        heps = torch.from_numpy(eps).pin_memory()
        hl = torch.empty(n).pin_memory()
        hs = torch.empty(n, 3).pin_memory()
        pipe = dx.ops.HostScorePipeline(cuda_device, chunk_rows=chunk, depth=3)
        d = dx.IsotropicGaussianSO3(dev(eps, cuda_device), mode="auto")
        logp, score = d.log_prob_and_score(dev(R, cuda_device))
        for _ in range(2):
            hl.zero_(); hs.zero_()
            pipe.run(hR, heps, hl, hs, mode="auto")
            assert torch.equal(hl, logp[:, 0].cpu()) and torch.equal(hs, score.cpu())
        l2, s2 = d.log_prob_and_score_host(hR, chunk_rows=chunk)
        assert torch.equal(l2, logp.cpu()) and torch.equal(s2, score.cpu())
        # streamed batches: two different batches back to back without joining the streams in between (the second
        # batch's uploads overlap the first one's drain; slots are guarded by events that persist across calls)
        R2, eps2 = eset(n, 62)
        hR2, heps2 = torch.from_numpy(R2).pin_memory(), torch.from_numpy(eps2).pin_memory()
        hl2, hs2 = torch.empty(n).pin_memory(), torch.empty(n, 3).pin_memory()
        logp2, score2 = dx.IsotropicGaussianSO3(dev(eps2, cuda_device), mode="auto").log_prob_and_score(dev(R2, cuda_device))
        hl.zero_(); hs.zero_()
        pipe.run(hR, heps, hl, hs, mode="auto", wait=False, join=False)
        pipe.run(hR2, heps2, hl2, hs2, mode="auto", wait=False, join=False)
        pipe.finish(wait=True)
        assert torch.equal(hl, logp[:, 0].cpu()) and torch.equal(hs, score.cpu())
        assert torch.equal(hl2, logp2[:, 0].cpu()) and torch.equal(hs2, score2.cpu())


# ---------------------------------------------------------------------------------------------
# behaviour around the kernels (round-1 advisor findings)
# ---------------------------------------------------------------------------------------------
def test_random_stream_follows_torch_seeding(dx, cuda_device):
    """Without dx.manual_seed the sampling kernels follow torch's CUDA generator: torch.manual_seed(s) restarts the stream
    even when s is the SAME seed as before (the usual way to reproduce a run), consecutive launches differ, and torch's own
    random ops in between shift the stream deterministically.  dx.manual_seed(s) selects the explicit stream instead."""
    p = dx.SO3Diffusion(None).to(cuda_device)
    x0 = dev(rand_rots(3000, 91)[0], cuda_device)
    t = torch.randint(0, 1000, (3000,), device=cuda_device)
    dx.ops.rng._explicit = False                      # (earlier tests of this module seeded the explicit stream)
    torch.manual_seed(5)
    a1 = p.q_sample(x0, t)
    a2 = p.q_sample(x0, t)
    torch.manual_seed(5)                              # same seed again
    b1 = p.q_sample(x0, t)
    b2 = p.q_sample(x0, t)
    assert torch.equal(a1, b1) and torch.equal(a2, b2) and not torch.equal(a1, a2)
    torch.manual_seed(5)
    torch.rand(7, device=cuda_device)                 # a torch op consumes part of the stream first
    c1 = p.q_sample(x0, t)
    torch.manual_seed(5)
    torch.rand(7, device=cuda_device)
    c2 = p.q_sample(x0, t)
    assert torch.equal(c1, c2) and not torch.equal(c1, a1)
    torch.manual_seed(6)
    assert not torch.equal(p.q_sample(x0, t), a1)
    dx.manual_seed(5)
    e1 = p.q_sample(x0, t)
    dx.manual_seed(5)
    e2 = p.q_sample(x0, t)
    assert torch.equal(e1, e2)


def test_tables_follow_the_schedule_buffers(dx, cuda_device):
    """The cached CDF tables belong to the schedule buffers they were built from: loading a state dict with other betas
    (same T) or editing the buffers in place rebuilds them on the next call -- noise is never drawn from stale tables."""
    p = dx.SO3Diffusion(None, timesteps=50).to(cuda_device)
    fwd0 = p.tables()[0].clone()
    assert p.tables()[0].data_ptr() == p.tables()[0].data_ptr()          # cached while nothing changes
    other = dx.SO3Diffusion(None, timesteps=50, betas=np.linspace(1e-4, 0.05, 50)).to(cuda_device)
    p.load_state_dict(other.state_dict())
    fwd1 = p.tables()[0]
    assert not torch.equal(fwd0, fwd1) and torch.equal(fwd1, other.tables()[0])
    g1 = p.guides()[0]
    assert torch.equal(g1, other.guides()[0])
    p.sqrt_one_minus_alphas_cumprod.mul_(0.5)                             # in-place edit
    assert not torch.equal(p.tables()[0], fwd1)
    s = dx.SE3Diffusion(None, timesteps=50).to(cuda_device)
    sig0 = s._sigma().clone()
    s.posterior_log_variance_clipped.add_(1.0)
    assert torch.allclose(s._sigma(), sig0 * math.exp(0.5))


def test_graph_cache_keys_and_batched_mean_sample(dx, cuda_device):
    """(a) p_sample_loop(cuda_graph=True) of a Projected* process is keyed on the projection closure: a second projection
    with the same batch shape captures its own graph instead of replaying the first one (aircraft_test.py:73 sets a
    projection per item).  (b) IsotropicGaussianSO3 / IGSO3xR3 with a scalar eps and a batched mean broadcast the mean
    against the noise like the reference (diffusion.py:482)."""
    torch.manual_seed(2)
    net = torch.nn.Sequential(torch.nn.Linear(10, 32), torch.nn.SiLU(), torch.nn.Linear(32, 3)).to(cuda_device)
    calls = []

    def denoise(x, t):
        return net(torch.cat([x.flatten(-2), (t.float() / 20)[:, None]], -1))

    proc = dx.ProjectedSO3Diffusion(denoise, timesteps=20).to(cuda_device)
    Ra = dev(rand_rots(1, 5)[0], cuda_device)[0]
    Rb = dev(rand_rots(1, 6)[0], cuda_device)[0]
    proj_a = lambda x: (calls.append("a"), x @ Ra)[1]
    proj_b = lambda x: (calls.append("b"), x @ Rb)[1]
    dx.manual_seed(1)
    proc.p_sample_loop((64,), proj_a, cuda_graph=True)
    n_a = calls.count("a")
    dx.manual_seed(1)
    proc.p_sample_loop((64,), proj_b, cuda_graph=True)
    assert calls.count("b") > 0 and len(proc._loop_graphs) == 2           # captured again with the new projection
    calls.clear()
    proc.p_sample_loop((64,), proj_a, cuda_graph=True)                    # replay: the closure is not called again
    assert calls == [] and n_a > 0
    # (b)
    B = 37
    mean = dev(rand_rots(B, 7)[0], cuda_device)
    d = dx.IsotropicGaussianSO3(torch.tensor(0.2, device=cuda_device), mean=mean)
    smp = d.sample()
    assert smp.shape == (B, 3, 3)
    rel = host(mean.transpose(-1, -2) @ smp)
    assert np.max(np.abs(rel @ np.swapaxes(rel, -1, -2) - np.eye(3))) < 1e-5
    from diffusion_extensions_b200.distributions import IGSO3xR3
    from diffusion_extensions_b200.util import AffineT
    pm = AffineT(mean, torch.randn(B, 3, device=cuda_device))
    s3 = IGSO3xR3(torch.tensor(0.3, device=cuda_device), mean=pm, shift_scale=75.0).sample()
    assert s3.rot.shape == (B, 3, 3) and s3.shift.shape == (B, 3)
    assert hasattr(pm, "clone") and torch.equal(pm.clone().rot, pm.rot)
