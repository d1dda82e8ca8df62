"""GPU tier: the kernels that draw random numbers, draw by draw, against the independent restatement of tests/draws_ref.py.

Every draw is a fixed function of (seed, row_offset + row, rng_offset, t) (include/so3d.h): numpy Philox4x32-10, the device
conversion of the uniforms, the exact index of the inverse-CDF lookup in table row t, and fp64 from there on.  Every schedule
step t in [0, T) gets PER_T rows of its own, shuffled so that t varies within a warp, for several (seed, rng_offset,
row_offset) streams, rows crossing 2^32 and above 2^40, a ragged n and an input view that is only 4-byte aligned.  Errors
are reported per kernel and per band of t (strata.Report, printed with -s).

Tolerances (units of U24 = 2^-24):
  AXIS_TOL, per component of the drawn axis: MUFU sin / cos of the azimuth (2^-20.9 absolute, so3d_math.cuh sincos_draw),
    the azimuth's fp32 constants and FMA (6.4 U24), MUFU.RSQ and the roundings of r = sqrt(4 ua (1 - ua)) (6 U24), the
    product r cos (1 U24): 2^-20.9 + 14 U24.
  angle: the restated fp32 lookup to 1 ulp (the device contracts the lerp into an FMA).
  a drawn rotation Rodrigues(axis, angle), geodesic: exp is 1-Lipschitz on SO(3), so |d angle| + angle |d axis| plus
    8 U24 for the fp32 quaternion and matrix.
  the rest reuses the forms of test_gpu_fwd_strata.py (so3_scale, step_tolerance) and test_gpu_grad.py (the score).

Each check also recomputes the restated draws from table row t - 1 and t + 1 (and eps of t +- 1 for the target) and asserts
that almost all rows then fail its tolerance: the bounds tell neighbouring schedule steps apart.
"""
import math

import numpy as np
import pytest
import torch

from oracle import so3_oracle as O
from tests import draws_ref as D
from tests.strata import U24, Report, check_step, polar, unit_axes

pytestmark = pytest.mark.gpu

PER_T = 64
EXTRA = 37                                            # n = T * PER_T + EXTRA: ragged
EDGES = [0, 1, 10, 100, 500, 900, 990, 1000]
BANDS = [f"t in [{a},{b})" for a, b in zip(EDGES, EDGES[1:])]
STREAMS = [(0x1234_5678_9ABC_DEF0, 3, 0),             # (seed, rng_offset, row_offset)
           (2**64 - 1, 2**40 + 1, 2**32 - 20_000),    # global rows cross 2^32
           (77, 2**62 + 5, 2**40 + 123)]              # rows above 2^40
MUFU = 2.0 ** -20.9
AXIS_TOL = MUFU + 14 * U24
AXIS_TOL2 = math.sqrt(3.0) * AXIS_TOL                 # Euclidean norm of the axis error
NEIGHBOUR_FAIL = 0.97                                 # fraction of rows a neighbouring step's draws must fail


def angle_tol(ang):
    return D.ulp32(ang)


def rot_geo_tol(ang):
    ang = np.asarray(ang, np.float64)
    return D.ulp32(ang) + ang * AXIS_TOL2 + 8 * U24


@pytest.fixture(scope="module")
def S(cuda_device):
    import diffusion_extensions_b200 as dx

    p = dx.SO3Diffusion(None).to(cuda_device)
    fwd, post, _ = p.tables()
    fg, pg = p.guides()
    sigma = (0.5 * p.posterior_log_variance_clipped).exp()           # what the posterior table was built from
    h = lambda x: x.detach().cpu().numpy()
    grid, haar, trap_loc = (h(x) for x in dx.ops.cdf_grid(cuda_device))  # the reference's fp32 grid, as torch computes it
    return dict(dx=dx, p=p, fwd=fwd, post=post, fg=fg, pg=pg, sigma=sigma, fwd_h=h(fwd), post_h=h(post), fg_h=h(fg),
                pg_h=h(pg), eps32=h(p.sqrt_one_minus_alphas_cumprod), sig32=h(sigma), sc32=h(p.sqrt_alphas_cumprod),
                sched=[h(getattr(p, k)).astype(np.float64) for k in ("sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod",
                                                                     "posterior_mean_coef1", "posterior_mean_coef2")],
                grid=grid, haar=haar, loc=trap_loc, T=p.num_timesteps)


def layout(seed, T):
    """Step index per row: PER_T rows of every t and EXTRA more, shuffled."""
    rng = np.random.default_rng(seed)
    t = np.concatenate([np.repeat(np.arange(T), PER_T), rng.integers(0, T, EXTRA)])
    rng.shuffle(t)
    return t


def band_of(t):
    return np.searchsorted(np.asarray(EDGES), t, side="right") - 1


def per_band(rep, t, what, err, tol):
    b = band_of(t)
    tol = np.broadcast_to(tol, np.shape(err))
    for i, name in enumerate(BANDS):
        m = b == i
        if m.any():
            rep.add(name, what, err[m], tol[m])


def neighbours(rep, t, T, what, ratio_fn, rows=True):
    """ratio_fn(t') -> err/tol of the kernel's output against the draws restated at step t' instead of t: it must exceed 1
    on at least NEIGHBOUR_FAIL of the rows (of `rows`) that have that neighbour."""
    for d in (-1, 1):
        ok = (t + d >= 0) & (t + d < T) & rows
        r = ratio_fn(np.clip(t + d, 0, T - 1))
        frac = float(np.mean(~(r[ok] <= 1.0)))
        rep.add("t +- 1", f"{what} t{d:+d}: 1 - fail", np.array([1.0 - frac]), 1.0 - NEIGHBOUR_FAIL)


def dev(a, device):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(device)


def host(x):
    return x.detach().cpu().numpy().astype(np.float64)


def geo(a, b):
    return O.geodesic_angle(a, b)


def global_rows(row_offset, n):
    return np.uint64(row_offset) + np.arange(n, dtype=np.uint64)


def rotations(rng, n, max_angle=3.1):
    return O.rodrigues(unit_axes(rng, n), rng.uniform(0, max_angle, n)).astype(np.float32)


def misaligned(x):
    """The same values in a view whose data pointer is 4 bytes past a 16-byte boundary."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(x.shape)
    v.copy_(x)
    assert v.data_ptr() % 16 != 0
    return v


# ---------------------------------------------------------------------------------------------
# a. the CDF tables and their guide records
# ---------------------------------------------------------------------------------------------
def guide_edges():
    """[a_k, b_k], the range of u record k serves (include/so3d.h so3d_igso3_cdf_guide)."""
    log_edges = np.concatenate([(np.float32(2.0) ** -o) * (1 + np.arange(64, dtype=np.float32) / 64) for o in range(13, 3, -1)]
                               + [np.float32([0.125])]).astype(np.float32)
    lower_a = np.concatenate([np.float32([0.0]), log_edges[:-1]])
    mid = np.arange(128, 898, dtype=np.float32) / np.float32(1024)
    a_k = np.concatenate([lower_a, mid[:-1], (np.float32(1) - log_edges).astype(np.float32)])
    b_k = np.concatenate([log_edges, mid[1:], (np.float32(1) - lower_a).astype(np.float32)])
    return a_k, b_k


def test_tables_and_guides_every_row(S):
    """Both tables against the fp64-density oracle at the fp32 schedule values, every row, within the 2.4e-7 (2 ulp at 1) of
    the golden checks; finite rows non-decreasing and ending at exactly 1.  The posterior row 0 has sigma_0 = 1e-10
    (posterior variance clipped at 1e-20): every fp32 density value of the grid is 0 there (its first angle, 3.1e-9 rad, is
    31 sigma out), so the row is 0/0 = NaN in every entry, on the device as in the oracle; the reverse step never reads it
    (t = 0 returns the mean).  Every record of both guides equals the record rebuilt from the device table by searchsorted."""
    rep = Report("CDF tables and guides")
    a_k, b_k = guide_edges()
    for name, tab, g, e in (("forward", S["fwd_h"], S["fg_h"], S["eps32"]), ("posterior", S["post_h"], S["pg_h"], S["sig32"])):
        with np.errstate(invalid="ignore"):
            want, _ = O.igso3_cdf_table(e, S["grid"], S["haar"])
        nan_rows = np.isnan(want).all(1)
        assert np.array_equal(np.isnan(tab), np.isnan(want)), name
        fin = ~nan_rows
        assert np.isfinite(tab[fin]).all()
        if name == "posterior":
            assert nan_rows.tolist() == [True] + [False] * (S["T"] - 1) and abs(float(e[0]) - 1e-10) < 1e-15
        else:
            assert not nan_rows.any()
        rows = np.arange(S["T"])
        per_band(rep, rows[fin], f"{name} table", np.abs(tab[fin] - want[fin]).max(1), 2.4e-7)
        assert np.all(np.diff(tab[fin], axis=1) >= 0), name
        assert np.all(tab[fin, -1] == 1.0), name
        assert g.shape == (S["T"], a_k.size, 4)
        bits = tab.view(np.uint32)
        for r in range(S["T"]):
            lo = np.searchsorted(tab[r], a_k, side="right")
            hi = np.searchsorted(tab[r], b_k, side="right")
            lohi = g[r, :, 0].astype(np.int64) & 0xFFFFFFFF
            assert np.array_equal(lohi & 0xFFFF, lo) and np.array_equal(lohi >> 16, hi), (name, r)
            for j, off in enumerate((-1, 0, 1)):
                assert np.array_equal(g[r, :, 1 + j].view(np.uint32), bits[r][np.clip(lo + off, 0, tab.shape[1] - 1)]), (name, r)
    rep.check()


# ---------------------------------------------------------------------------------------------
# b. the table sampler
# ---------------------------------------------------------------------------------------------
def check_sample(rep, tag, t, tab, loc, seed, off, row_offset, ang, axis, R, T):
    ref = D.igso3_draw(tab, t, loc, seed, off, global_rows(row_offset, len(t)))
    per_band(rep, t, f"{tag} angle (ulp)", np.abs(ang - ref["angle"]), angle_tol(ref["angle"]))
    per_band(rep, t, f"{tag} axis", np.abs(axis - ref["axis"]).max(1), AXIS_TOL)
    per_band(rep, t, f"{tag} R", geo(R, ref["noise"]), rot_geo_tol(ref["angle"]))
    neighbours(rep, t, T, f"{tag} angle", lambda tn: np.abs(ang - D.angle_lookup(tab, tn, ref["u"], loc)) / angle_tol(ref["angle"]))


@pytest.mark.parametrize("table", ["forward", "posterior"])
def test_table_sampler_every_row(S, cuda_device, table):
    """ops.igso3_sample over every row of the table: per-row row_idx with and without the guide records, and the shared-row
    path (guide built in shared memory) launched once per row.  Angle to 1 ulp of the restated lookup, axis to AXIS_TOL, R to
    rot_geo_tol."""
    ops = S["dx"].ops
    tab_d, g_d, tab = (S["fwd"], S["fg"], S["fwd_h"]) if table == "forward" else (S["post"], S["pg"], S["post_h"])
    T, loc = S["T"], S["loc"]
    rep = Report(f"table sampler, {table} table")
    for k, (seed, off, r0) in enumerate(STREAMS):
        t = layout(10 + k, T)
        ti = torch.tensor(t, device=cuda_device)
        for guide in (None, g_d):
            R, ang, ax = ops.igso3_sample(tab_d, (len(t),), row_idx=ti, seed=seed, rng_offset=off, row_offset=r0, want_angle=True,
                                          want_axis=True, guide=guide)
            check_sample(rep, f"row_idx{' guide' if guide is not None else ''}", t, tab, loc, seed, off, r0, host(ang), host(ax), host(R), T)
    seed, off, r0 = STREAMS[1]
    outs = [ops.igso3_sample(tab_d, (PER_T,), row=r, seed=seed, rng_offset=off, row_offset=r0 + r * PER_T, want_angle=True, want_axis=True)
            for r in range(T)]
    t = np.repeat(np.arange(T), PER_T)
    R, ang, ax = (host(torch.cat([o[i] for o in outs])) for i in range(3))
    check_sample(rep, "shared row", t, tab, loc, seed, off, r0, ang, ax, R, T)
    rep.check()


# ---------------------------------------------------------------------------------------------
# c. forward noising
# ---------------------------------------------------------------------------------------------
K_ANG, K_AXIS = 6, 4     # test_gpu_fwd_strata.py: relative angle and absolute axis error of the lean log of x0


def q_refs(S, t, x0, seed, off, r0):
    """The restated draws of every row from table rows t, t - 1 and t + 1 (clipped), and so3_scale(x0, sqrt_ac[t]) in fp64."""
    rows = global_rows(r0, len(t))
    T = S["T"]
    draws = {d: D.igso3_draw(S["fwd_h"], np.clip(t + d, 0, T - 1), S["loc"], seed, off, rows) for d in (-1, 0, 1)}
    sc = S["sc32"][t].astype(np.float64)
    lv = O.log_vec(polar(x0))
    th = np.linalg.norm(lv, axis=-1)
    scaled = O.exp_vec(sc[:, None] * lv)
    ref = draws[0]
    a = ref["angle"].astype(np.float64)
    eps = S["eps32"][t].astype(np.float64)
    # so3_scale's bound (test_gpu_fwd_strata.py), the noise's, and the product
    ref["x_t_tol"] = U24 * (4 + (K_ANG + K_AXIS + 2) * sc * th) + rot_geo_tol(a) + 4 * U24
    # ang * rcp(eps) * axis: 1 ulp of the angle, MUFU.RCP, two roundings, and the axis
    ref["target_tol"] = (a / eps) * (6 * U24 + AXIS_TOL2) + 1e-30
    g = D.score_g(a, eps)
    ref["score"] = g[:, None] * ref["axis"]
    # test_gpu_grad.py: 1e-5 of max(|g|, omega / (2 eps^2), 1) for the closed-form score, plus the axis
    ref["score_tol"] = 1e-5 * np.maximum.reduce([np.abs(g), a / (2 * eps ** 2), np.ones_like(a)]) + np.abs(g) * AXIS_TOL2
    for d in (-1, 0, 1):
        draws[d]["x_t"] = scaled @ draws[d]["noise"]
        e = S["eps32"][np.clip(t + d, 0, T - 1)].astype(np.float64)
        draws[d]["target_eps"] = (a / e)[:, None] * ref["axis"]         # the right draw over the eps of step t + d
    return draws


def check_q(rep, S, tag, t, draws, out, neighbour_checks):
    ref = draws[0]
    x_t = host(out["x_t"])
    per_band(rep, t, f"{tag} x_t", geo(x_t, ref["x_t"]), ref["x_t_tol"])
    tg = host(out["target"])
    per_band(rep, t, f"{tag} target", np.linalg.norm(tg - ref["target_eps"], axis=-1), ref["target_tol"])
    noise = host(out["noise"]) if out["noise"] is not None else None
    if noise is not None:
        per_band(rep, t, f"{tag} noise", geo(noise, ref["noise"]), rot_geo_tol(ref["angle"]))
    if out["score"] is not None:
        per_band(rep, t, f"{tag} score", np.linalg.norm(host(out["score"]) - ref["score"], axis=-1), ref["score_tol"])
    if neighbour_checks:
        dd = lambda tn: np.sign(tn - t)   # +-1 where the neighbour exists
        if noise is not None:
            neighbours(rep, t, S["T"], f"{tag} noise",
                       lambda tn: geo(noise, np.where((dd(tn) > 0)[:, None, None], draws[1]["noise"], draws[-1]["noise"])) / rot_geo_tol(ref["angle"]))
        neighbours(rep, t, S["T"], f"{tag} x_t",
                   lambda tn: geo(x_t, np.where((dd(tn) > 0)[:, None, None], draws[1]["x_t"], draws[-1]["x_t"])) / ref["x_t_tol"])
        neighbours(rep, t, S["T"], f"{tag} target, eps",
                   lambda tn: np.linalg.norm(tg - np.where((dd(tn) > 0)[:, None], draws[1]["target_eps"], draws[-1]["target_eps"]), axis=-1)
                   / ref["target_tol"])


@pytest.mark.parametrize("lanes", ["1", "2"])
def test_forward_noising_every_step(S, cuda_device, monkeypatch, lanes):
    """ops.q_sample_fused at every t with SO3D_QS_LANES = 1 / 2, with and without the guide: noise (one-row kernel, which
    the noise output selects), x_t, target and score against the restatement.  x_t: so3_scale's bound from
    test_gpu_fwd_strata.py plus the noise's; target: 1 ulp of the angle, MUFU.RCP and the axis; score: test_gpu_grad.py's
    1e-5 of its scale plus the axis."""
    monkeypatch.setenv("SO3D_QS_LANES", lanes)
    ops, T = S["dx"].ops, S["T"]
    p = S["p"]
    rep = Report(f"forward noising, SO3D_QS_LANES={lanes}")
    for k, (seed, off, r0) in enumerate(STREAMS):
        t = layout(20 + k, T)
        rng = np.random.default_rng(30 + k)
        x0 = rotations(rng, len(t))
        x0d, ti = dev(x0, cuda_device), torch.tensor(t, device=cuda_device)
        if k == 2:
            x0d = misaligned(x0d)
        draws = q_refs(S, t, x0, seed, off, r0)
        for guide in (None, S["fg"]):
            gt = " guide" if guide is not None else ""
            for want_noise, want_score in ((True, True), (False, True), (False, False)):
                out = ops.q_sample_fused(x0d, ti, p.sqrt_alphas_cumprod, p.sqrt_one_minus_alphas_cumprod, S["fwd"], seed=seed,
                                         rng_offset=off, row_offset=r0, want_noise=want_noise, want_score=want_score, guide=guide)
                tag = ("noise+score" if want_noise else "score" if want_score else "x_t") + gt
                check_q(rep, S, f"s{k} {tag}", t, draws, out, neighbour_checks=k == 0)
    rep.check()


# ---------------------------------------------------------------------------------------------
# d. the reverse step with noise
# ---------------------------------------------------------------------------------------------
def post_draw(S, t, seed, off, r0):
    return D.igso3_draw(S["post_h"], t, S["loc"], seed, off, global_rows(r0, len(t)))


def check_reverse(rep, S, tag, t, X, pred, out, mean_only, seed, off, r0):
    """t = 0 rows: exactly the mean-only step; t > 0: mean @ noise from posterior row t, check_step's bound plus the noise's."""
    A, B, C1, C2 = S["sched"]
    z = t == 0
    assert np.array_equal(out[z], mean_only[z]), tag
    ref = post_draw(S, t, seed, off, r0)
    nz = ~z
    tn = np.zeros(len(t), np.int64)
    names = BANDS
    lab = band_of(t)
    p64 = pred.astype(np.float64)
    check_step(rep, names, lab[nz], tn[nz], out[nz], X[nz], p64[nz], A[t[nz]], B[t[nz]], C1[t[nz]], C2[t[nz]], tag,
               noise=ref["noise"][nz], noise_tol=rot_geo_tol(ref["angle"][nz]), per_t=False)
    check_step(rep, names, lab[z], tn[z], out[z], X[z], p64[z], A[t[z]], B[t[z]], C1[t[z]], C2[t[z]], f"{tag} t=0 mean", per_t=False)

    return ref


def reverse_neighbours(rep, S, tag, t, X, pred, out, seed, off, r0, ref):
    A, B, C1, C2 = S["sched"]
    nz = t > 0
    p64 = pred.astype(np.float64)

    def ratio(tn):
        alt = D.igso3_draw(S["post_h"], tn, S["loc"], seed, off, global_rows(r0, len(t)))
        err, tol = check_step(Report(""), ["all"], np.zeros(nz.sum(), np.int64), t[nz], out[nz], X[nz], p64[nz], A[t[nz]], B[t[nz]],
                              C1[t[nz]], C2[t[nz]], "", noise=alt["noise"][nz], noise_tol=rot_geo_tol(ref["angle"][nz]), per_t=False)
        r = np.zeros(len(t))
        r[nz] = err / tol
        return r

    neighbours(rep, t, S["T"], f"{tag} out", ratio, rows=nz)


@pytest.mark.parametrize("lanes", ["1", "2"])
def test_reverse_step_every_step(S, cuda_device, monkeypatch, lanes):
    """ops.p_sample_fused with noise at every t: per-row t with post_guide given and None (SO3D_PS_LANES = 1 / 2), and every
    t as a shared step (two-row kernel; with want_x0_hat the one-row kernel).  t = 0 rows equal the mean-only step bit for
    bit; the others are mean @ noise_ref with noise_ref drawn from posterior row t, within step_tolerance plus the noise's
    bound, the mean from the fp64 p_mean_truth (strata.check_step)."""
    monkeypatch.setenv("SO3D_PS_LANES", lanes)
    ops, T = S["dx"].ops, S["T"]
    p = S["p"]
    sched = p._sched4()
    A, B, C1, C2 = S["sched"]
    rep = Report(f"reverse step with noise, SO3D_PS_LANES={lanes}")
    for k, (seed, off, r0) in enumerate(STREAMS):
        t = layout(40 + k, T)
        rng = np.random.default_rng(50 + k)
        X = rotations(rng, len(t))
        mag = np.exp(rng.uniform(math.log(1e-6), math.log(1.0), len(t)))
        pred = (unit_axes(rng, len(t)) * (mag / B[t])[:, None]).astype(np.float32)
        Xd, pd, ti = dev(X, cuda_device), dev(pred, cuda_device), torch.tensor(t, device=cuda_device)
        if k == 2:
            Xd = misaligned(Xd)
        mean_only = host(ops.p_sample_fused(Xd, pd, ti, *sched))
        for guide in (None, S["pg"]):
            out = host(ops.p_sample_fused(Xd, pd, ti, *sched, post_cdf=S["post"], post_guide=guide, seed=seed, rng_offset=off, row_offset=r0))
            ref = check_reverse(rep, S, f"s{k} per-row t{' guide' if guide is not None else ''}", t, X, pred, out, mean_only, seed, off, r0)
            if k == 0:
                reverse_neighbours(rep, S, f"s{k} per-row t{' guide' if guide is not None else ''}", t, X, pred, out, seed, off, r0, ref)
    if lanes == "1":   # shared t does not read SO3D_PS_LANES: run it once
        seed, off, r0 = STREAMS[1]
        t = np.repeat(np.arange(T), PER_T)
        rng = np.random.default_rng(60)
        X = rotations(rng, len(t))
        pred = (unit_axes(rng, len(t)) * (np.exp(rng.uniform(math.log(1e-6), 0.0, len(t))) / B[t])[:, None]).astype(np.float32)
        Xd, pd = dev(X, cuda_device), dev(pred, cuda_device)
        for x0h in (False, True):
            outs, means = [], []
            for r in range(T):
                sl = slice(r * PER_T, (r + 1) * PER_T)
                tt = torch.full((1,), r, dtype=torch.int64, device=cuda_device)
                o = ops.p_sample_fused(Xd[sl], pd[sl], tt, *sched, post_cdf=S["post"], seed=seed, rng_offset=off, row_offset=r0 + r * PER_T,
                                       want_x0_hat=x0h)
                outs.append(o[0] if x0h else o)
                means.append(ops.p_sample_fused(Xd[sl], pd[sl], tt, *sched))
            out, mean_only = host(torch.cat(outs)), host(torch.cat(means))
            tag = "shared t" + (" (x0_hat: one-row kernel)" if x0h else "")
            ref = check_reverse(rep, S, tag, t, X, pred, out, mean_only, seed, off, r0)
            reverse_neighbours(rep, S, tag, t, X, pred, out, seed, off, r0, ref)
    rep.check()


# ---------------------------------------------------------------------------------------------
# e. SE(3): the translation normals (rng_offset | 2^63) and one rotation check per kernel
# ---------------------------------------------------------------------------------------------
def normal_tol(t2):
    """Per-component bound of a device Box-Muller normal given the restated radial variates t = -2 ln u: MUFU.LG2 (2^-20.9
    absolute in log2 u, times 2 ln 2) and the roundings of t (2 U24 relative) move t by dt; the radius sqrt(t) then moves by
    at most sqrt(t + dt) - sqrt(t - dt) (it is not Lipschitz at t = 0, u = 1); MUFU.RSQ and the product add 6 U24 relative;
    the azimuth's MUFU sin / cos and fp32 argument (2^-20.9 + 6.4 U24) move the unit factor, and the final product 1 U24."""
    dt = 2 * math.log(2) * MUFU + 2 * U24 * t2
    r = np.sqrt(t2)
    dr = np.sqrt(t2 + dt) - np.sqrt(np.maximum(t2 - dt, 0)) + 6 * U24 * r
    tol = dr + r * (MUFU + 7.4 * U24)
    return np.repeat(tol, 2, axis=-1)          # (a, b) share radius a, (c, d) radius b


def se3_normals(seed, off, r0, n):
    z, t2 = D.normal4(D.philox(seed, global_rows(r0, n), off | D.SHIFT_STREAM))
    return z[:, :3], normal_tol(t2)[:, :3]


def test_se3_noising_every_step(S, cuda_device, monkeypatch):
    """ops.se3_q_sample_fused at every t, the two-row kernel (default) and the one-row kernel (SO3D_SE3_QS_LANES=1), with the
    guide: target_shift = z, the first three normals of Philox(seed, row, rng_offset | 2^63), within normal_tol; shift_t =
    sqrt_ac[t] shift0 + sqrt_1m_ac[t] shift_scale z; the rotation as the SO(3) noising (x_t)."""
    dx, T = S["dx"], S["T"]
    q = dx.SE3Diffusion(None).to(cuda_device)
    fwd = q.tables()[0]
    fg = q.guides()[0]
    rep = Report("SE(3) noising")
    seed, off, r0 = STREAMS[1]
    t = layout(70, T)
    rng = np.random.default_rng(71)
    x0 = rotations(rng, len(t))
    shift0 = (rng.standard_normal((len(t), 3)) * 10).astype(np.float32)
    z, ztol = se3_normals(seed, off, r0, len(t))
    draws = q_refs(S, t, x0, seed, off, r0)
    sc, eps = S["sc32"][t].astype(np.float64)[:, None], S["eps32"][t].astype(np.float64)[:, None]
    ss = float(np.float32(q.shift_scale))
    s64 = shift0.astype(np.float64)
    want = sc * s64 + eps * ss * z
    # ns = eps shift_scale (1 rounding), ns z (1), the FMA (1)
    stol = eps * ss * ztol + 3 * U24 * (np.abs(sc * s64) + np.abs(eps * ss * z))
    for lanes in ("2", "1"):
        monkeypatch.setenv("SO3D_SE3_QS_LANES", lanes)
        out = dx.ops.se3_q_sample_fused(dev(x0, cuda_device), dev(shift0, cuda_device), torch.tensor(t, device=cuda_device), q.sqrt_alphas_cumprod,
                                        q.sqrt_one_minus_alphas_cumprod, fwd, q.shift_scale, seed=seed, rng_offset=off, row_offset=r0, guide=fg)
        tag = f"SO3D_SE3_QS_LANES={lanes}"
        per_band(rep, t, f"{tag} target_shift", np.abs(host(out["target_shift"]) - z), ztol)
        per_band(rep, t, f"{tag} shift_t", np.abs(host(out["shift"]) - want), stol)
        per_band(rep, t, f"{tag} rot", geo(host(out["rot"]), draws[0]["x_t"]), draws[0]["x_t_tol"])
        per_band(rep, t, f"{tag} target_rot", np.linalg.norm(host(out["target_rot"]) - draws[0]["target_eps"], axis=-1), draws[0]["target_tol"])
    rep.check()


def test_se3_reverse_step_every_step(S, cuda_device):
    """ops.se3_p_sample_fused with noise, per-row t with the guide and shared t (two-row kernel) at every t: shift_out = the fp64
    posterior mean (test_gpu_fwd_strata.py's 4 U24 of its terms) + sigma[t] shift_scale z for t > 0; the rotation as the SO(3)
    reverse step."""
    dx, T = S["dx"], S["T"]
    q = dx.SE3Diffusion(None).to(cuda_device)
    post = q.tables()[1]
    pg = q.guides()[1]
    sig = q._sigma()
    sig64 = host(sig)
    A, B, C1, C2 = S["sched"]
    rep = Report("SE(3) reverse step with noise")
    seed, off, r0 = STREAMS[2]
    ss = float(np.float32(q.shift_scale))
    for shared in (False, True):
        t = np.repeat(np.arange(T), PER_T) if shared else layout(80, T)
        n = len(t)
        rng = np.random.default_rng(81 + shared)
        X = rotations(rng, n)
        pred = (unit_axes(rng, n) * (np.exp(rng.uniform(math.log(1e-6), 0.0, n)) / B[t])[:, None]).astype(np.float32)
        shift = (rng.standard_normal((n, 3)) * 10).astype(np.float32)
        pshift = rng.standard_normal((n, 3)).astype(np.float32)
        args = [dev(a, cuda_device) for a in (X, shift, pred, pshift)]
        if shared:
            outs = [dx.ops.se3_p_sample_fused(*[a[r * PER_T:(r + 1) * PER_T] for a in args], torch.full((1,), r, dtype=torch.int64, device=cuda_device),
                                              *q._sched(), sig, q.shift_scale, post_cdf=post, seed=seed, rng_offset=off, row_offset=r0 + r * PER_T)
                    for r in range(T)]
            rot, sh = host(torch.cat([o[0] for o in outs])), host(torch.cat([o[1] for o in outs]))
        else:
            rot, sh = dx.ops.se3_p_sample_fused(*args, torch.tensor(t, device=cuda_device), *q._sched(), sig, q.shift_scale, post_cdf=post,
                                                seed=seed, rng_offset=off, row_offset=r0, post_guide=pg)
            rot, sh = host(rot), host(sh)
        tag = "shared t" if shared else "per-row t guide"
        z, ztol = se3_normals(seed, off, r0, n)
        a, b, c1, c2 = A[t][:, None], B[t][:, None], C1[t][:, None], C2[t][:, None]
        x, ps = shift.astype(np.float64), pshift.astype(np.float64)
        on = (t > 0)[:, None]
        ns = sig64[t][:, None] * ss
        want = c1 * (x * a - ps * b) + c2 * x + np.where(on, ns * z, 0.0)
        size = c1 * (np.abs(x) * a + np.abs(ps) * b) + c2 * np.abs(x)
        stol = 4 * U24 * size + np.where(on, ns * ztol + 2 * U24 * np.abs(ns * z), 0.0)
        per_band(rep, t, f"{tag} shift_out", np.abs(sh - want), stol)
        ref = post_draw(S, t, seed, off, r0)
        nz = t > 0
        check_step(rep, BANDS, band_of(t)[nz], np.zeros(nz.sum(), np.int64), rot[nz], X[nz], pred[nz].astype(np.float64), A[t[nz]], B[t[nz]],
                   C1[t[nz]], C2[t[nz]], f"{tag} rot", noise=ref["noise"][nz], noise_tol=rot_geo_tol(ref["angle"][nz]), per_t=False)
    rep.check()


# ---------------------------------------------------------------------------------------------
# f. Bingham
# ---------------------------------------------------------------------------------------------
def test_bingham_device_normals(S, cuda_device):
    """ops.bingham_sample with device normals: q = L z / |L z| and R = quat_to_rmat(q) against fp64 from the restated z of
    Philox(seed, row, rng_offset).  |dq| <= 2 |L|_2 |dz| / |L z| (the normalisation at most doubles a perturbation) + 4 U24,
    R's entries within 4 |dq| + 8 U24."""
    dx = S["dx"]
    rng = np.random.default_rng(90)
    M = rng.standard_normal((4, 4))
    L = np.linalg.cholesky(M @ M.T + 0.5 * np.eye(4)).astype(np.float32)
    L64 = L.astype(np.float64)
    rep = Report("Bingham sampler")
    n = 50_000 + 7
    for seed, off, r0 in STREAMS:
        q, R = dx.ops.bingham_sample(dev(L, cuda_device), (n,), seed=seed, rng_offset=off, row_offset=r0, want_quat=True, want_rmat=True)
        z, t2 = D.normal4(D.philox(seed, global_rows(r0, n), off))
        ztol = normal_tol(t2)
        v = z @ L64.T
        qref = v / np.linalg.norm(v, axis=-1, keepdims=True)
        qtol = 2 * np.linalg.norm(L64, 2) * np.linalg.norm(ztol, axis=-1) / np.linalg.norm(v, axis=-1) + 4 * U24
        eq = np.linalg.norm(host(q) - qref, axis=-1)
        rep.add(f"row_offset={r0}", "q", eq, qtol)
        rep.add(f"row_offset={r0}", "R entries", np.abs(host(R) - O.quat_to_rmat(qref)).reshape(n, 9).max(-1), 4 * qtol + 8 * U24)
        # the same rows from the translation stream are other normals
        zo, _ = D.normal4(D.philox(seed, global_rows(r0, n), off | D.SHIFT_STREAM))
        vo = zo @ L64.T
        rep.add(f"row_offset={r0}", "other stream: 1 - fail", np.array([np.mean(np.linalg.norm(host(q) - vo / np.linalg.norm(vo, axis=-1, keepdims=True), axis=-1) <= qtol)]),
                1.0 - NEIGHBOUR_FAIL)
    rep.check()
