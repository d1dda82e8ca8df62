"""The forward SO(3) maps and the fused reverse step against float64, by stratum of the rotation angle (tests/strata.py)
and over the whole diffusion schedule.

Truth is the fp64 map evaluated at the rotation the fp32 input represents, its polar factor.  Every tolerance is
c * 2^-24 times a conditioning factor stated where it is used; near 0 there is none, so the tiny strata are checked to
relative precision.  Where the axis of a rotation by exactly pi has no defined sign (log is discontinuous there), the
comparison is up to that sign.  Each check prints its per-stratum table with -s.

The row-engine maps run on the lean arithmetic of so3d_math.cuh (axis_angle_fast, atan2_pos, MUFU rsqrt / rcp): both
row engines (SO3D_ROW_LANES = 1 / 2) are covered, with a ragged size above the persistent-engine threshold and a view
that is only 4-byte aligned.
"""
import math

import numpy as np
import pytest
import torch

from oracle import so3_oracle as O
from tests.strata import FWD_STRATA, U24, Report, fwd_stratum, polar, unit_axes

pytestmark = pytest.mark.gpu

N_PER = 1500
BIG = 256 * 148 * 6 + 13      # above the persistent engine's one-wave size, ragged
AMBIG = 4e-7                  # pi - theta below this: the sign of the axis of an fp32 matrix is not determined


@pytest.fixture(scope="module")
def dx(cuda_device):
    import diffusion_extensions_b200 as pkg

    pkg._lib.load()
    return pkg


def dev(a, device):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(device)


def host(t):
    return t.detach().cpu().numpy().astype(np.float64)


def strata_rows(seed, n=N_PER):
    rng = np.random.default_rng(seed)
    names = list(FWD_STRATA)
    R = np.concatenate([fwd_stratum(rng, n, k) for k in names])
    label = np.repeat(np.arange(len(names)), n)
    return names, label, R


TINY_TRUTH = 1e-4


def truth_log(R):
    """(polar factor, rotation vector, angle, unit axis) of each fp32 matrix (axis (0,0,1) at the identity).

    Below TINY_TRUTH the rotation vector is taken from the skew part of the fp32 matrix itself (fp64 log formula): an fp64
    matrix holds a rotation near I only to ~1e-16 absolute, so its SVD cannot give theta = 1e-20 to relative precision,
    while the polar factor's rotation vector differs from vee((R - R^T)/2) theta/sin(theta) by a relative |R^T R - I| / 2
    <= 2^-25 (the fp32 rounding of the diagonal)."""
    P = polar(R)
    lv = O.log_vec(P)
    raw = O.log_vec(np.asarray(R, np.float64))
    lv = np.where((np.linalg.norm(raw, axis=-1) < TINY_TRUTH)[:, None], raw, lv)
    th = np.linalg.norm(lv, axis=-1)
    ax = np.where(th[:, None] > 0, lv / np.maximum(th, 1e-300)[:, None], O.DEFAULT_AXIS)
    return P, lv, th, ax


def up_to_sign(err_plus, err_minus, th):
    """err_plus where the sign of the axis is determined, min(err_plus, err_minus) where theta is within AMBIG of pi."""
    return np.where(math.pi - th < AMBIG, np.minimum(err_plus, err_minus), err_plus)


def by_stratum(rep, names, label, what, err, tol):
    for i, k in enumerate(names):
        m = label == i
        if m.any():
            rep.add(k, what, err[m], np.broadcast_to(tol, err.shape)[m])


@pytest.fixture(scope="module")
def base():
    names, label, R = strata_rows(2024)
    P, lv, th, ax = truth_log(R)
    return dict(names=names, label=label, R=R, P=P, lv=lv, th=th, ax=ax)


# ---------------------------------------------------------------------------------------------
# log_rmat, log_vec, rmat_to_aa
# ---------------------------------------------------------------------------------------------
K_ANG = 6      # angle: relative 6 * 2^-24 (atan2_pos 2e-8 + MUFU.RCP, and the rounding of s and c)
K_AXIS = 4     # axis: 4 * 2^-24 absolute, at every angle (the symmetric-part axis above c = -0.9 keeps it away from 1/sin)


def check_log_outputs(rep, names, label, th, ax, lv, got_lv, got_skew, got_ax, got_ang, tag):
    e_lv = up_to_sign(np.linalg.norm(got_lv - lv, axis=-1), np.linalg.norm(got_lv + lv, axis=-1), th)
    # |theta n - theta' n'| <= |theta - theta'| + theta |n - n'|
    tol_lv = U24 * (K_ANG + K_AXIS) * th + 1e-45
    by_stratum(rep, names, label, f"log_vec{tag}", e_lv, tol_lv)
    sk = np.stack((got_skew[:, 2, 1], got_skew[:, 0, 2], got_skew[:, 1, 0]), -1)
    e_sk = up_to_sign(np.linalg.norm(sk - lv, axis=-1), np.linalg.norm(sk + lv, axis=-1), th)
    asym = np.abs(got_skew + np.swapaxes(got_skew, -1, -2)).reshape(-1, 9).max(-1)
    by_stratum(rep, names, label, f"log_rmat{tag}", np.maximum(e_sk, asym), tol_lv)
    by_stratum(rep, names, label, f"aa angle{tag}", np.abs(got_ang - th), U24 * K_ANG * th + 1e-45)
    e_ax = up_to_sign(np.linalg.norm(got_ax - ax, axis=-1), np.linalg.norm(got_ax + ax, axis=-1), th)
    by_stratum(rep, names, label, f"aa axis{tag}", e_ax, U24 * K_AXIS)


@pytest.mark.parametrize("lanes", ["1", "2"])
def test_log_maps_by_stratum(dx, cuda_device, base, monkeypatch, lanes):
    """log_rmat, log_vec and rmat_to_aa on every stratum, from exactly 0 (axis (0,0,1), angle 0, log 0 exactly) to
    exactly pi, including the subnormal-skew rows (|vee(R - R^T)|^2 below FLT_MIN) and the kNearPiCos switch.  Angle to
    relative K_ANG 2^-24, axis to K_AXIS 2^-24 absolute, log to the sum; no allowance near 0.  The same rows tiled to a
    ragged BIG rows and read through a 4-byte-aligned view give the same answers."""
    monkeypatch.setenv("SO3D_ROW_LANES", lanes)
    U = dx.util
    names, label, R, th, ax, lv = base["names"], base["label"], base["R"], base["th"], base["ax"], base["lv"]
    rep = Report(f"log maps by stratum, SO3D_ROW_LANES={lanes}")
    Rd = dev(R, cuda_device)
    got_ax, got_ang = U.rmat_to_aa(Rd)
    outs = [host(dx.ops.log_vec(Rd)), host(U.log_rmat(Rd)), host(got_ax), host(got_ang)[:, 0]]
    for o in outs:
        assert np.isfinite(o).all()
    check_log_outputs(rep, names, label, th, ax, lv, *outs, "")
    assert np.array_equal(outs[2][label == 0], np.tile([0.0, 0.0, 1.0], ((label == 0).sum(), 1)))
    # ragged size above the persistent-engine threshold, and a 4-byte-aligned view
    reps = -(-BIG // len(R))
    idx = np.arange(BIG) % len(R)
    big = dev(np.tile(R, (reps, 1, 1))[:BIG], cuda_device)
    view = torch.empty(BIG + 1, 3, 3, device=cuda_device)[1:]
    view.copy_(big)
    assert view.data_ptr() % 16 != 0
    for src, tag in ((big, " big"), (view, " view")):
        a, g = U.rmat_to_aa(src)
        o = [host(dx.ops.log_vec(src)), host(U.log_rmat(src)), host(a), host(g)[:, 0]]
        check_log_outputs(rep, names, label[idx], th[idx], ax[idx], lv[idx], *o, tag)
    rep.check()


# ---------------------------------------------------------------------------------------------
# so3_scale
# ---------------------------------------------------------------------------------------------
SCALES = [0.0, -0.37, -3.0, 0.37, 1.0, 1.9, 3.0, 100.0, 20300.0]   # s theta crosses pi and 2 pi; 2.03e4 ~ the schedule's top


def geo(a, b):
    return O.geodesic_angle(a, b)


@pytest.mark.parametrize("lanes", ["1", "2"])
def test_so3_scale_by_stratum(dx, cuda_device, base, monkeypatch, lanes):
    """so3_scale(R, s) vs exp(s log P) in fp64, per-row and shared s.  The rotation vector s theta n carries the angle's
    and the axis's relative errors times |s| theta, and the argument reduction of sincos adds 2^-24 |s| theta: geodesic
    error <= 2^-24 (4 + (K_ANG + K_AXIS + 2) |s| theta).  Rows at exactly pi (sign of the axis undetermined) may match
    either branch."""
    monkeypatch.setenv("SO3D_ROW_LANES", lanes)
    U = dx.util
    names, label, R, P, th, lv = base["names"], base["label"], base["R"], base["P"], base["th"], base["lv"]
    rep = Report(f"so3_scale by stratum, SO3D_ROW_LANES={lanes}")
    Rd = dev(R, cuda_device)
    rng = np.random.default_rng(7)
    for sv in SCALES:
        for shared in (False, True):
            s = np.full(len(R), sv, np.float32)
            if not shared:
                s = (s * rng.uniform(0.98, 1.02, len(R))).astype(np.float32)
            got = host(U.so3_scale(Rd, float(sv) if shared else dev(s, cuda_device)))
            assert np.isfinite(got).all()
            s64 = s.astype(np.float64)[:, None]
            e = up_to_sign(geo(got, O.exp_vec(s64 * lv)), geo(got, O.exp_vec(-s64 * lv)), th)
            tol = U24 * (4 + (K_ANG + K_AXIS + 2) * np.abs(s64[:, 0]) * th)
            by_stratum(rep, names, label, f"s={sv:g}{' shared' if shared else ''}", e, tol)
    rep.check()


# ---------------------------------------------------------------------------------------------
# so3_lerp, rmat_dist
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lanes", ["1", "2"])
def test_lerp_and_dist_by_stratum(dx, cuda_device, monkeypatch, lanes):
    """so3_lerp(A, B, w) with the relative rotation A^T B drawn per stratum, w in [0, 1] and outside it, vs
    P_A exp(w log(P_A^T P_B)); rmat_dist vs sqrt(2) angle(P_A^T P_B).  The kernel forms A^T B in fp32, which holds the
    relative rotation to ~2^-24 absolute (not relative): lerp error <= 2^-24 (6 + 6 |w| + (K_ANG + K_AXIS) |w| theta),
    dist error <= 2^-24 (6 + K_ANG theta).  Relative angles within AMBIG of pi may match either branch."""
    monkeypatch.setenv("SO3D_ROW_LANES", lanes)
    U = dx.util
    names, label, C = strata_rows(99, 800)
    rng = np.random.default_rng(100)
    A = O.rodrigues(unit_axes(rng, len(C)), rng.uniform(0, math.pi, len(C))).astype(np.float32)
    B = (A.astype(np.float64) @ C.astype(np.float64)).astype(np.float32)
    PA, PB = polar(A), polar(B)
    rel = np.swapaxes(PA, -1, -2) @ PB
    lv = O.log_vec(rel)
    th = np.linalg.norm(lv, axis=-1)
    rep = Report(f"so3_lerp / rmat_dist by stratum, SO3D_ROW_LANES={lanes}")
    Ad, Bd = dev(A, cuda_device), dev(B, cuda_device)
    for wname, w in (("w in [0,1]", rng.uniform(0, 1, len(C))), ("w in [-2,-0]", -rng.uniform(0, 2, len(C))), ("w in [1,3]", rng.uniform(1, 3, len(C))),
                     ("w=0", np.zeros(len(C))), ("w=1", np.ones(len(C)))):
        w = w.astype(np.float32)
        got = host(U.so3_lerp(Ad, Bd, dev(w[:, None], cuda_device)))
        assert np.isfinite(got).all()
        w64 = w.astype(np.float64)[:, None]
        e = up_to_sign(geo(got, PA @ O.exp_vec(w64 * lv)), geo(got, PA @ O.exp_vec(-w64 * lv)), th)
        by_stratum(rep, names, label, f"lerp {wname}", e, U24 * (6 + 6 * np.abs(w64[:, 0]) + (K_ANG + K_AXIS) * np.abs(w64[:, 0]) * th))
    d = host(U.rmat_dist(Ad, Bd))
    by_stratum(rep, names, label, "rmat_dist", np.abs(d - math.sqrt(2.0) * th), U24 * (6 + K_ANG * th))
    same = host(U.rmat_dist(Ad, Ad))
    rep.add("A = B", "rmat_dist", same, 6 * U24)
    rep.check()


# ---------------------------------------------------------------------------------------------
# rmat_to_quat, quat_to_rmat
# ---------------------------------------------------------------------------------------------
def test_quaternion_maps(dx, cuda_device, base):
    """rmat_to_quat on every stratum, including its branch boundaries (tr R = 0, tied largest diagonals): unit length,
    real part >= 0, equal to (cos theta/2, sin theta/2 n) of the polar factor (up to sign where the real part is within
    rounding of 0) to 4 2^-24, and quat_to_rmat(q) returns to P.  quat_to_rmat against util.py:222-252 in fp64 for |q|
    from 1e-15 to 1e15: the reference formula is finite in fp32 for |q| in [1.1e-19, 1.8e19] (|q|^2 a normal float)."""
    U = dx.util
    names, label, R, P, th, ax = base["names"], base["label"], base["R"], base["P"], base["th"], base["ax"]
    rep = Report("rmat_to_quat / quat_to_rmat")
    q = host(U.rmat_to_quat(dev(R, cuda_device)))
    assert np.isfinite(q).all() and np.all(q[:, 0] >= 0)
    qt = np.concatenate([np.cos(th / 2)[:, None], np.sin(th / 2)[:, None] * ax], -1)
    amb = qt[:, 0] < 4 * U24
    e = np.where(amb, np.minimum(np.linalg.norm(q - qt, axis=-1), np.linalg.norm(q + qt, axis=-1)), np.linalg.norm(q - qt, axis=-1))
    by_stratum(rep, names, label, "q vs truth", e, 4 * U24)
    by_stratum(rep, names, label, "|q| - 1", np.abs(np.linalg.norm(q, axis=-1) - 1), 3 * U24)
    by_stratum(rep, names, label, "round trip", geo(O.quat_to_rmat(q), P), 8 * U24)
    rng = np.random.default_rng(5)
    n = 20000
    mag = np.exp(rng.uniform(math.log(1e-15), math.log(1e15), n))
    qq = (rng.standard_normal((n, 4)) * (mag / 2)[:, None]).astype(np.float32)
    qq[:4] = [[1, 0, 0, 0], [0, 1, 0, 0], [1e-15, 0, 0, 0], [0, 0, 0, 1e15]]
    got = host(U.quat_to_rmat(dev(qq, cuda_device)))
    assert np.isfinite(got).all()
    want = O.quat_to_rmat(qq.astype(np.float64))
    # each entry: two_s (2 roundings) times a sum of two products (3 roundings) of size <= |q|^2
    rep.add("|q| in [1e-15,1e15]", "quat_to_rmat entries", np.abs(got - want).reshape(n, 9).max(-1), 8 * U24)
    rep.check()


# ---------------------------------------------------------------------------------------------
# exp_vec, aa_to_rmat
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lanes", ["1", "2"])
def test_exp_maps(dx, cuda_device, monkeypatch, lanes):
    """exp_vec(v) for |v| from 0 (and subnormal) to 500, and aa_to_rmat(axis, angle) with axis norms 1e-3 .. 1e3 and
    angles in [-500, 500] (tiny ones of both signs), vs fp64 Rodrigues.  The fp32 angle (|v|, or the angle operand) is
    reduced modulo 2 pi with an error of ~2^-24 |angle|: entries within 2^-24 (6 + 3 |angle|); for FLT_MIN <= |v| <= 1e-2
    the skew part carries v itself, checked to relative 6 2^-24."""
    monkeypatch.setenv("SO3D_ROW_LANES", lanes)
    U = dx.util
    rng = np.random.default_rng(11)
    rep = Report(f"exp_vec / aa_to_rmat, SO3D_ROW_LANES={lanes}")
    n = 4000
    for name, lo, hi in (("|v|=0", 0, 0), ("subnormal", 1e-45, 1e-38), ("[1e-38,1e-7]", 1e-38, 1e-7), ("[1e-7,1e-2]", 1e-7, 1e-2),
                         ("[1e-2,pi]", 1e-2, math.pi), ("[pi,4pi]", math.pi, 4 * math.pi), ("[4pi,500]", 4 * math.pi, 500.0)):
        p = np.zeros(n) if hi == 0 else (np.exp(rng.uniform(math.log(lo), math.log(hi), n)) if lo < 1e-2 or lo > 4 else rng.uniform(lo, hi, n))
        v = (unit_axes(rng, n) * p[:, None]).astype(np.float32)
        got = host(U.exp_vec(dev(v, cuda_device)))
        assert np.isfinite(got).all(), name
        v64 = v.astype(np.float64)
        want = O.exp_vec(v64)
        L = np.linalg.norm(v64, axis=-1)
        rep.add(name, "exp_vec entries", np.abs(got - want).reshape(n, 9).max(-1), U24 * (6 + 3 * L))
        if 1e-38 <= lo and hi <= 1e-2:
            # the skew part is v sin|v|/|v|, relative: k = sin(t/2) MUFU.RSQ(t^2), then k v, w (2 k v), the average of two
            # entries: ~6 roundings.  (A vector whose length is below FLT_MIN comes out as the identity: absolute error
            # < 1.2e-38, covered by the entries check above.)
            skew = lambda m: O.skew2vec((m - np.swapaxes(m, -1, -2)) / 2)
            rep.add(name, "exp_vec skew (rel)", np.linalg.norm(skew(got) - skew(want), axis=-1) / L, 6 * U24)
        ang = p.astype(np.float32) * rng.choice([-1.0, 1.0], n).astype(np.float32)
        nrm = np.exp(rng.uniform(math.log(1e-3), math.log(1e3), n))
        axes = (unit_axes(rng, n) * nrm[:, None]).astype(np.float32)
        if hi == 0:
            ang[:] = 0
        got = host(U.aa_to_rmat(dev(axes, cuda_device), dev(ang[:, None], cuda_device)))
        assert np.isfinite(got).all(), name
        want = O.aa_to_rmat(axes.astype(np.float64), ang.astype(np.float64)[:, None])
        rep.add(name, "aa_to_rmat entries", np.abs(got - want).reshape(n, 9).max(-1), U24 * (6 + 3 * np.abs(ang.astype(np.float64))))
    rep.check()


# ---------------------------------------------------------------------------------------------
# log_prob_and_score near the identity
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["closed", "auto", "series"])
@pytest.mark.parametrize("lanes", ["1", "2"])
def test_log_prob_and_score_near_identity(dx, cuda_device, monkeypatch, mode, lanes):
    """IGSO(3) log-density and score of rotations in the subnormal-skew and normal-tiny strata: finite, the density equals
    f(omega ~ 0) to 1e-5 relative (f is flat there: f(omega) - f(0) ~ omega^2), and the score, whose size is
    proportional to omega, goes to 0 with it: within 1e-5 |omega| / eps^2 of the fp64 score, plus an absolute 1e-10 (the
    fp32 evaluators' floor near 0, against scores of size ~1e-3 at omega = 1e-7)."""
    monkeypatch.setenv("SO3D_LOGP_LANES", lanes)
    rng = np.random.default_rng(12)
    rep = Report(f"log_prob_and_score near the identity, mode={mode} SO3D_LOGP_LANES={lanes}")
    n = 6000
    for name in ("subnormal skew", "normal tiny", "theta=0"):
        R = fwd_stratum(rng, n, name)
        _, _, th, ax = truth_log(R)
        eps = np.exp(rng.uniform(math.log(0.05), math.log(1.0 if mode == "closed" else 2.0), n)).astype(np.float32)
        d = dx.IsotropicGaussianSO3(dev(eps, cuda_device), mode=mode, series_terms=2000)
        lp, sc = d.log_prob_and_score(dev(R, cuda_device))
        lp, sc = host(lp)[:, 0], host(sc)
        assert np.isfinite(lp).all() and np.isfinite(sc).all(), name
        e64 = eps.astype(np.float64)
        f0, _ = O.igso3_series(np.zeros(n), e64)
        rep.add(name, "log f - log f(0)", np.abs(lp - np.log(f0)), 1e-5 * np.maximum(1.0, np.abs(np.log(f0))))
        # d log f / d omega -> -omega (1/(2 eps^2) ...) : the fp64 slope at 1e-3 eps, scaled down to omega
        _, g1 = O.igso3_series(1e-3 * e64, e64)
        want = (g1 / (1e-3 * e64) * th)[:, None] * ax
        rep.add(name, "score", np.linalg.norm(sc - want, axis=-1), 1e-5 * th / e64 ** 2 + 1e-10)
    rep.check()


# ---------------------------------------------------------------------------------------------
# the fused reverse step over the whole schedule
# ---------------------------------------------------------------------------------------------
T_STEPS = [1, 2, 10, 100, 400, 600, 800, 900, 990, 998, 999]
K0, K1, K2 = 16, 8, 8


def step_rows(seed, t_list, n_per):
    """x_t over every stratum, a step index per row from t_list, and pred with |b pred| small, near pi and beyond pi."""
    names, label, X = strata_rows(seed, n_per)
    rng = np.random.default_rng(seed + 1)
    n = len(X)
    t = rng.choice(np.asarray(t_list), n)
    kind = rng.integers(0, 3, n)
    mag = np.where(kind == 0, np.exp(rng.uniform(math.log(1e-6), math.log(1.0), n)),
                   np.where(kind == 1, math.pi + rng.uniform(-1e-3, 1e-3, n), rng.uniform(math.pi, 3 * math.pi, n)))
    return names, label, X, t, kind, mag


def other_branch(lv):
    """The rotation vector (theta - 2 pi) n: the same rotation as theta n, the other branch of log at pi."""
    th = np.linalg.norm(lv, axis=-1)
    return lv * ((th - 2 * math.pi) / np.maximum(th, 1e-300))[:, None]


def p_mean_truth(w, pred, a, b, c1, c2):
    """fp64 mean of diffusion.py:291-313 for x_t = exp(hat(w)) (w the rotation vector of x_t's polar factor) with the
    fp32 scalars the kernel reads: x0_hat = exp(a w) exp(b pred)^T, mean = exp(c1 log x0_hat) exp(c2 w), for both branches
    of log at pi of x0_hat."""
    x0 = O.exp_vec(a[:, None] * w) @ np.swapaxes(O.exp_vec(b[:, None] * pred), -1, -2)
    lv0 = O.log_vec(x0)
    th0 = np.linalg.norm(lv0, axis=-1)
    q4 = O.exp_vec(c2[:, None] * w)
    return x0, th0, O.exp_vec(lv0 * c1[:, None]) @ q4, O.exp_vec(other_branch(lv0) * c1[:, None]) @ q4


def step_tolerance(th, a, b, pred, c1, c2):
    """First-order propagation of fp32 rounding through the step (all terms in units of 2^-24, geodesic):
      x0_hat = exp(a theta n) exp(-b pred): the fp32 rotation vectors a theta n and b pred carry relative errors of a few
      units and sincos reduces them modulo 2 pi with ~1 unit per unit of angle, so  e0 = K1 (|a| theta + |b| |pred|) + K0;
      scale(x0_hat, c1) moves that error by c1 (c1 <= 1) and reads x0_hat's axis from a quaternion, which is well
      conditioned at every angle (no 1/sin);  so3_scale(x_t, c2) adds K2 c2 theta (axis and angle of x_t, relative);
    tol = 2^-24 (K0 + K1 c1 (|a| theta + |b| |pred|) + K2 c2 theta) for the mean, and e0 for x0_hat."""
    bp = np.abs(b) * np.linalg.norm(pred, axis=-1)
    e0 = U24 * (K0 + K1 * (np.abs(a) * th + bp))
    return U24 * (K0 + K1 * c1 * (np.abs(a) * th + bp) + K2 * c2 * th), e0


def check_step(rep, names, label, t, got_mean, X, pred, a, b, c1, c2, tag, got_x0=None):
    """x_t rows at pi within AMBIG (no defined axis sign) may take either branch of their log, consistently in both uses."""
    _, w, th, _ = truth_log(X)
    tol, e0 = step_tolerance(th, a, b, pred, c1, c2)
    x0, th0, m1, m2 = p_mean_truth(w, pred, a, b, c1, c2)
    near = math.pi - th0 <= e0          # x0_hat within its own error bound of pi: either branch of scale(x0_hat, c1)
    err = np.where(near, np.minimum(geo(got_mean, m1), geo(got_mean, m2)), geo(got_mean, m1))
    e_x0 = geo(got_x0, x0) if got_x0 is not None else None
    amb = math.pi - th < AMBIG
    if amb.any():
        x0b, th0b, m1b, m2b = p_mean_truth(other_branch(w[amb]), pred[amb], a[amb], b[amb], c1[amb], c2[amb])
        nb = math.pi - th0b <= e0[amb]
        eb = np.where(nb, np.minimum(geo(got_mean[amb], m1b), geo(got_mean[amb], m2b)), geo(got_mean[amb], m1b))
        err[amb] = np.minimum(err[amb], eb)
        near[amb] &= nb
        if got_x0 is not None:
            e_x0[amb] = np.minimum(e_x0[amb], geo(got_x0[amb], x0b))
    for tv in np.unique(t):
        m = t == tv
        by_stratum(rep, names, label[m], f"{tag} t={tv}", err[m], tol[m])
    rep.add("all", f"{tag} rows at x0_hat ~ pi", np.array([near.mean()]), 0.02)
    if got_x0 is not None:
        for tv in np.unique(t):
            m = t == tv
            by_stratum(rep, names, label[m], f"{tag} x0_hat t={tv}", e_x0[m], e0[m])


def sched(p):
    return [p.__getattr__(k).detach().cpu().numpy().astype(np.float64) for k in
            ("sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1", "posterior_mean_coef2")]


@pytest.mark.parametrize("ps_lanes", ["1", "2"])
def test_reverse_step_whole_schedule(dx, cuda_device, monkeypatch, ps_lanes):
    """p_mean_variance (per-row t, and every t shared through t[:1]) and x0_hat vs the fp64 mean of diffusion.py:291-313
    for t in T_STEPS, every x_t stratum and |b pred| small, near pi and beyond pi.  Tolerance: step_tolerance.  scale(x0_hat,
    c1) is discontinuous where x0_hat's angle is pi; rows whose fp64 x0_hat is within its error bound of pi may match either
    branch, and they must be under 2 % of the rows."""
    monkeypatch.setenv("SO3D_PS_LANES", ps_lanes)
    p = dx.SO3Diffusion(None).to(cuda_device)
    A, B, C1, C2 = sched(p)
    names, label, X, t, kind, mag = step_rows(31, T_STEPS, 300)
    rng = np.random.default_rng(32)
    pred = (unit_axes(rng, len(X)) * (mag / B[t])[:, None]).astype(np.float32)
    rep = Report(f"reverse step over the schedule, SO3D_PS_LANES={ps_lanes}")
    Xd, predd = dev(X, cuda_device), dev(pred, cuda_device)
    p.denoise_fn = lambda xx, tt: predd
    p64 = pred.astype(np.float64)
    mean = host(p.p_mean_variance(Xd, torch.tensor(t, device=cuda_device))[0])
    assert np.isfinite(mean).all()
    check_step(rep, names, label, t, mean, X, p64, A[t], B[t], C1[t], C2[t], "per-row")
    if ps_lanes == "1":
        mean_x, x0h = dx.ops.p_sample_fused(Xd, predd, torch.tensor(t, device=cuda_device), *p._sched4(), want_x0_hat=True)
        check_step(rep, names, label, t, host(mean_x), X, p64, A[t], B[t], C1[t], C2[t], "x0 kernel", got_x0=host(x0h))
    for tv in T_STEPS:   # shared step
        m = t == tv
        p.denoise_fn = lambda xx, tt, m=m: dev(pred[m], cuda_device)
        got = host(p.p_mean_variance(dev(X[m], cuda_device), torch.full((1,), tv, device=cuda_device))[0])
        check_step(rep, names, label[m], t[m], got, X[m], p64[m], A[t[m]], B[t[m]], C1[t[m]], C2[t[m]], "shared")
    rep.check()


@pytest.mark.parametrize("lanes", ["1", "2"])
def test_se3_reverse_step_whole_schedule(dx, cuda_device, monkeypatch, lanes):
    """The SE(3) posterior mean (se3_p_sample_fused without noise, per-row t and shared t) vs oracle se3_p_mean: the
    rotation within step_tolerance, the translation c1 (a x - b pred) + c2 x within 2^-24 (4 |terms| summed)."""
    monkeypatch.setenv("SO3D_ROW_LANES", lanes)
    p = dx.SE3Diffusion(None).to(cuda_device)
    A, B, C1, C2 = sched(p)
    names, label, X, t, kind, mag = step_rows(41, T_STEPS, 150)
    rng = np.random.default_rng(42)
    n = len(X)
    pred = (unit_axes(rng, n) * (mag / B[t])[:, None]).astype(np.float32)
    shift = (rng.standard_normal((n, 3)) * 10).astype(np.float32)
    pshift = rng.standard_normal((n, 3)).astype(np.float32)
    rep = Report(f"SE(3) reverse step over the schedule, SO3D_ROW_LANES={lanes}")
    sig = p._sigma()

    def run(sel, tt):
        r, s = dx.ops.se3_p_sample_fused(dev(X[sel], cuda_device), dev(shift[sel], cuda_device), dev(pred[sel], cuda_device),
                                         dev(pshift[sel], cuda_device), tt, *p._sched(), sig, p.shift_scale, post_cdf=None)
        return host(r), host(s)

    def check(sel, rot, sh, tag):
        ts = t[sel]
        a, b, c1, c2 = A[ts], B[ts], C1[ts], C2[ts]
        check_step(rep, names, label[sel], ts, rot, X[sel], pred[sel].astype(np.float64), a, b, c1, c2, tag)
        x, ps = shift[sel].astype(np.float64), pshift[sel].astype(np.float64)
        want = c1[:, None] * (x * a[:, None] - ps * b[:, None]) + c2[:, None] * x
        size = c1[:, None] * (np.abs(x) * a[:, None] + np.abs(ps) * b[:, None]) + c2[:, None] * np.abs(x)
        rep.add("all", f"{tag} translation", np.abs(sh - want) / size, 4 * U24)

    allr = np.arange(n)
    rot, sh = run(allr, torch.tensor(t, device=cuda_device))
    check(allr, rot, sh, "per-row")
    for tv in T_STEPS:
        m = np.nonzero(t == tv)[0]
        rot, sh = run(m, torch.full((1,), tv, device=cuda_device))
        check(m, rot, sh, "shared")
    rep.check()


def test_device_seeded_steps_at_t0(dx, cuda_device):
    """The device-seeded (CUDA-graph) SO(3) and SE(3) steps at t = 0, where no noise is drawn: the output is the posterior
    mean, vs fp64 within step_tolerance."""
    names, label, X, _, _, mag = step_rows(51, [0], 200)
    n = len(X)
    rng = np.random.default_rng(52)
    t = np.zeros(n, np.int64)
    rep = Report("device-seeded steps at t = 0")
    p = dx.SO3Diffusion(None).to(cuda_device)
    A, B, C1, C2 = sched(p)
    pred = (unit_axes(rng, n) * (mag / B[0])[:, None]).astype(np.float32)
    seed = torch.tensor([1234], dtype=torch.int64, device=cuda_device)
    post = p.tables()[1]
    out = dx.ops.p_sample_fused(dev(X, cuda_device), dev(pred, cuda_device), torch.zeros(1, dtype=torch.int64, device=cuda_device), *p._sched4(),
                                post_cdf=post, seed=seed, rng_offset=0)
    check_step(rep, names, label, t, host(out), X, pred.astype(np.float64), A[t], B[t], C1[t], C2[t], "so3 dseed")
    q = dx.SE3Diffusion(None).to(cuda_device)
    shift = (rng.standard_normal((n, 3)) * 10).astype(np.float32)
    pshift = rng.standard_normal((n, 3)).astype(np.float32)
    rot, sh = dx.ops.se3_p_sample_fused(dev(X, cuda_device), dev(shift, cuda_device), dev(pred, cuda_device), dev(pshift, cuda_device),
                                        torch.zeros(1, dtype=torch.int64, device=cuda_device), *q._sched(), q._sigma(), q.shift_scale,
                                        post_cdf=q.tables()[1], seed=seed, rng_offset=0)
    check_step(rep, names, label, t, host(rot), X, pred.astype(np.float64), A[t], B[t], C1[t], C2[t], "se3 dseed")
    rep.check()
