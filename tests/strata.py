"""Rotation strata and the per-stratum error report shared by the fp64 comparison tests (test_gpu_grad.py,
test_gpu_fwd_strata.py, test_gpu_draws.py).

Inputs are drawn by stratum of the rotation angle so that every region where an SO(3) kernel switches formula or loses
precision gets rows of its own, and a failure names the region.  All rotations are built in fp64 (Rodrigues) and then
rounded to fp32, which is what a caller hands the kernels.
"""
import math

import numpy as np

from oracle import so3_oracle as O

U24 = 2.0 ** -24


class Report:
    """Per-stratum maximum of err / tol; the test fails if any stratum exceeds 1 and names it."""

    def __init__(self, title):
        self.title, self.rows = title, []

    def add(self, stratum, what, err, tol):
        err, tol = np.broadcast_to(np.asarray(err, np.float64), np.shape(tol) or np.shape(err)), np.asarray(tol, np.float64)
        ratio = err / tol
        ratio = np.where(np.isnan(ratio), np.inf, ratio)
        self.rows.append((stratum, what, float(np.max(err, initial=0.0)), float(np.max(ratio, initial=0.0))))

    def check(self):
        print(f"\n{self.title}")
        for st, what, e, r in self.rows:
            print(f"  {st:24s} {what:22s} max err {e:9.2e}   max err/tol {r:6.3f}")
        bad = [(st, what, e, r) for st, what, e, r in self.rows if not r <= 1.0]
        assert not bad, f"{self.title}: over tolerance in {bad}"


def unit_axes(rng, n):
    ax = rng.standard_normal((n, 3))
    return ax / np.linalg.norm(ax, axis=-1, keepdims=True)


THETA_STRATA = [
    ("theta=0", 0.0, 0.0), ("[1e-7,1e-4]", 1e-7, 1e-4), ("s=1e-4+-1%", 0.99e-4, 1.01e-4), ("[1e-4,1e-2]", 1e-4, 1e-2),
    ("[1e-2,2.8]", 1e-2, 2.8), ("[2.8,3.0]", 2.8, 3.0), ("[3.0,3.1]", 3.0, 3.1), ("[3.1,pi-1e-3]", 3.1, math.pi - 1e-3),
    ("theta=pi", math.pi, math.pi),
]


def rot_stratum(rng, n, lo, hi):
    """fp32 rotations (Rodrigues in fp64, then rounded) with angles in [lo, hi] (log-uniform below 1e-2)."""
    if lo == hi:
        th = np.full(n, lo)
    elif hi <= 1e-2:
        th = np.exp(rng.uniform(math.log(lo), math.log(hi), n))
    else:
        th = rng.uniform(lo, hi, n)
    R = O.rodrigues(unit_axes(rng, n), th).astype(np.float32)
    if lo == 0.0:
        R[:] = np.eye(3, dtype=np.float32)
    return R


def pi_amp(th):
    """1/sin(theta) above pi/2, 1 below.  Near pi an fp32 matrix holds its axis only to ~2^-24/sin(theta), which bounds
    every gradient taken through log there; near 0 the problem is well conditioned and gets no allowance."""
    th = np.asarray(th, np.float64)
    return np.where(th > math.pi / 2, 1.0 / np.sin(np.minimum(th, math.pi - 1e-300)), 1.0)


def angle_of(R):
    """angle of the fp32 matrix (fp64 evaluation)."""
    return O.rmat_to_aa(R.astype(np.float64))[1][:, 0]


# ---------------------------------------------------------------------------------------------
# strata of the forward maps: every THETA_STRATA region plus the places where the lean (row-engine) arithmetic switches
# ---------------------------------------------------------------------------------------------
C_NEAR_PI = -0.9     # csrc/so3d_math.cuh kNearPiCos: below it the axis comes from the symmetric part
THETA_NEAR_PI_SWITCH = math.acos(C_NEAR_PI)   # 2.6906


def _tied_axes(rng, n, pair):
    """Unit axes with n_i = +-n_j for the index pair (i, j) and |n_i| >= |n_k|, so that R_ii = R_jj exactly in fp64 and in
    fp32, and that tie is the largest diagonal once the angle is above 2 pi / 3."""
    a = rng.uniform(0.5, 1.0, n)
    b = rng.uniform(-1.0, 1.0, n) * a
    ax = np.zeros((n, 3))
    i, j = pair
    k = 3 - i - j
    ax[:, i] = a
    ax[:, j] = a * rng.choice([-1.0, 1.0], n)
    ax[:, k] = b
    return ax / np.linalg.norm(ax, axis=-1, keepdims=True)


def _angles(rng, n, lo, hi, log=False):
    if log:
        return np.exp(rng.uniform(math.log(lo), math.log(hi), n))
    return rng.uniform(lo, hi, n)


def fwd_stratum(rng, n, name):
    """fp32 rotations of the named FWD_STRATA entry (fp64 Rodrigues, then rounded)."""
    lo, hi, kind = FWD_STRATA[name]
    axes = unit_axes(rng, n)
    if kind == "zero":
        return np.tile(np.eye(3, dtype=np.float32), (n, 1, 1))
    if kind == "log":
        th = _angles(rng, n, lo, hi, log=True)
    elif kind == "lin":
        th = _angles(rng, n, lo, hi)
    elif kind == "const":
        th = np.full(n, lo)
    elif kind == "cos":            # (tr R - 1)/2 uniform in [lo, hi]
        th = np.arccos(rng.uniform(lo, hi, n))
    elif kind == "pi-":            # pi - delta, delta log-uniform in [lo, hi]
        th = math.pi - _angles(rng, n, lo, hi, log=True)
    elif kind in ("tie01", "tie12"):
        axes = _tied_axes(rng, n, (0, 1) if kind == "tie01" else (1, 2))
        th = _angles(rng, n, lo, hi)
    else:
        raise ValueError(kind)
    return O.rodrigues(axes, th).astype(np.float32)


FWD_STRATA = {  # name -> (lo, hi, kind)
    "theta=0": (0.0, 0.0, "zero"),
    "subnormal skew": (1e-22, 1e-19, "log"),          # |vee(R - R^T)|^2 below FLT_MIN
    "normal tiny": (1e-19, 1e-7, "log"),
    "[1e-7,1e-4]": (1e-7, 1e-4, "log"),
    "[1e-4,1e-2]": (1e-4, 1e-2, "log"),
    "[1e-2,2.6]": (1e-2, 2.6, "lin"),
    "tr=0 (2pi/3)": (-0.5 - 3e-7, -0.5 + 3e-7, "cos"),   # rmat_to_quat: tr R > 0 switch
    "c=-0.9+-1e-4": (C_NEAR_PI - 1e-4, C_NEAR_PI + 1e-4, "cos"),
    "[2.8,3.0]": (2.8, 3.0, "lin"),
    "[3.0,3.1]": (3.0, 3.1, "lin"),
    "[3.1,pi-1e-3]": (3.1, math.pi - 1e-3, "lin"),
    "[pi-1e-3,pi)": (1e-6, 1e-3, "pi-"),
    "theta=pi": (math.pi, math.pi, "const"),
    "R00=R11": (2 * math.pi / 3, math.pi, "tie01"),
    "R11=R22": (2 * math.pi / 3, math.pi, "tie12"),
}


def polar(R):
    """The rotation an fp32 matrix represents: the orthogonal polar factor U V^T of its fp64 value."""
    u, _, vt = np.linalg.svd(np.asarray(R, np.float64))
    return u @ vt


# ---------------------------------------------------------------------------------------------
# the fused reverse step (diffusion.py:291-326): fp64 truth of its mean and the error bound (test_gpu_fwd_strata.py,
# and with the noise factor test_gpu_draws.py)
# ---------------------------------------------------------------------------------------------
AMBIG = 4e-7                  # pi - theta below this: the sign of the axis of an fp32 matrix is not determined

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


def by_stratum(rep, names, label, what, err, tol):
    for i, k in enumerate(names):
        m = label == i
        if m.any():
            rep.add(k, what, err[m], np.broadcast_to(tol, err.shape)[m])


K0, K1, K2 = 16, 8, 8


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


def check_step(rep, names, label, t, got_mean, X, pred, a, b, c1, c2, tag, got_x0=None, noise=None, noise_tol=0.0, per_t=True):
    """The reverse step's output against the fp64 mean (step_tolerance), per t and stratum (per_t=False: per stratum only).
    x_t rows at pi within AMBIG (no defined axis sign) may take either branch of their log, consistently in both uses.
    noise: fp64 rotations the output is the mean times (the step with noise, out = mean @ noise), which add noise_tol.
    Returns the per-row error and tolerance."""
    _, w, th, _ = truth_log(X)
    tol, e0 = step_tolerance(th, a, b, pred, c1, c2)
    tol = tol + noise_tol
    x0, th0, m1, m2 = p_mean_truth(w, pred, a, b, c1, c2)
    if noise is not None:
        m1, m2 = m1 @ noise, m2 @ noise
    near = math.pi - th0 <= e0          # x0_hat within its own error bound of pi: either branch of scale(x0_hat, c1)
    err = np.where(near, np.minimum(O.geodesic_angle(got_mean, m1), O.geodesic_angle(got_mean, m2)), O.geodesic_angle(got_mean, m1))
    e_x0 = O.geodesic_angle(got_x0, x0) if got_x0 is not None else None
    amb = math.pi - th < AMBIG
    if amb.any():
        x0b, th0b, m1b, m2b = p_mean_truth(other_branch(w[amb]), pred[amb], a[amb], b[amb], c1[amb], c2[amb])
        if noise is not None:
            m1b, m2b = m1b @ noise[amb], m2b @ noise[amb]
        nb = math.pi - th0b <= e0[amb]
        eb = np.where(nb, np.minimum(O.geodesic_angle(got_mean[amb], m1b), O.geodesic_angle(got_mean[amb], m2b)), O.geodesic_angle(got_mean[amb], m1b))
        err[amb] = np.minimum(err[amb], eb)
        near[amb] &= nb
        if got_x0 is not None:
            e_x0[amb] = np.minimum(e_x0[amb], O.geodesic_angle(got_x0[amb], x0b))
    groups = [(f" t={tv}", t == tv) for tv in np.unique(t)] if per_t else [("", np.ones(len(t), bool))]
    for gt, m in groups:
        by_stratum(rep, names, label[m], f"{tag}{gt}", err[m], tol[m])
    rep.add("all", f"{tag} rows at x0_hat ~ pi", np.array([near.mean()]), 0.02)
    if got_x0 is not None:
        for gt, m in groups:
            by_stratum(rep, names, label[m], f"{tag} x0_hat{gt}", e_x0[m], e0[m])
    return err, tol
