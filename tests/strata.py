"""Rotation strata and the per-stratum error report shared by the fp64 comparison tests (test_gpu_grad.py,
test_gpu_fwd_strata.py).

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
