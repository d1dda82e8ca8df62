"""CPU tier: the pathwise angle derivative dw/deps of the exact IGSO(3) sampler (so3d_math.cuh igso3_angle_deps, compiled for
the host) against the fp64 law of tests/igso3_angle_law.py and its eps-derivatives in tests/igso3_angle_deps_law.py.

Truth is implicit differentiation at the fp32 angle, -(dF/deps)(w) / p(w) in fp64 (the closed image sum below eps = 1, the
series above), cross-checked against the series form and against central differences of the fp64 inverse CDF at fixed u.
The fp32 code evaluates the same quantity as -2 eps d log f / dw (DESIGN.md, "Reparameterised IGSO(3) sampling"), so these
checks also test that identity.  Tolerance (igso3_angle_deps_law.deps_tol): 8 2^-24 (|dw/deps| (1 + 4 eps^2) + [eps <= 1] w / eps)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from tests import igso3_angle_deps_law as D
from tests import igso3_angle_law as A

HERE = os.path.dirname(os.path.abspath(__file__))
F32P = ctypes.POINTER(ctypes.c_float)
SWITCH = np.float32(0.3)
EPS = np.float32([1e-3, 3e-3, 0.01, 0.03, 0.1, 0.2, np.nextafter(SWITCH, np.float32(0)), SWITCH, np.nextafter(SWITCH, np.float32(1)),
                  0.4, 0.5, 0.7, 1.0, np.nextafter(np.float32(1), np.float32(2)), 1.5, 2.0, 3.0, 4.0])
U = np.concatenate([[1e-9, 2.0 ** -24], np.logspace(-8, -2, 13), np.linspace(0.02, 0.98, 33), 1 - np.logspace(-2, -7, 11)]).astype(np.float32)


@pytest.fixture(scope="module")
def hr(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("igso3_rsample") / "igso3_rsample.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "host_math", "igso3_rsample.cpp")])
    return ctypes.CDLL(so)


def _f32(a, shape=None):
    a = np.asarray(a, np.float32)
    return np.ascontiguousarray(np.broadcast_to(a, shape) if shape is not None else a, np.float32)


def icdf32(hr, u, eps):
    u = _f32(u)
    eps = _f32(eps, u.shape)
    w = np.empty_like(u)
    hr.hr_igso3_angle_icdf(u.ctypes.data_as(F32P), eps.ctypes.data_as(F32P), w.ctypes.data_as(F32P), ctypes.c_long(u.size))
    return w


def deps32(hr, w, eps, u=0.0):
    w = _f32(w)
    eps = _f32(eps, w.shape)
    u = _f32(u, w.shape)
    d = np.empty_like(w)
    hr.hr_igso3_angle_deps(w.ctypes.data_as(F32P), eps.ctypes.data_as(F32P), u.ctypes.data_as(F32P), d.ctypes.data_as(F32P),
                           ctypes.c_long(w.size))
    return d


def test_truth_forms_agree():
    """dF/deps by the image sum and by the series agree where both are accurate, and the truth matches central
    differences of the fp64 inverse CDF at fixed u (fourth-order stencil)."""
    w = np.array([0.05, 0.3, 1.0, 2.0, 3.0])
    for eps in (0.3, 0.5, 0.8, 1.2):
        s, im = D.igso3_angle_cdf_deps(w, eps), D.igso3_angle_cdf_images_deps(w, eps)
        assert np.abs(s - im).max() < 1e-12 * max(1.0, np.abs(s).max()), eps
    u = np.array([1e-7, 1e-3, 0.3, 0.7, 0.99, 1 - 1e-5])
    worst = 0.0
    for eps in (0.002, 0.05, 0.2, 0.3, 0.6, 1.0, 2.0):
        cdf = A.igso3_angle_cdf if eps >= 1.0 else A.igso3_angle_cdf_images
        h = 1e-3 * eps
        q = {k: A.igso3_angle_icdf(u, eps + k * h, cdf) for k in (-2, -1, 1, 2)}
        cd = (8 * (q[1] - q[-1]) - (q[2] - q[-2])) / (12 * h)
        t = D.igso3_angle_deps(A.igso3_angle_icdf(u, eps, cdf), eps)
        rel = np.abs(cd / t - 1).max()
        worst = max(worst, rel)
        assert rel < 5e-6, (eps, rel)
    print(f"central differences vs implicit truth: max rel {worst:.2e}")


def test_host_build_of_the_fp32_derivative(hr):
    """fp32 dw/deps at the fp32 sampler's own angle, eps in [1e-3, 4] (0.3 and 1 with their neighbours), u in [1e-9, 1 - 1e-7]."""
    worst, where = 0.0, None
    for eps in EPS:
        w32 = icdf32(hr, U, eps)
        w = w32.astype(np.float64)
        e = float(eps)
        t = D.igso3_angle_deps(w, e)
        d = deps32(hr, w32, eps).astype(np.float64)
        r = np.abs(d - t) / D.deps_tol(w, e, t)
        i = int(np.argmax(r))
        print(f"eps {e:.9g}: max err/tol {r[i]:.3f} at u {U[i]:.3g} (w {w[i]:.4g}), max rel {np.max(np.abs(d - t) / np.abs(t)):.2e}")
        if r[i] > worst:
            worst, where = r[i], (e, float(U[i]))
        assert np.all(r <= 1.0), (e, U[r > 1.0])
        # odd in eps
        assert np.array_equal(deps32(hr, w32, -eps), -deps32(hr, w32, eps))
    print(f"largest err/tol {worst:.3f} at (eps, u) = {where}")


def _small_angle_slope(eps):
    """lim_{w->0} (dw/deps) / w from the leading term of F = c3(eps) w^3 + O(w^5): dw/deps = -(c3' / 3 c3) w + O(w^3), with
    c3 = f0 / 6 pi, f0 = f(0) = sum_l (2l+1)^2 e^{-l(l+1) eps^2} (fp64, every term positive)."""
    l = np.arange(0, int(math.sqrt(45.0) / eps) + 2, dtype=np.float64)
    a = (2 * l + 1) ** 2 * np.exp(-l * (l + 1) * eps * eps)
    return 2 * eps * np.sum(l * (l + 1) * a) / (3 * np.sum(a))


def test_tiny_angles_keep_relative_accuracy(hr):
    """Down to w = 1e-27 eps, far below what a 24-bit u yields, the relative error stays at the rounding level; w = 0 gives 0."""
    for eps in np.float32([1e-3, 0.1, 0.3, 0.7, 1.5, 4.0]):
        e = float(eps)
        w = (e * np.array([1e-27, 1e-17, 1e-9, 1e-5])).astype(np.float32)
        d = deps32(hr, w, eps).astype(np.float64)
        rel = np.abs(d / (_small_angle_slope(e) * w.astype(np.float64)) - 1)
        print(f"eps {e:.3g}: max rel {rel.max():.2e}")
        assert rel.max() < 8 * 2.0 ** -24 * (1 + 4 * e * e), (e, rel)
        assert deps32(hr, np.float32([0.0]), eps)[0] == 0.0


def test_special_values(hr):
    # eps = 0: the eps -> 0+ limit 2 x0(u), x0 the Maxwell quantile (F(x) = erf x - 2 x e^{-x^2} / sqrt(pi))
    u = np.float32([1e-6, 0.1, 0.5, 0.9, 1 - 1e-6])
    d0 = deps32(hr, np.zeros(5), np.float32(0.0), u).astype(np.float64)
    from scipy import optimize, special
    x0 = np.array([optimize.brentq(lambda x: special.erf(x) - 2 * x * math.exp(-x * x) / math.sqrt(math.pi) - float(uu), 0, 8, xtol=1e-15)
                   for uu in u])
    # x0 is the sampler's fp32 inversion: |F(x0) - u| within the sampler's 2.7e-7 (in the upper tail that is a few 1e-3 of x0)
    xm = d0 / 2
    assert np.abs(special.erf(xm) - 2 * xm * np.exp(-xm * xm) / math.sqrt(math.pi) - u).max() < 3e-7
    assert np.abs(xm / x0 - 1)[:4].max() < 4e-6, xm / x0 - 1
    # ... and the limit of the eps > 0 derivative at the sampled angle
    for eps in np.float32([1e-3, 1e-5]):
        d = deps32(hr, icdf32(hr, u, eps), eps).astype(np.float64)
        assert np.abs(d / d0 - 1)[:4].max() < 1e-5
    # -0.0 takes the same limit; u = 0 gives 0; NaN eps gives NaN
    assert np.array_equal(deps32(hr, np.zeros(5), np.float32(-0.0), u), d0.astype(np.float32))
    assert deps32(hr, np.float32([0.0]), np.float32(0.0), np.float32(0.0))[0] == 0.0
    assert np.isnan(deps32(hr, np.float32([0.5]), np.float32(np.nan))[0])
