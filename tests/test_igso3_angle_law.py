"""CPU tier: the fp64 IGSO(3) angle law the exact sampler is checked against (tests/igso3_angle_law.py), and the fp32
inversion of so3d_math.cuh compiled for the host.

The law's two fp64 CDF forms (series antiderivative, closed image sum) are checked against each other and against
scipy.integrate.quad of the oracle's fp64 density; the inverse against the CDF."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest
from scipy import integrate

from oracle import so3_oracle as O
from tests import igso3_angle_law as A

HERE = os.path.dirname(os.path.abspath(__file__))


def _density(eps):
    if eps <= 0.5:
        return lambda t: float(O.igso3_closed(t, eps)) * (1 - math.cos(t)) / math.pi
    return lambda t: float(O.igso3_series(t, eps)[0][0]) * (1 - math.cos(t)) / math.pi


@pytest.mark.parametrize("eps", [0.001, 0.005, 0.05, 0.5, 2.0, 4.0])
def test_cdf_forms_agree_with_quad_of_the_density(eps):
    ws = np.array([w for w in (0.1, 1.0, 3.0, math.pi, eps, 3 * eps, 6 * eps) if w <= math.pi])
    series = A.igso3_angle_cdf(ws, eps)
    images = A.igso3_angle_cdf_images(ws, eps)
    dens = _density(eps)
    quad = np.array([integrate.quad(dens, 0.0, w, epsabs=1e-14, epsrel=1e-12, limit=400,
                                    points=[p for p in (eps, 3 * eps, 10 * eps) if p < w] or None)[0] for w in ws])
    print(eps, np.abs(series - images).max(), np.abs(series - quad).max())
    assert np.abs(series - images).max() < 1e-12
    assert np.abs(series - quad).max() < 1e-9
    assert abs(A.igso3_angle_cdf(math.pi, eps) - 1.0) < 1e-13
    # the density form agrees with the oracle's density too
    pd = A.igso3_angle_pdf(ws, eps)
    assert np.allclose(pd, [dens(w) for w in ws], rtol=1e-9, atol=1e-300)


def test_icdf_inverts_the_cdf():
    u = np.concatenate([np.logspace(-9, -2, 8), np.linspace(0.05, 0.95, 7), 1 - np.logspace(-2, -7, 6)])
    for eps in (0.001, 0.05, 0.3, 1.0, 4.0):
        w = A.igso3_angle_icdf(u, eps)
        assert np.all((w > 0) & (w <= math.pi))
        assert np.abs(A.igso3_angle_cdf_images(w, eps) - u).max() < 1e-13
        assert np.all(np.diff(w) > 0)
    assert A.igso3_angle_icdf(0.0, 0.1) == 0.0


@pytest.fixture(scope="module")
def hx(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("igso3_exact") / "igso3_exact.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "host_math", "igso3_exact.cpp")])
    return ctypes.CDLL(so)


def _icdf32(hx, u, eps):
    F = ctypes.POINTER(ctypes.c_float)
    u = np.ascontiguousarray(u, np.float32)
    eps = np.ascontiguousarray(np.broadcast_to(np.float32(eps), u.shape), np.float32)
    w = np.empty_like(u)
    hx.hx_igso3_angle_icdf(u.ctypes.data_as(F), eps.ctypes.data_as(F), w.ctypes.data_as(F), ctypes.c_long(u.size))
    return w


def test_host_build_of_the_fp32_inversion(hx):
    u = np.concatenate([np.logspace(-9, -2, 30), np.linspace(0.01, 0.99, 50), 1 - np.logspace(-2, -7.2, 30)]).astype(np.float32)
    for eps in np.float32([1e-3, 0.01, 0.1, 0.29, 0.3, 0.5, 1.0, 4.0]):
        w = _icdf32(hx, u, eps).astype(np.float64)
        assert np.all((w > 0) & (w <= np.float32(math.pi)))
        assert np.abs(A.igso3_angle_cdf_images(w, float(eps)) - u).max() < 1e-6, eps
    # special inputs: u = 0 -> 0, NaN eps / u -> NaN
    w = _icdf32(hx, np.float32([0.0, 0.5, np.nan]), np.float32([0.1, np.nan, 0.1]))
    assert w[0] == 0.0 and np.isnan(w[1]) and np.isnan(w[2])
