"""CPU tier: the IGSO(3) entropy and its eps-derivative (so3d_math.cuh igso3_entropy, compiled for the host) against the fp64
law of tests/igso3_entropy_law.py.

The two fp64 forms (image form in x = w / (2 eps), series delta-form) are checked against each other, de Bruijn's identity
against central differences of H, and the small-eps limit against the entropy of the tangent Gaussian.  Tolerance
(igso3_entropy_law.entropy_tol, c = 8): 8 2^-24 (|H| + eps |dH/deps| + [eps <= 1]) for H, 8 2^-24 |dH/deps| (1 + 4 eps^2)
for dH/deps, plus FLT_MIN."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from tests import igso3_entropy_law as E

HERE = os.path.dirname(os.path.abspath(__file__))
F32P = ctypes.POINTER(ctypes.c_float)


def _around(x):
    x = np.float32(x)
    return [np.nextafter(x, np.float32(0)), x, np.nextafter(x, np.float32(10))]


EPS = np.float32(np.concatenate([np.logspace(-20, math.log10(6.0), 160), _around(0.3), _around(1.0)]))


@pytest.fixture(scope="module")
def hr(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("igso3_entropy") / "igso3_entropy.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "host_math", "igso3_entropy.cpp")])
    return ctypes.CDLL(so)


def entropy32(hr, eps):
    eps = np.ascontiguousarray(eps, np.float32)
    H, d = np.empty_like(eps), np.empty_like(eps)
    hr.hr_igso3_entropy(eps.ctypes.data_as(F32P), H.ctypes.data_as(F32P), d.ctypes.data_as(F32P), ctypes.c_long(eps.size))
    return H.astype(np.float64), d.astype(np.float64)


def test_truth_forms_agree():
    for eps in (0.3, 0.5, 0.8, 1.0, 1.2, 1.5):
        (hi, di), (hs, ds) = E.entropy_images(eps), E.entropy_series(eps)
        assert abs(hi - hs) < 1e-13 * max(1.0, abs(hs)) + 1e-15, (eps, hi, hs)
        assert abs(di / ds - 1) < 1e-12, (eps, di, ds)


def test_de_bruijn_matches_central_difference():
    for eps in (0.01, 0.05, 0.1, 0.3, 0.5, 1.0, 2.0):
        h = 1e-5 * eps
        cd = (E.entropy(eps + h)[0] - E.entropy(eps - h)[0]) / (2 * h)
        d = E.entropy(eps)[1]
        assert abs(cd / d - 1) < 5e-8, (eps, cd, d)


def test_limits():
    # eps -> 0+: the tangent Gaussian, H - asymptote = O(eps^2), dH/deps -> 3/eps
    for eps in (1e-3, 1e-2):
        H, d = E.entropy(eps)
        assert abs(H - E.entropy_small_asymptote(eps)) < eps * eps, eps
        assert abs(d * eps / 3 - 1) < eps * eps, eps
    # eps large: -H ~ (9/2) e^{-4 eps^2} (the l = 1 term; the next is e^{-8 eps^2} smaller)
    for eps in (2.0, 2.5, 3.0):
        H, _ = E.entropy(eps)
        assert abs(-H / (4.5 * math.exp(-4 * eps * eps)) - 1) < 1e-3, eps


def test_host_build_of_the_fp32_entropy(hr):
    """eps on a log grid over [1e-20, 6], plus 0.3 and 1 with their fp32 neighbours."""
    H, d = entropy32(hr, EPS)
    worst_h = worst_d = 0.0
    for e, h, dd in zip(EPS.astype(np.float64), H, d):
        th, td = E.entropy(e)
        tol_h, tol_d = E.entropy_tol(e, th, td)
        rh, rd = abs(h - th) / tol_h, abs(dd - td) / tol_d
        assert rh <= 1.0 and rd <= 1.0, (e, h, th, dd, td)
        worst_h, worst_d = max(worst_h, rh), max(worst_d, rd)
    print(f"largest err/tol: H {worst_h:.3f}, dH/deps {worst_d:.3f}")
    # even / odd in eps
    Hn, dn = entropy32(hr, -EPS)
    assert np.array_equal(Hn, H) and np.array_equal(dn, -d)


def test_special_values(hr):
    H, d = entropy32(hr, np.float32([0.0, -0.0, np.nan, np.inf, -np.inf, 8.0]))
    assert H[0] == -np.inf and d[0] == np.inf
    assert H[1] == -np.inf and d[1] == np.inf
    assert np.isnan(H[2]) and np.isnan(d[2])
    assert np.all(H[3:] == 0.0) and np.all(d[3:] == 0.0)
