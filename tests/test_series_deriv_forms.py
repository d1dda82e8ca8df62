"""The series' derivative chain in kappa = 4 sin^2(w/2) (SO3D_SERIES_DERIV=1, the default) and in w (=0, the earlier form),
on the host build of so3d_math.cuh: both against the fp64 oracle, and against each other."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import so3_oracle as O
from tests.test_host_math import _truth, eset, fp

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_math", "host_math.cpp")


@pytest.fixture(scope="module")
def forms(tmp_path_factory):
    d = tmp_path_factory.mktemp("series_deriv")
    libs = {}
    for deriv in (1, 0):
        lib = str(d / f"hm_deriv{deriv}.so")
        subprocess.check_call(["g++", "-O2", "-march=native", "-shared", "-fPIC", f"-DSO3D_SERIES_DERIV={deriv}", "-o", lib, SRC])
        libs[deriv] = ctypes.CDLL(lib)
    return libs


def series(hm, om, eps, L=2000):
    n = om.shape[0]
    F = np.empty(n, np.float32)
    Fp = np.empty(n, np.float32)
    hm.hm_series(fp(om), fp(eps), fp(F), fp(Fp), ctypes.c_long(n), L)
    return F, Fp


def logf_g(hm, om, eps, mode, L=2000):
    n = om.shape[0]
    lf = np.empty(n, np.float32)
    g = np.empty(n, np.float32)
    hm.hm_logf_g(fp(om), fp(eps), fp(lf), fp(g), ctypes.c_long(n), mode, L)
    return lf, g


def test_kappa_form_against_oracle(forms):
    """f and d log f / dw of the kappa form within 1e-5 of fp64 below the conditioning guard (omega <= 4.2 eps), dF/dw
    exactly 0 at omega = 0 (kappa' = 0 there)."""
    n = 20000
    om, eps, _ = eset(n, 31)
    om[:40] = 0.0
    F, Fp = series(forms[1], om, eps)
    ft, gt = _truth(om, eps)
    f = 2.0 * F.astype(np.float64)
    g = Fp.astype(np.float64) / F.astype(np.float64)
    well = om <= 4.2 * eps
    assert np.max(np.abs(f - ft)[well] / ft[well]) < 1e-5
    ok = well & (om > 0)
    assert np.max(np.abs(g - gt)[ok] / np.abs(gt[ok])) < 1e-5
    assert np.all(Fp[om == 0] == 0)


def test_kappa_and_w_forms_agree(forms):
    """F is the same recurrence in both forms (bit-identical); dF/dw differs by rounding only: within 12 float32 ulps of
    |F'| on the E-set below the guard (measured 8.5), 256 beyond it, where the alternating sum's condition number grows
    to ~400 (measured 71).  The guarded modes' closed-form rows are bit-identical."""
    n = 20000
    om, eps, _ = eset(n, 37)
    F1, Fp1 = series(forms[1], om, eps)
    F0, Fp0 = series(forms[0], om, eps)
    assert np.array_equal(F1, F0)
    rel = np.abs(Fp1.astype(np.float64) - Fp0) / np.maximum(np.abs(Fp0.astype(np.float64)), 1e-30) / 2.0 ** -23
    well = (om <= 4.2 * eps) & (om > 0)
    assert rel[well].max() < 12 and rel[om > 0].max() < 256
    for mode in (0, 3):  # series, series_adaptive
        lf1, g1 = logf_g(forms[1], om, eps, mode)
        lf0, g0 = logf_g(forms[0], om, eps, mode)
        guarded = om > 4.2 * eps
        assert np.array_equal(lf1, lf0) and np.array_equal(g1[guarded], g0[guarded])


@pytest.mark.parametrize("L", [1, 2, 33, 100, 2001, 2896])
def test_kappa_form_truncations(forms, L):
    """Short and long truncations: the kappa form's dF/dw against the fp64 derivative of the same truncated series."""
    om, eps, _ = eset(512, 41)
    eps = np.maximum(eps, 0.5).astype(np.float32) if L <= 100 else eps
    F, Fp = series(forms[1], om, eps, L)
    ft, gt = O.igso3_series(om.astype(np.float64), eps.astype(np.float64), L)
    f0, _ = O.igso3_series(np.zeros_like(om, np.float64), eps.astype(np.float64), L)  # sum of |terms| bound
    assert np.max(np.abs(2.0 * F - ft) / f0) < 2e-6
    well = (om <= 4.2 * eps) & (om > 0)
    dF = Fp.astype(np.float64) * 2.0  # f' = 2 F'
    assert np.max(np.abs(dF - gt * ft)[well] / (np.abs(gt * ft)[well] + f0[well] * 1e-3)) < 1e-5
