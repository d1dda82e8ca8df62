"""fp64 eps-derivatives of the IGSO(3) rotation-angle law  --  TEST INFRASTRUCTURE ONLY.

The pathwise derivative of the exact sampler's angle, dw/deps of w = F^{-1}(u; eps) at fixed u, is checked against
implicit differentiation in fp64, -(dF/deps)(w) / p(w), with the CDF forms of tests/igso3_angle_law.py:

  * igso3_angle_cdf_deps: dF/deps of the series antiderivative, term by term;
  * igso3_angle_cdf_images_deps: dF/deps of the closed image-sum antiderivative, term by term in v = eps^2 (_dH_dv);
  * igso3_angle_deps: the implicit derivative itself, and deps_tol: the error bound of the fp32 code.
"""
from __future__ import annotations

import math

import numpy as np
from scipy import special

from tests.igso3_angle_law import _H, _images, _series_terms, igso3_angle_pdf


def igso3_angle_cdf_deps(w, eps, L=None):
    """dF/deps at fixed w by the series antiderivative, fp64: pi dF/deps = sum_{l>=1} (a'_l - a'_{l-1}) sin(l w) / l with
    a'_l = -2 eps l (l + 1) a_l (a'_0 = 0).  Loses relative accuracy at small w (the terms are O(w), the sum O(w^3))."""
    w, eps = np.broadcast_arrays(np.asarray(w, dtype=np.float64), np.asarray(eps, dtype=np.float64))
    out = np.empty(w.shape)
    for e in np.unique(eps):
        sel = eps == e
        ww = w[sel]
        n = int(L) if L is not None else _series_terms(e)
        acc = np.zeros(ww.shape)
        da_prev = 0.0
        for l in range(1, n):
            da = -2 * e * l * (l + 1) * (2 * l + 1) * math.exp(-l * (l + 1) * e * e)
            acc += (da - da_prev) / l * np.sin(l * ww)
            da_prev = da
        out[sel] = acc / math.pi
    return out


def _dH_dv(s, v):
    """d_v H(s, v) = int_0^s t sin(t/2) (t^2 / 4v^2) e^{-t^2/4v} dt in closed form.  With e = e^{-t^2/4v},
    t^2 e / 4v^2 = e_tt + e / 2v; two integrations by parts of t sin(t/2) e_tt give
        d_v H = -e(s) [s^2 sin(s/2) / 2v + sin(s/2) + (s/2) cos(s/2)] + Cc(s) + H (1/2v - 1/4),
    Cc(s) = int_0^s cos(t/2) e dt = sqrt(pi v) e^{-v/4} Re erf((s - i v) / (2 sqrt v))."""
    e = np.exp(-s * s / (4 * v))
    cc = np.sqrt(math.pi * v) * np.exp(-v / 4) * special.erf((s - 1j * v) / (2 * np.sqrt(v))).real
    return -e * (s * s * np.sin(s / 2) / (2 * v) + np.sin(s / 2) + 0.5 * s * np.cos(s / 2)) + cc + _H(s, v) * (0.5 / v - 0.25)


def igso3_angle_cdf_images_deps(w, eps):
    """dF/deps at fixed w from the closed image-sum antiderivative, fp64: F = K(v) sum_k [H(w - 2 pi k) - H(-2 pi k)],
    v = eps^2, differentiated term by term (K'/K = 1/4 - 3/(2v), d_v H by _dH_dv), times dv/deps = 2 eps."""
    w, v = np.broadcast_arrays(np.asarray(w, dtype=np.float64), np.asarray(eps, dtype=np.float64) ** 2)
    K = v ** -1.5 * np.exp(v / 4) / math.sqrt(math.pi)
    acc = np.zeros(w.shape)
    dacc = np.zeros(w.shape)
    for k in range(-_images(v), _images(v) + 1):
        s0 = np.full(w.shape, -2 * math.pi * k)
        acc += _H(w - 2 * math.pi * k, v) - _H(s0, v)
        dacc += _dH_dv(w - 2 * math.pi * k, v) - _dH_dv(s0, v)
    return 2 * np.sqrt(v) * K * ((0.25 - 1.5 / v) * acc + dacc)


def igso3_angle_deps(w, eps):
    """The pathwise derivative dw/deps of w = F^{-1}(u; eps) at fixed u, by implicit differentiation at the angle w:
    -(dF/deps)(w) / p(w), fp64, eps > 0, w and eps broadcast.  dF/deps comes from the image sum below eps = 1 and from the
    series at and above it: there the law is within e^{-2 eps^2} of uniform, dF/deps is that small, and the image sum of
    O(1) terms would keep only its absolute 1e-16.  p comes from igso3_angle_pdf."""
    w, eps = np.broadcast_arrays(np.asarray(w, dtype=np.float64), np.asarray(eps, dtype=np.float64))
    dF = np.empty(w.shape)
    img = eps < 1.0
    if img.any():
        dF[img] = igso3_angle_cdf_images_deps(w[img], eps[img])
    if (~img).any():
        dF[~img] = igso3_angle_cdf_deps(w[~img], eps[~img])
    return -dF / igso3_angle_pdf(w, eps)


def deps_tol(w, eps, truth, c=8.0):
    """Error bound of the fp32 dw/deps at (w, eps) (so3d_math.cuh igso3_angle_deps): c 2^-24 (|dw/deps| (1 + 4 eps^2) +
    [eps <= 1] w / eps).  The first term is the rounding of the result plus that of the exponent l (l + 1) eps^2 of the
    weights the series regime (eps > 1) scales by: dw/deps ~ e^{-2 eps^2} there, and an exponent rounded by 2^-24 relative
    moves it by ~4 eps^2 2^-24.  The second is the closed form's cancellation: d log f / dw = -w / (2 eps^2) + ..., whose
    terms are w / eps after the factor -2 eps and cancel towards dw/deps -> 0 at w = pi.  Below eps = 0.3 nothing cancels
    and that term is at most the first."""
    w, eps, truth = (np.asarray(a, dtype=np.float64) for a in (w, eps, truth))
    return c * 2.0 ** -24 * (np.abs(truth) * (1 + 4 * eps * eps) + np.where(np.abs(eps) <= 1.0, w / np.abs(eps), 0.0))
