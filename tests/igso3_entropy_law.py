"""fp64 entropy of the IGSO(3) law and its eps-derivative  --  TEST INFRASTRUCTURE ONLY.

With f the density w.r.t. normalised Haar measure and p(w) = f(w) (1 - cos w) / pi the angle law on [0, pi],
    H(eps) = -int_0^pi p log f dw,        dH/deps = 2 eps E_p[(d log f / dw)^2]   (de Bruijn's identity on SO(3)).
The fp32 code (so3d_math.cuh igso3_entropy) is checked against two independent fp64 forms, each through scipy's quad:

  * entropy_images: the Poisson-dual (image) form in x = w / (2 eps).  With v = eps^2, c0 = (1/2) log pi + v/4 - 3 log eps,
        log f = c0 - x^2 - log sinc(w/2) + log1p(I(w)),   I(w) = sum_{k != 0} (-1)^k (1 + 2 pi k / w) exp(-pi k (w + pi k) / v),
    and x has the density q(x) = (4/sqrt(pi)) e^{v/4} x^2 sinc(w/2) e^{-x^2} (1 + I(w)) of mass 1, so
        H = -c0 + E_q[x^2 + log sinc(w/2) - log1p(I)],   g = d log f / dw = -x/eps + phi(w) + I'/(1 + I).
    The explicit 3 log eps keeps it exact down to eps = 1e-20 and beyond; its images need eps below ~1.5.
  * entropy_series: the series delta-form on [0, pi].  f = 1 + delta, delta = sum_{l>=1} a_l chi_l(w), a_l = (2l+1)
    exp(-l(l+1) v), and E_haar[delta] = 0, so -H = E_haar[(1 + delta) log1p(delta) - delta] with no cancellation as H -> 0-
    (at eps = 3 the image form, like any -int p log f, keeps no digit: -H ~ 1e-15).  It needs eps above ~0.3: below, 1 + delta
    keeps no digit in the upper tail.

`entropy` picks the image form below eps = 1 and the series above.  `entropy_tol` is the error bound of the fp32 code.
"""
from __future__ import annotations

import math

import numpy as np
from scipy import integrate

from tests.igso3_angle_law import _series_terms

HALF_LOG_PI = 0.5 * math.log(math.pi)
QUAD = dict(limit=400, epsabs=1e-16, epsrel=1e-13)


def _phi(w):
    """1/w - cot(w/2)/2, by its Taylor series near 0."""
    return w / 12 + w ** 3 / 720 + w ** 5 / 30240 if w < 1e-2 else 1 / w - 0.5 / math.tan(0.5 * w)


def _log_sinc(t):
    return -t * t / 6 - t ** 4 / 180 if t < 1e-4 else math.log(math.sin(t) / t)


def _images(w, v, K=3):
    """I(w) and I'(w) with images k = +-1 .. +-K."""
    i = di = 0.0
    for k in range(-K, K + 1):
        if k == 0:
            continue
        E = (-1) ** k * math.exp(-math.pi * k * (w + math.pi * k) / v)
        a = 1 + 2 * math.pi * k / w
        i += a * E
        di += (-2 * math.pi * k / (w * w) - a * math.pi * k / v) * E
    return i, di


def entropy_images(eps):
    """(H, dH/deps) of IGSO(3)(eps) by the image form in x = w / (2 eps), fp64 (eps > 0, below ~1.5)."""
    e = abs(float(eps))
    v = e * e
    K = 4 / math.sqrt(math.pi) * math.exp(v / 4)
    top = min(math.pi / (2 * e), 12.0)  # e^{-144} of the mass lies beyond x = 12

    def parts(x):
        w = 2 * e * x
        i, di = _images(w, v)
        ls = _log_sinc(0.5 * w)
        q = K * x * x * math.exp(ls - x * x) * (1 + i)
        g = -x / e + _phi(w) + di / (1 + i)
        return q, x * x + ls - math.log1p(i), g

    s = integrate.quad(lambda x: parts(x)[0] * parts(x)[1], 0, top, **QUAD)[0]
    s2 = integrate.quad(lambda x: parts(x)[0] * parts(x)[2] ** 2, 0, top, **QUAD)[0]
    return -(HALF_LOG_PI + v / 4 - 3 * math.log(e)) + s, 2 * e * s2


def _delta_term(d):
    """(1 + d) log1p(d) - d, by its series where the direct form cancels."""
    if d <= -1.0:  # f below the fp64 rounding of the sum (eps near 0.2, w near pi): f log f -> 0
        return -d
    if abs(d) < 1e-2:
        return d * d * sum((-d) ** (k - 2) / (k * (k - 1)) for k in range(2, 12))
    return (1 + d) * math.log1p(d) - d


def entropy_series(eps):
    """(H, dH/deps) of IGSO(3)(eps) by the series delta-form on [0, pi], fp64 (eps above ~0.2)."""
    e = abs(float(eps))
    l = np.arange(1, _series_terms(e) + 1, dtype=np.float64)
    T = np.cumsum(((2 * l + 1) * np.exp(-l * (l + 1) * e * e))[::-1])[::-1]  # T_m = sum_{l>=m} a_l

    def parts(w):
        delta = T[0] + 2 * np.sum(T * np.cos(l * w))
        ddelta = -2 * np.sum(l * T * np.sin(l * w))
        haar = (1 - math.cos(w)) / math.pi
        return haar, delta, ddelta

    def h_int(w):
        haar, d, _ = parts(w)
        return haar * _delta_term(d)

    def g_int(w):
        haar, d, dd = parts(w)
        return haar * dd * dd / (1 + d) if d > -1.0 else 0.0

    return -integrate.quad(h_int, 0, math.pi, **QUAD)[0], 2 * e * integrate.quad(g_int, 0, math.pi, **QUAD)[0]


def entropy(eps):
    """(H, dH/deps) at |eps| > 0: the image form below 1, the series delta-form from 1 on."""
    e = abs(float(eps))
    return entropy_images(e) if e < 1.0 else entropy_series(e)


def entropy_small_asymptote(eps):
    """eps -> 0+: H = 3 log eps + (3/2) log(4 pi e) - log(8 pi^2) + O(eps^2), the entropy of the tangent Gaussian."""
    return 3 * math.log(eps) + 1.5 * math.log(4 * math.pi * math.e) - math.log(8 * math.pi ** 2)


U32 = 2.0 ** -24
TINY = 2.0 ** -126  # results below FLT_MIN (eps beyond ~4.65) may flush to 0


def entropy_tol(eps, H, dH, c=8.0):
    """Error bound of the fp32 H and dH/deps (DESIGN.md, "IGSO(3) entropy"): c 2^-24 times
      H:       |H| + eps |dH/deps| + [eps <= 1]   (the rounding of log f and of eps^2, with |dH/deps| eps = 8 eps^2 |H| at
               large eps; below eps = 1 an absolute part for the O(1) terms of the sums),
      dH/deps: |dH/deps| (1 + 4 eps^2)           (dH/deps ~ eps e^{-4 eps^2}: eps^2 enters through the exponent),
    plus FLT_MIN for results that leave the normal range."""
    e = abs(float(eps))
    tol_h = c * U32 * (abs(H) + e * abs(dH) + (1.0 if e <= 1.0 else 0.0)) + TINY
    tol_d = c * U32 * abs(dH) * (1 + 4 * e * e) + TINY
    return tol_h, tol_d
