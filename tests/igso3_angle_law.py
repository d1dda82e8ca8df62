"""fp64 CDF and inverse CDF of the IGSO(3) rotation-angle law  --  TEST INFRASTRUCTURE ONLY.

The angle of an IGSO(3)(eps) rotation has the density  p(w) = f_eps(w) (1 - cos w) / pi  on [0, pi], f_eps the density of
oracle.so3_oracle.igso3_series / igso3_closed.  This module gives its CDF F(w) in two independent fp64 forms and the
inverse by bracketing plus scipy.optimize.brentq; the exact sampler (ops.igso3_sample_exact) is checked against them.

  * igso3_angle_cdf: the series antiderivative.  With a_l = (2l+1) exp(-l(l+1) eps^2) (the density's series weights) and
    a_0 = 1, f (1 - cos w) = sum_l a_l [cos(l w) - cos((l+1) w)], so
        F(w) = (1/pi) [ w + sum_{l>=1} (a_l - a_{l-1}) sin(l w) / l ],   F(pi) = 1.
  * igso3_angle_cdf_images: the Poisson-dual (image) form of the same law,
        p(w) = K sum_k h(w - 2 pi k),   h(s) = s sin(s/2) exp(-s^2 / 4v),   K = v^{-3/2} exp(v/4) / sqrt(pi),   v = eps^2,
    whose antiderivative is closed: H(s) = int_0^s h = -2v exp(-s^2/4v) sin(s/2) + v sqrt(pi v) exp(-v/4) Re erf((s - i v) / (2 sqrt v)).
    It costs a few complex erf per row at every eps, where the series needs ~6.5/eps terms; the tests use it for large
    batches of small eps and check it against the series.
"""
from __future__ import annotations

import math

import numpy as np
from scipy import optimize, special


def _series_terms(eps):
    """Smallest L with l (l + 1) eps^2 > 45 for l >= L (every further weight is below 1e-17)."""
    return int(math.sqrt(45.0 / (float(eps) ** 2)) + 2)


def igso3_angle_cdf(w, eps, L=None):
    """F_eps(w) by the series antiderivative, fp64.  w and eps broadcast; L terms (default: enough for 1e-16)."""
    w, eps = np.broadcast_arrays(np.asarray(w, dtype=np.float64), np.asarray(eps, dtype=np.float64))
    out = np.empty(w.shape)
    for e in np.unique(eps):
        sel = eps == e
        ww = w[sel]
        n = int(L) if L is not None else _series_terms(e)
        acc = ww.copy()
        a_prev = 1.0
        for l in range(1, n):
            a = (2 * l + 1) * math.exp(-l * (l + 1) * e * e)
            acc += (a - a_prev) / l * np.sin(l * ww)
            a_prev = a
            if a_prev == 0.0:
                break
        out[sel] = acc / math.pi
    return out


def igso3_angle_pdf(w, eps):
    """p_eps(w) = f_eps(w) (1 - cos w) / pi by the image sum, fp64."""
    w, v = np.broadcast_arrays(np.asarray(w, dtype=np.float64), np.asarray(eps, dtype=np.float64) ** 2)
    K = v ** -1.5 * np.exp(v / 4) / math.sqrt(math.pi)
    out = np.zeros(w.shape)
    for k in range(-_images(v), _images(v) + 1):
        s = w - 2 * math.pi * k
        out += s * np.sin(s / 2) * np.exp(-s * s / (4 * v))
    return K * out


def _images(v):
    """Images k with |k| <= this carry everything above 1e-17 of the image sum on [0, pi]."""
    return int(math.ceil((math.sqrt(4 * float(np.max(v)) * 41.0) + math.pi) / (2 * math.pi)))


def _H(s, v):
    z = (s - 1j * v) / (2 * np.sqrt(v))
    return -2 * v * np.exp(-s * s / (4 * v)) * np.sin(s / 2) + v * np.sqrt(math.pi * v) * np.exp(-v / 4) * special.erf(z).real


def igso3_angle_cdf_images(w, eps):
    """F_eps(w) by the closed antiderivative of the image sum, fp64 (complex erf)."""
    w, v = np.broadcast_arrays(np.asarray(w, dtype=np.float64), np.asarray(eps, dtype=np.float64) ** 2)
    K = v ** -1.5 * np.exp(v / 4) / math.sqrt(math.pi)
    acc = np.zeros(w.shape)
    for k in range(-_images(v), _images(v) + 1):
        acc += _H(w - 2 * math.pi * k, v) - _H(np.full(w.shape, -2 * math.pi * k), v)
    return K * acc


def igso3_angle_icdf(u, eps, cdf=igso3_angle_cdf_images):
    """w = F_eps^{-1}(u) in [0, pi] by bracketing and brentq, fp64.  u and eps broadcast."""
    u, eps = np.broadcast_arrays(np.asarray(u, dtype=np.float64), np.asarray(eps, dtype=np.float64))
    out = np.empty(u.shape)
    for idx in np.ndindex(u.shape):
        uu, e = float(u[idx]), float(eps[idx])
        if uu <= 0.0:
            out[idx] = 0.0
            continue
        if uu >= 1.0:
            out[idx] = math.pi
            continue
        # bracket: grow hi from the small-eps scale until F(hi) >= u
        hi = min(math.pi, 4.0 * e)
        while hi < math.pi and cdf(hi, e) < uu:
            hi = min(math.pi, 2.0 * hi)
        out[idx] = optimize.brentq(lambda x: float(cdf(x, e)) - uu, 0.0, hi, xtol=1e-15, rtol=1e-14, maxiter=200)
    return out
