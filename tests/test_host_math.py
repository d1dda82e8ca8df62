"""CPU-tier check of the per-rotation arithmetic the sm_100a kernels inline.

diffusion_extensions_b200/csrc/so3d_math.cuh is host+device; tests/host_math/host_math.cpp compiles
it with g++ so that, in the GPU-less build container, the same code is compared with the oracle.
(The GPU tier repeats these comparisons through the real kernels and the C-ABI.)
"""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import so3_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_math", "host_math.cpp")
LIB = os.path.join(HERE, "host_math", "_host_math.so")
HDR = os.path.join(HERE, "..", "diffusion_extensions_b200", "csrc", "so3d_math.cuh")

F = ctypes.POINTER(ctypes.c_float)
D = ctypes.POINTER(ctypes.c_double)


def fp(a):
    return a.ctypes.data_as(F)


@pytest.fixture(scope="module")
def hm():
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        subprocess.check_call(["g++", "-O2", "-march=native", "-shared", "-fPIC", "-o", LIB, SRC])
    return ctypes.CDLL(LIB)


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def rand_rots(n, seed, max_angle=math.pi):
    rng = np.random.default_rng(seed)
    R, axis, ang = O.random_rotations(n, rng, max_angle)
    return f32(R), axis, ang


def test_axis_angle_and_log(hm):
    n = 4096
    R, _, _ = rand_rots(n, 0)
    axis = np.empty((n, 3), np.float32); ang = np.empty(n, np.float32); v = np.empty((n, 3), np.float32)
    hm.hm_axis_angle(fp(R), fp(axis), fp(ang), ctypes.c_long(n))
    hm.hm_log_vec(fp(R), fp(v), ctypes.c_long(n))
    ax_t, ang_t = O.rmat_to_aa(R)
    assert np.max(np.abs(ang - ang_t[:, 0])) < 1e-6
    # axis error allowed to grow only near pi (sign flips at pi are legitimate) -> compare rotations
    back = O.rodrigues(axis.astype(np.float64), ang.astype(np.float64))
    assert np.max(np.abs(back - R)) < 2e-6
    assert np.max(np.abs(v - O.log_vec(R))[ang_t[:, 0] < 3.1]) < 3e-6


def test_log_edge_cases(hm):
    # identity, exact pi about generic axes, tiny angles
    rng = np.random.default_rng(3)
    ax = rng.standard_normal((64, 3)); ax /= np.linalg.norm(ax, axis=-1, keepdims=True)
    Rpi = f32(O.rodrigues(ax, np.full(64, math.pi)))
    Rtiny = f32(O.rodrigues(ax, np.full(64, 1e-5)))
    R = np.concatenate([f32(np.eye(3))[None], Rpi, Rtiny])
    n = R.shape[0]
    axis = np.empty((n, 3), np.float32); ang = np.empty(n, np.float32)
    hm.hm_axis_angle(fp(R), fp(axis), fp(ang), ctypes.c_long(n))
    assert ang[0] == 0 and np.array_equal(axis[0], [0, 0, 1])
    assert np.max(np.abs(ang[1:65] - math.pi)) < 1e-6
    # axis at pi is defined up to sign (Q4: the reference gets it wrong; fp64 truth is +-ax)
    dots = np.abs((axis[1:65] * ax).sum(-1))
    assert np.min(dots) > 1 - 1e-6
    assert np.max(np.abs(ang[65:] - 1e-5)) < 1e-9
    assert np.min((axis[65:] * ax).sum(-1)) > 1 - 1e-5


def test_exp_scale_quat(hm):
    n = 2048
    rng = np.random.default_rng(1)
    R, _, _ = rand_rots(n, 1, 3.0)
    axes = f32(rng.standard_normal((n, 3)) * 2); ang = f32(rng.uniform(0, math.pi, n))
    out = np.empty((n, 3, 3), np.float32)
    hm.hm_aa_to_rmat(fp(axes), fp(ang), fp(out), ctypes.c_long(n))
    assert np.max(np.abs(out - O.aa_to_rmat(axes, ang[:, None]))) < 1e-6
    v = f32(rng.standard_normal((n, 3)) * np.exp(rng.uniform(-12, 1, (n, 1))))
    hm.hm_exp_vec(fp(v), fp(out), ctypes.c_long(n))
    assert np.max(np.abs(out - O.exp_vec(v))) < 1e-6
    s = f32(np.exp(rng.uniform(math.log(1e-4), math.log(3.0), n)))
    hm.hm_scale(fp(R), fp(s), fp(out), ctypes.c_long(n))
    assert np.max(np.abs(out - O.so3_scale(R, s))) < 3e-6
    q = f32(rng.standard_normal((n, 4)))
    hm.hm_quat_to_rmat(fp(q), fp(out), ctypes.c_long(n))
    assert np.max(np.abs(out - O.quat_to_rmat(q))) < 1e-6
    q2 = np.empty((n, 4), np.float32)
    hm.hm_rmat_to_quat(fp(R), fp(q2), ctypes.c_long(n))
    assert np.max(np.abs(np.linalg.norm(q2, axis=-1) - 1)) < 1e-6 and np.all(q2[:, 0] >= 0)
    assert np.max(np.abs(O.quat_to_rmat(q2) - R)) < 2e-6


def test_l0_maps_on_lean_primitives(hm):
    """The forward L0 kernels (log / exp / so3_scale) run the branch-free quaternion primitives: same tolerances
    against the fp64 oracle as the general-purpose versions above, including identity, pi and tiny angles."""
    n = 4096
    rng = np.random.default_rng(11)
    R, _, ang_t = rand_rots(n, 12)
    v = np.empty((n, 3), np.float32)
    hm.hm_log_vec_fast(fp(R), fp(v), ctypes.c_long(n))
    assert np.max(np.abs(v - O.log_vec(R))[ang_t < 3.1]) < 3e-6
    assert np.max(np.abs(np.linalg.norm(v, axis=-1) - ang_t)) < 2e-6
    ax = rng.standard_normal((64, 3)); ax /= np.linalg.norm(ax, axis=-1, keepdims=True)
    Re = np.concatenate([f32(np.eye(3))[None], f32(O.rodrigues(ax, np.full(64, math.pi))), f32(O.rodrigues(ax, np.full(64, 1e-5)))])
    ve = np.empty((129, 3), np.float32)
    hm.hm_log_vec_fast(fp(Re), fp(ve), ctypes.c_long(129))
    assert np.array_equal(ve[0], [0, 0, 0])
    assert np.max(np.abs(np.linalg.norm(ve[1:65], axis=-1) - math.pi)) < 2e-6
    assert np.min(np.abs((ve[1:65] / math.pi * ax).sum(-1))) > 1 - 1e-6          # axis at pi: defined up to sign
    assert np.max(np.abs(ve[65:] - 1e-5 * ax)) < 1e-9
    w = f32(rng.standard_normal((n, 3)) * np.exp(rng.uniform(-12, 1, (n, 1))))
    out = np.empty((n, 3, 3), np.float32)
    hm.hm_exp_vec_fast(fp(w), fp(out), ctypes.c_long(n))
    assert np.max(np.abs(out - O.exp_vec(w))) < 1e-6
    R3, _, _ = rand_rots(n, 13, 3.0)
    s = f32(np.exp(rng.uniform(math.log(1e-4), math.log(3.0), n)))
    hm.hm_scale_fast(fp(R3), fp(s), fp(out), ctypes.c_long(n))
    assert np.max(np.abs(out - O.so3_scale(R3, s))) < 3e-6


def eset(n, seed, kmax=4.0):
    rng = np.random.default_rng(seed)
    eps = np.exp(rng.uniform(math.log(6.4e-3), 0.0, n)).astype(np.float32)
    k = rng.uniform(0, kmax, n)
    om = np.minimum(eps * math.sqrt(2.0) * k, 3.0).astype(np.float32)
    return om, eps, om / (math.sqrt(2.0) * eps)


def _truth(om, eps):
    """fp64 truth: the series where it is well conditioned in fp64, the stable closed form (3 images,
    <= 4e-9 of the series for eps < 1, tests/test_oracle_golden.py) for small eps far in the tail."""
    om64, e64 = om.astype(np.float64), eps.astype(np.float64)
    ft, gt = O.igso3_series(om64, e64)
    # (the fp64 closed-form derivative itself cancels like 1/w - cot(w/2)/2 at small w: series there)
    small = (e64 < 0.4) & (om64 > 3.0 * e64)
    ft = np.where(small, O.igso3_closed(om64, e64), ft)
    gt = np.where(small, O.igso3_closed_dlog(om64, e64), gt)
    return ft, gt


@pytest.mark.parametrize("mode", [1, 2])
def test_closed_and_auto_fp32(hm, mode):
    """fp32 closed form (eps <= 1) and the auto evaluator (any eps) vs fp64 truth on the E-set
    (omega = eps sqrt2 k, k in [0,4], clipped to 3.0): <= 1e-5 relative on density and score."""
    n = 40000
    om, eps, k = eset(n, 5)
    if mode == 2:  # auto also covers eps > 1 where the 3-image closed form breaks down
        eps[: n // 4] = np.random.default_rng(6).uniform(1.0, 2.0, n // 4).astype(np.float32)
        om[: n // 4] = np.minimum(om[: n // 4], 3.0)
    om[:50] = 0.0
    om[50:100] = np.float32(1e-7)
    logf = np.empty(n, np.float32); g = np.empty(n, np.float32)
    hm.hm_logf_g(fp(om), fp(eps), fp(logf), fp(g), ctypes.c_long(n), mode, 2000)
    ft, gt = _truth(om, eps)
    assert np.max(np.abs(np.exp(logf.astype(np.float64) - np.log(ft)) - 1)) < 1e-5
    ok = om > 0
    assert np.max((np.abs(g - gt) / np.maximum(np.abs(gt), 1e-30))[ok]) < 1e-5
    assert np.all(g[~ok] == 0)


def test_auto_full_angle_range(hm):
    """omega over all of [0, pi]: density <= 1e-5 relative; the score goes through zero at pi
    (f is symmetric about pi), so there its error is measured against the score scale 1/eps."""
    n = 40000
    rng = np.random.default_rng(8)
    eps = np.exp(rng.uniform(math.log(0.15), math.log(2.0), n)).astype(np.float32)  # f(pi) > 1e-48: fp64 truth exists
    om = rng.uniform(0, math.pi, n).astype(np.float32)
    om[:64] = np.float32(math.pi)
    logf = np.empty(n, np.float32); g = np.empty(n, np.float32)
    hm.hm_logf_g(fp(om), fp(eps), fp(logf), fp(g), ctypes.c_long(n), 2, 2000)
    ft, gt = _truth(om, eps)
    assert np.max(np.abs(np.exp(logf.astype(np.float64) - np.log(ft)) - 1)) < 2e-5
    assert np.max(np.abs(g - gt) / np.maximum(np.abs(gt), 1.0 / eps)) < 1e-5


def test_series_fp32(hm):
    """The raw fp32 L=2000 series (character form, Reinsch-Clenshaw recurrence; mode "series_pure") vs the fp64
    series.  1e-5 while the alternating sum is well conditioned (cond <= 14: omega <= 4.2 eps, k <= 2.97); beyond
    that the error of ANY fp32 summation grows like ~4 u cond (oracle/proto_series_fp32.py): measured bounds."""
    n = 6000
    om, eps, k = eset(n, 7)
    om[:20] = 0.0
    k[:20] = 0.0
    F = np.empty(n, np.float32); Fp = np.empty(n, np.float32)
    hm.hm_series(fp(om), fp(eps), fp(F), fp(Fp), ctypes.c_long(n), 2000)
    ft, gt = _truth(om, eps)
    f = 2.0 * F.astype(np.float64)
    g = Fp.astype(np.float64) / F.astype(np.float64)  # hm_series returns dF/dw in its second output
    ef = np.abs(f - ft) / ft
    eg = np.abs(g - gt) / np.maximum(np.abs(gt), 1e-30)
    well = om <= 4.2 * eps
    assert ef[well].max() < 1e-5 and eg[well & (om > 0)].max() < 1e-5
    assert np.all(g[om == 0] == 0)
    assert ef[k <= 3.5].max() < 3e-5 and ef.max() < 2e-4 and eg[om > 0].max() < 2e-4


@pytest.mark.parametrize("mode", [0, 3])
def test_series_guarded_meets_north_star_on_whole_eset(hm, mode):
    """Modes "series" / "series_adaptive": every row runs its L terms, rows with omega > 4.2 eps (eps <= 1) are then
    replaced by the closed form -> density AND score <= 1e-5 relative on the whole E-set (k <= 4), and the guard does
    not touch the rows below it (bit-identical to the raw series there)."""
    n = 40000
    om, eps, k = eset(n, 21)
    om[:50] = 0.0
    logf = np.empty(n, np.float32); g = np.empty(n, np.float32)
    hm.hm_logf_g(fp(om), fp(eps), fp(logf), fp(g), ctypes.c_long(n), mode, 2000)
    ft, gt = _truth(om, eps)
    assert np.max(np.abs(np.exp(logf.astype(np.float64) - np.log(ft)) - 1)) < 1e-5
    ok = om > 0
    assert np.max((np.abs(g - gt) / np.maximum(np.abs(gt), 1e-30))[ok]) < 1e-5
    lp = np.empty(n, np.float32); gp = np.empty(n, np.float32)
    hm.hm_logf_g(fp(om), fp(eps), fp(lp), fp(gp), ctypes.c_long(n), 4, 2000)
    below = om <= 4.2 * eps
    assert np.array_equal(lp[below], logf[below]) and np.array_equal(gp[below], g[below])
    assert (~below).mean() > 0.2      # the guard is exercised: ~26 % of the E-set


def test_series_short_L(hm):
    om, eps, _ = eset(512, 9)
    eps = np.maximum(eps, 0.5).astype(np.float32)
    for L in (1, 2, 31, 32, 33, 64, 100):
        F = np.empty(512, np.float32); Fp = np.empty(512, np.float32)
        hm.hm_series(fp(om), fp(eps), fp(F), fp(Fp), ctypes.c_long(512), L)
        ft, gt = O.igso3_series(om.astype(np.float64), eps.astype(np.float64), L)
        f0, _ = O.igso3_series(np.zeros_like(om, np.float64), eps.astype(np.float64), L)  # sum of |terms| bound
        assert np.max(np.abs(2.0 * F - ft) / f0) < 2e-6, L


def test_table_density_f64(hm, golden):
    g = golden("igso3")
    loc = g["grid_loc"].astype(np.float64)
    for e, ref in zip(g["eps_list"], g["trap"]):
        f = np.empty(1000, np.float64)
        ee = np.full(1000, float(e))
        hm.hm_closed_f64(loc.ctypes.data_as(D), ee.ctypes.data_as(D), f.ctypes.data_as(D), ctypes.c_long(1000), 0)
        assert np.max(np.abs(f - O.igso3_closed(loc, float(e))) / np.maximum(O.igso3_closed(loc, float(e)), 1e-300)) < 1e-10
    # quirk mode reproduces the reference's zeroed tail at the schedule's smallest eps
    om = g["q_omega"].astype(np.float64)
    f = np.empty(om.shape[0], np.float64)
    ee = np.full(om.shape[0], float(g["q_eps"]))
    hm.hm_closed_f64(om.ctypes.data_as(D), ee.ctypes.data_as(D), f.ctypes.data_as(D), ctypes.c_long(om.shape[0]), 1)
    assert np.array_equal(f[1:] == 0, g["q_density"][1:] == 0)


def test_inverse_cdf_lookup(hm, golden):
    g = golden("igso3")
    loc = f32(g["trap_loc"])
    for k in range(len(g["eps_list"])):
        trap = f32(g["trap"][k]); u = f32(g["u_draw"][k])
        ang = np.empty(u.shape[0], np.float32)
        hm.hm_angle_from_uniform(fp(trap), fp(loc), fp(u), fp(ang), ctypes.c_long(u.shape[0]))
        want = O.igso3_angle_from_uniform(u, trap, loc)
        assert np.max(np.abs(ang - want)) <= 1e-7   # same fp32 arithmetic; FMA contraction only
        ref_ang = O.rmat_to_aa(g["samples"][k])[1][:, 0]
        assert np.max(np.abs(ang - ref_ang)) < 1e-5  # vs the reference's own samples (north star)
    # edge uniforms
    trap = f32(g["trap"][2])
    u = f32([0.0, 1e-12, trap[0], trap[10], np.nextafter(np.float32(1), np.float32(0)), 1.0])
    ang = np.empty(u.shape[0], np.float32)
    hm.hm_angle_from_uniform(fp(trap), fp(loc), fp(u), fp(ang), ctypes.c_long(u.shape[0]))
    want = O.igso3_angle_from_uniform(u[:-1], trap, loc)
    assert np.max(np.abs(ang[:-1] - want)) <= 1e-7 and np.isfinite(ang[-1])


def test_inverse_cdf_guide_records(hm, golden):
    """The 16-byte guide records resolve the lookup to exactly the index (hence the angle) of the full search,
    for random uniforms, bucket edges, CDF values themselves and their float neighbours."""
    g = golden("igso3")
    loc = f32(g["trap_loc"])
    rng = np.random.default_rng(33)
    for k in range(len(g["eps_list"])):
        trap = f32(g["trap"][k])
        edges = np.arange(1024, dtype=np.float32) / np.float32(1024)
        # the float-format buckets of the two tails: 64 per octave of u (and of 1 - u) down to 2^-13, and far below
        log_edges = (np.float32(2.0) ** -np.arange(3, 33, dtype=np.float32))[:, None] * (1 + np.arange(64, dtype=np.float32) / 64)[None, :]
        log_edges = log_edges.reshape(-1).astype(np.float32)
        up_edges = (np.float32(1) - log_edges[log_edges >= 2.0 ** -24]).astype(np.float32)
        tiny = (rng.integers(0, 2 ** 20, 4000).astype(np.float64) * 2.0 ** -32).astype(np.float32)   # the generator's lattice near 0
        near1 = (np.float32(1) - rng.integers(1, 2 ** 12, 4000).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)
        special = np.concatenate([edges, log_edges, up_edges, trap[:-1], f32([0.0, 0.125, 0.875])])
        u = np.concatenate([rng.random(20000, dtype=np.float32), tiny, near1, special, np.nextafter(special, np.float32(0)),
                            np.nextafter(special, np.float32(1)), f32([np.nextafter(np.float32(1), np.float32(0))])]).astype(np.float32)
        u = np.ascontiguousarray(u[(u >= 0) & (u < 1)])
        a = np.empty(u.shape[0], np.float32); b = np.empty(u.shape[0], np.float32)
        hm.hm_angle_from_uniform(fp(trap), fp(loc), fp(u), fp(a), ctypes.c_long(u.shape[0]))
        hm.hm_angle_from_record(fp(trap), fp(loc), fp(u), fp(b), ctypes.c_long(u.shape[0]))
        assert np.array_equal(a, b)
        # every u lies in the range its record was built for; records are ordered; the search path is rare
        kk = np.empty(u.shape[0], np.int32); lo = np.empty_like(a); hi = np.empty_like(a); one = np.empty(u.shape[0], np.int32)
        ip = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_int))
        hm.hm_guide_bucket(fp(trap), fp(u), ip(kk), fp(lo), fp(hi), ip(one), ctypes.c_long(u.shape[0]))
        assert kk.min() >= 0 and kk.max() < hm.hm_guide_records() == 2051
        assert np.all(lo <= u) and np.all(u <= hi)
        order = np.argsort(u, kind="stable")
        us, ks = u[order], kk[order]
        assert np.all(np.diff(ks[us <= 0.875]) >= 0) and np.all(np.diff(ks[us > 0.875]) <= 0)   # the upper tail counts down from 1
        assert ks[us <= 0.875].max() < ks[us > 0.875].min()
        assert one[:20000].mean() > 0.985   # (uniform 1/1024 buckets: 0.93-0.95)
        # the shared-memory guide of the shared-row kernels (uint16 counts at sg_edge): same index as the full search, every u
        # inside its bucket's edges, edges non-decreasing
        nb = hm.hm_sg_buckets()
        assert nb == 1282
        edges_sg = np.empty(nb + 1, np.float32)
        hm.hm_sg_edges(fp(edges_sg))
        assert edges_sg[0] == 0 and edges_sg[-1] == 1 and np.all(np.diff(edges_sg) >= 0)
        us = np.ascontiguousarray(np.concatenate([u, edges_sg[:-1], np.nextafter(edges_sg[1:], np.float32(0))]).astype(np.float32))
        us = np.ascontiguousarray(us[(us >= 0) & (us < 1)])
        a2 = np.empty(us.shape[0], np.float32); c2 = np.empty(us.shape[0], np.float32)
        bk = np.empty(us.shape[0], np.int32); op1 = np.empty(us.shape[0], np.int32)
        hm.hm_angle_from_uniform(fp(trap), fp(loc), fp(us), fp(a2), ctypes.c_long(us.shape[0]))
        hm.hm_angle_from_smem_guide(fp(trap), fp(loc), fp(us), fp(c2), ip(bk), ip(op1), ctypes.c_long(us.shape[0]))
        assert np.array_equal(a2, c2)
        assert bk.min() >= 0 and bk.max() < nb
        assert np.all(edges_sg[bk] <= us) and np.all(us <= edges_sg[bk + 1])
        assert op1[:20000].mean() > 0.97   # (1024 uniform buckets: 0.93-0.95)
    # out-of-range and non-finite inputs land on a valid record (and take the full search)
    bad = f32([-1.0, -0.0, 1.0, 2.0, 1e30, -1e30, np.inf, -np.inf, np.nan])
    kk = np.empty(bad.shape[0], np.int32); lo = np.empty_like(bad); hi = np.empty_like(bad); one = np.empty(bad.shape[0], np.int32)
    hm.hm_guide_bucket(fp(trap), fp(bad), ip(kk), fp(lo), fp(hi), ip(one), ctypes.c_long(bad.shape[0]))
    assert kk.min() >= 0 and kk.max() < 2051


def test_philox_known_answer_and_draws(hm):
    # Random123 known-answer test for philox4x32-10: counter = key = 0 and the "pi" vector
    out = np.empty(4, np.uint32)
    hm.hm_philox(ctypes.c_ulonglong(0), ctypes.c_ulonglong(0), ctypes.c_ulonglong(0), out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), ctypes.c_long(1))
    assert [hex(x) for x in out] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    seed = (0xa4093822 | (0x299f31d0 << 32))
    row = (0x243f6a88 | (0x85a308d3 << 32))
    off = (0x13198a2e | (0x03707344 << 32))
    hm.hm_philox(ctypes.c_ulonglong(seed), ctypes.c_ulonglong(row), ctypes.c_ulonglong(off), out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), ctypes.c_long(1))
    assert [hex(x) for x in out] == ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]
    # precomputed key schedule == plain generator, including 64-bit rows / offsets and the SE(3) stream bit
    rng = np.random.default_rng(9)
    for seed, row0, off in [(0, 0, 0), (1234, 2**32 - 3, 7), (2**64 - 1, 2**40 + 5, 2**63 | 12345), (int(rng.integers(0, 2**62)), int(rng.integers(0, 2**62)), int(rng.integers(0, 2**62)))]:
        a = np.empty(4 * 64, np.uint32); b = np.empty(4 * 64, np.uint32)
        hm.hm_philox(ctypes.c_ulonglong(seed), ctypes.c_ulonglong(row0), ctypes.c_ulonglong(off), a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), ctypes.c_long(64))
        hm.hm_philox_keyed(ctypes.c_ulonglong(seed), ctypes.c_ulonglong(row0), ctypes.c_ulonglong(off), b.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), ctypes.c_long(64))
        assert np.array_equal(a, b)
    n = 200000
    axis = np.empty((n, 3), np.float32); u = np.empty(n, np.float32)
    hm.hm_draw(ctypes.c_ulonglong(1234), ctypes.c_ulonglong(0), ctypes.c_ulonglong(0), fp(axis), fp(u), ctypes.c_long(n))
    assert np.max(np.abs(np.linalg.norm(axis, axis=-1) - 1)) < 1e-6
    assert np.all((u >= 0) & (u < 1))
    assert np.max(np.abs(axis.mean(0))) < 0.01 and abs(u.mean() - 0.5) < 0.01
    assert np.max(np.abs((axis ** 2).mean(0) - 1 / 3)) < 0.01


def test_backward_pieces(hm):
    """Closed-form backward of log / aa_to_rmat / exp against central differences of the oracle."""
    n = 256
    rng = np.random.default_rng(11)
    R, _, _ = rand_rots(n, 11, 2.8)
    G = f32(rng.standard_normal((n, 3, 3)))
    out = np.empty((n, 3, 3), np.float32)
    hm.hm_log_bwd(fp(R), fp(G), fp(out), ctypes.c_long(n))
    h = 1e-6
    num = np.zeros((n, 3, 3))
    R64 = R.astype(np.float64)
    for i in range(3):
        for j in range(3):
            d = np.zeros((3, 3)); d[i, j] = h
            lp = O.log_rmat(R64 + d, reference_quirks=True); lm = O.log_rmat(R64 - d, reference_quirks=True)
            num[:, i, j] = ((lp - lm) * G).sum((-1, -2)) / (2 * h)
    assert np.max(np.abs(out - num) / np.maximum(np.abs(num).max((-1, -2), keepdims=True), 1.0)) < 2e-4
    # near pi: the tangent part vee_adj(R^T g) is the derivative of log along R exp(hat(xi)), Jr^-T(phi) vee_adj(G),
    # to ~2^-24/sin(theta) (the reference formula's own tangent part is off by ~2^-24/sin^2(theta) on an fp32 matrix)
    th = rng.uniform(2.6, math.pi - 1e-3, n)
    ax = rng.standard_normal((n, 3)); ax /= np.linalg.norm(ax, axis=-1, keepdims=True)
    Rp = f32(O.rodrigues(ax, th))
    hm.hm_log_bwd(fp(Rp), fp(G), fp(out), ctypes.c_long(n))
    vadj = lambda m: np.stack((m[..., 2, 1] - m[..., 1, 2], m[..., 0, 2] - m[..., 2, 0], m[..., 1, 0] - m[..., 0, 1]), -1)
    phi = O.log_vec(Rp.astype(np.float64))
    t = np.linalg.norm(phi, axis=-1, keepdims=True)
    nn_, u = phi / t, vadj(G.astype(np.float64))
    nu = np.cross(nn_, u)
    want = u - t / 2 * nu + (1 - (t / 2) * np.sin(t) / (2 * np.sin(t / 2) ** 2)) * np.cross(nn_, nu)
    tau = vadj(np.swapaxes(Rp.astype(np.float64), -1, -2) @ out.astype(np.float64))
    err = np.linalg.norm(tau - want, axis=-1) / np.maximum(np.linalg.norm(want, axis=-1), 1.0)
    assert np.all(err < 2e-5 + 8 * 2.0 ** -24 / np.sin(t[:, 0]))
    # aa_to_rmat
    axes = f32(rng.standard_normal((n, 3)) * 2); ang = f32(rng.uniform(0.01, 3.0, n))
    ga = np.empty((n, 3), np.float32); gang = np.empty(n, np.float32)
    hm.hm_aa_bwd(fp(axes), fp(ang), fp(G), fp(ga), fp(gang), ctypes.c_long(n))
    a64, an64 = axes.astype(np.float64), ang.astype(np.float64)
    num_ang = ((O.aa_to_rmat(a64, (an64 + h)[:, None]) - O.aa_to_rmat(a64, (an64 - h)[:, None])) * G).sum((-1, -2)) / (2 * h)
    assert np.max(np.abs(gang - num_ang)) < 2e-4 * max(1.0, np.abs(num_ang).max())
    for k in range(3):
        d = np.zeros(3); d[k] = h
        nk = ((O.aa_to_rmat(a64 + d, an64[:, None]) - O.aa_to_rmat(a64 - d, an64[:, None])) * G).sum((-1, -2)) / (2 * h)
        assert np.max(np.abs(ga[:, k] - nk)) < 2e-4 * max(1.0, np.abs(nk).max())
    # exp
    w = f32(rng.standard_normal((n, 3)) * np.exp(rng.uniform(-6, 0.5, (n, 1))))
    gw = np.empty((n, 3), np.float32)
    hm.hm_expvec_bwd(fp(w), fp(G), fp(gw), ctypes.c_long(n))
    w64 = w.astype(np.float64)
    for k in range(3):
        d = np.zeros(3); d[k] = h
        nk = ((O.exp_vec(w64 + d) - O.exp_vec(w64 - d)) * G).sum((-1, -2)) / (2 * h)
        assert np.max(np.abs(gw[:, k] - nk)) < 2e-4 * max(1.0, np.abs(nk).max())


# ---- lean primitives of the HBM-bound fused kernels ------------------------------------------------
def test_sincos_fast_and_atan2_pos(hm):
    rng = np.random.default_rng(21)
    x = np.concatenate([rng.uniform(-8, 8, 20000), rng.uniform(-3.3e4, 3.3e4, 20000), [0.0, 1e-8, -1e-8, math.pi / 2, math.pi, 1e-3]]).astype(np.float32)
    s = np.empty_like(x); c = np.empty_like(x)
    hm.hm_sincos_fast(fp(x), fp(s), fp(c), ctypes.c_long(x.size))
    x64 = x.astype(np.float64)
    assert np.max(np.abs(s - np.sin(x64))) < 2e-7 and np.max(np.abs(c - np.cos(x64))) < 2e-7
    small = np.abs(x64) < 1.0
    assert np.max(np.abs(s[small] - np.sin(x64[small])) / np.maximum(np.abs(np.sin(x64[small])), 1e-30)) < 3e-7
    y = np.concatenate([np.abs(rng.standard_normal(20000)), [0.0, 0.0, 1e-20, 1.0, 1e-9]]).astype(np.float32)
    xx = np.concatenate([rng.standard_normal(20000), [1.0, -1.0, 1.0, 0.0, -1.0]]).astype(np.float32)
    r = np.empty_like(y)
    hm.hm_atan2_pos(fp(y), fp(xx), fp(r), ctypes.c_long(y.size))
    want = np.arctan2(y.astype(np.float64), xx.astype(np.float64))
    assert np.max(np.abs(r - want)) < 3e-7
    tiny = (want < 1e-2) & (want > 0)
    assert np.max(np.abs(r[tiny] - want[tiny]) / want[tiny]) < 3e-7


def test_axis_angle_fast(hm):
    n = 8192
    R, _, _ = rand_rots(n, 22)
    R[:8] = np.eye(3, dtype=np.float32)
    Rpi, _, _ = O.random_rotations(64, np.random.default_rng(23), math.pi)
    ax = np.random.default_rng(24).standard_normal((64, 3)); ax /= np.linalg.norm(ax, axis=-1, keepdims=True)
    R[8:72] = f32(O.rodrigues(ax, np.full(64, math.pi)))            # exactly pi
    R[72:136] = f32(O.rodrigues(ax, math.pi - np.geomspace(1e-6, 1e-1, 64)))
    axis = np.empty((n, 3), np.float32); ang = np.empty(n, np.float32)
    hm.hm_axis_angle_fast(fp(R), fp(axis), fp(ang), ctypes.c_long(n))
    _, ang_t = O.rmat_to_aa(R)
    assert np.max(np.abs(ang - ang_t[:, 0])) < 5e-7 + 0  # atan2 of the same fp32 inputs
    assert np.max(np.abs(np.linalg.norm(axis.astype(np.float64), axis=-1) - 1)) < 1e-6
    back = O.rodrigues(axis.astype(np.float64), ang.astype(np.float64))
    assert np.max(np.abs(back - R)) < 2e-6
    assert np.all(axis[:8] == np.array([0, 0, 1], np.float32)) and np.all(ang[:8] == 0)


def test_p_mean_quat_against_oracle(hm):
    """The quaternion formulation of the reverse-step mean equals the reference algebra
    (diffusion.py:291-313) evaluated in fp64, over the part of the schedule where fp32 inputs determine it."""
    n = 8192
    s = O.schedule_buffers(1000)
    x, _, _ = rand_rots(n, 25, 3.1)
    rng = np.random.default_rng(26)
    pred = (rng.standard_normal((n, 3)) * 0.7).astype(np.float32)
    pred[:16] = 0
    t = rng.integers(0, 400, n)
    a = f32(s["sqrt_recip_alphas_cumprod"][t]); b = f32(s["sqrt_recipm1_alphas_cumprod"][t])
    c1 = f32(s["posterior_mean_coef1"][t]); c2 = f32(s["posterior_mean_coef2"][t])
    mean = np.empty((n, 3, 3), np.float32); x0h = np.empty((n, 3, 3), np.float32)
    hm.hm_p_mean_quat(fp(x), fp(pred), fp(a), fp(b), fp(c1), fp(c2), fp(mean), fp(x0h), ctypes.c_long(n))
    want0 = O.predict_start_from_noise(x, pred, a.astype(np.float64), b.astype(np.float64))
    assert np.max(O.geodesic_angle(x0h, want0)) < 3e-6
    want = O.p_sample_mean(x, pred, a.astype(np.float64), b.astype(np.float64), c1.astype(np.float64), c2.astype(np.float64))
    assert np.max(O.geodesic_angle(mean, want)) < 5e-6
    assert np.max(np.abs(mean.astype(np.float64) @ np.swapaxes(mean, -1, -2) - np.eye(3))) < 2e-6


def test_pair_kernels(hm):
    """util.py:128-150 kernel values through the quaternion formulation of the all-pairs MMD kernel, against the
    oracle's matrix-log formulation: <= 1e-6 absolute, including angles at 0, near 0 and near / at pi."""
    n = 20000
    A, _, _ = rand_rots(n, 31)
    B, _, _ = rand_rots(n, 32)
    rng = np.random.default_rng(33)
    axis = rng.standard_normal((64, 3)); axis /= np.linalg.norm(axis, axis=-1, keepdims=True)
    special = np.concatenate([[0.0, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3], math.pi - np.array([0.0, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3]), rng.uniform(0, math.pi, 52)])
    B[:64] = f32(A[:64].astype(np.float64) @ O.rodrigues(axis, special))
    out = np.empty(n, np.float32)
    hm.hm_pair_kernel(fp(A), fp(B), fp(out), n, 1)
    want = O.rmat_gaussian_kernel(A, B)
    assert np.max(np.abs(out - want)) < 1e-6
    assert np.max(np.abs(out[:64] - np.exp(-math.sqrt(2.0) * special))) < 1e-6
    hm.hm_pair_kernel(fp(A), fp(B), fp(out), n, 0)
    assert np.max(np.abs(out - O.rmat_cosine_kernel(A, B))) < 1e-6


def test_box_muller_normals(hm):
    """The four normals per Philox block (Bingham / SE(3) translation noise): finite, standard moments, independent
    components, and a tail that reaches beyond 4 sigma."""
    n = 1 << 20
    z = np.empty((n, 4), np.float32)
    hm.hm_normal4(ctypes.c_ulonglong(99), ctypes.c_ulonglong(0), ctypes.c_ulonglong(3), fp(z), n)
    assert np.isfinite(z).all() and np.abs(z).max() < 5.8
    z = z.astype(np.float64)
    assert np.max(np.abs(z.mean(0))) < 4e-3 and np.max(np.abs(z.var(0) - 1)) < 6e-3
    assert np.max(np.abs(np.corrcoef(z.T) - np.eye(4))) < 4e-3
    assert np.max(np.abs((z ** 4).mean(0) - 3)) < 0.05 and np.abs(z).max() > 4.0
    # Kolmogorov distance to the normal CDF
    from scipy.stats import kstest
    assert kstest(z[:200000, 2], "norm").statistic < 4e-3


def test_lanes_header_restates_the_scalar_arithmetic_bit_for_bit(hm):
    """csrc/so3d_lanes.cuh (one rotation or TWO rotations per thread through the same IEEE operations, the two-lane form
    packed as FFMA2 / FMUL2 / FADD2 on the device): its one-lane and two-lane instantiations of the reverse step's mean and
    of the drawn direction equal the scalar functions of so3d_math.cuh bit for bit on the host build."""
    n = 20000
    R, _, _ = rand_rots(n, 77)
    R[:8] = np.eye(3, dtype=np.float32)                       # identity rows
    R[8:16] = O.rodrigues(np.tile([[0.6, 0.0, 0.8]], (8, 1)), np.full(8, math.pi)).astype(np.float32)   # rotations by pi
    rng = np.random.default_rng(78)
    pred = f32(rng.standard_normal((n, 3)) * 0.4)
    s = O.schedule_buffers(1000)
    t = rng.integers(0, 1000, n)
    a, b = f32(s["sqrt_recip_alphas_cumprod"][t]), f32(s["sqrt_recipm1_alphas_cumprod"][t])
    c1, c2 = f32(s["posterior_mean_coef1"][t]), f32(s["posterior_mean_coef2"][t])
    mean = np.empty((n, 9), np.float32); x0h = np.empty((n, 9), np.float32)
    hm.hm_lanes_p_mean.restype = ctypes.c_long
    for has_pred in (1, 0):
        bad = hm.hm_lanes_p_mean(fp(R), fp(pred), fp(a), fp(b), fp(c1), fp(c2), fp(mean), fp(x0h), ctypes.c_long(n), has_pred)
        assert bad == 0, (has_pred, bad)
        assert np.isfinite(mean).all()
    hm.hm_lanes_p_mean_rows.restype = ctypes.c_long   # per-row step indices (the two lanes carry different schedule scalars)
    assert hm.hm_lanes_p_mean_rows(fp(R), fp(pred), fp(a), fp(b), fp(c1), fp(c2), ctypes.c_long(n)) == 0
    # forward noising (q_sample_quat_l): x0 incl. identity / near-pi rows, schedule scales, drawn axis and angle
    sc = f32(s["sqrt_alphas_cumprod"][t])
    nax = rng.standard_normal((n, 3)); nax = f32(nax / np.linalg.norm(nax, axis=-1, keepdims=True))
    nang = f32(rng.uniform(0, np.pi, n)); nang[:3] = [0.0, np.pi, 1e-4]
    xt = np.empty((n, 9), np.float32)
    hm.hm_lanes_q_sample.restype = ctypes.c_long
    assert hm.hm_lanes_q_sample(fp(R), fp(sc), fp(nax), fp(nang), fp(xt), ctypes.c_long(n)) == 0
    assert np.isfinite(xt).all()
    ua, ub = f32(rng.uniform(0, 1, n)), f32(rng.uniform(0, 1, n))
    ua[:4] = [0.0, 1.0 - 2 ** -24, 0.5, 2 ** -24]
    axis = np.empty((n, 3), np.float32)
    hm.hm_lanes_sphere.restype = ctypes.c_long
    assert hm.hm_lanes_sphere(fp(ua), fp(ub), fp(axis), ctypes.c_long(n)) == 0
    assert np.max(np.abs(np.linalg.norm(axis.astype(np.float64), axis=-1) - 1)) < 1e-6


def test_series_warp_split(hm):
    """The one-warp-per-rotation form of the series (small batches: the L terms split over the 32 lanes, block results
    propagated by powers of the homogeneous transfer matrix, butterfly sum), emulated lane by lane in the kernel's reduction
    order: same 1e-5 bound against the fp64 series as the one-thread recurrence -- below the conditioning guard for the raw
    sum, on the whole E-set with the guard -- and within a few 1e-6 of the one-thread result."""
    n = 12000
    om, eps, k = eset(n, 23)
    om[:20] = 0.0
    ft, gt = _truth(om, eps)
    hm.hm_series_warp.restype = None
    for L in (2000, 1999, 64, 2896):
        lf = np.empty(n, np.float32); g = np.empty(n, np.float32)
        hm.hm_series_warp(fp(om), fp(eps), fp(lf), fp(g), ctypes.c_long(n), L, 1)
        if L < 1999:
            continue   # short truncations are only checked for finiteness below (the truth above is the full series)
        ef = np.abs(np.exp(lf.astype(np.float64) - np.log(ft)) - 1)
        eg = np.abs(g - gt) / np.maximum(np.abs(gt), 1e-30)
        assert ef.max() < 1e-5 and eg[om > 0].max() < 1e-5, L
        assert np.all(g[om == 0] == 0)
    # short truncations (one or two terms per lane; a truncated series is only meaningful once it has converged: eps >= 0.5)
    eb = np.maximum(eps, 0.5).astype(np.float32)
    for L in (1, 5, 33, 64):   # (below 32 terms, fewer than one per lane: no term l >= L may be summed)
        lw = np.empty(n, np.float32); gw = np.empty(n, np.float32); l1 = np.empty(n, np.float32); g1 = np.empty(n, np.float32)
        hm.hm_series_warp(fp(om), fp(eb), fp(lw), fp(gw), ctypes.c_long(n), L, 0)
        hm.hm_logf_g(fp(om), fp(eb), fp(l1), fp(g1), ctypes.c_long(n), 4, L)
        ok = om <= 4.2 * eb     # (beyond the guard both sums are rounding noise times the condition number)
        assert np.max(np.abs(np.exp(lw.astype(np.float64) - l1.astype(np.float64)) - 1)[ok]) < 8e-6, L   # (cond 14 at the guard: ~4 u cond each)
        if L == 1:
            assert np.all(lw == 0) and np.all(gw == 0)   # f = 1: log f = 0 and d log f / d omega = 0
    # raw sum: against the one-thread recurrence (mode series_pure)
    lw = np.empty(n, np.float32); gw = np.empty(n, np.float32); l1 = np.empty(n, np.float32); g1 = np.empty(n, np.float32)
    hm.hm_series_warp(fp(om), fp(eps), fp(lw), fp(gw), ctypes.c_long(n), 2000, 0)
    hm.hm_logf_g(fp(om), fp(eps), fp(l1), fp(g1), ctypes.c_long(n), 4, 2000)
    well = om <= 4.2 * eps
    assert np.max(np.abs(np.exp(lw.astype(np.float64) - l1.astype(np.float64)) - 1)[well]) < 8e-6
