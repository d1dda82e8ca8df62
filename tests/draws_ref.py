"""Independent restatement of the random draws of the sampling kernels (include/so3d.h, csrc/so3d_math.cuh), shared by
test_draws_ref.py (CPU tier) and test_gpu_draws.py (GPU tier).

Every draw of the table sampler, the forward noising, the reverse step, the SE(3) pair and the Bingham sampler is a fixed
function of (seed, row, rng_offset, t): Philox4x32-10 with key = seed and counter = (row_offset + row, rng_offset); the
axis from words x and y, the uniform from word z, four Box-Muller normals from a block, and the angle from the inverse-CDF
lookup in table row t.  Nothing here calls the library or its host build: the generator is numpy uint64 arithmetic, the
conversions follow the DEVICE branch of so3d_math.cuh, and everything after the lookup is fp64.
"""
import math

import numpy as np

from oracle import so3_oracle as O

MASK32 = 0xFFFFFFFF
SHIFT_STREAM = 1 << 63          # the SE(3) translation normals come from rng_offset | 2^63 (kShiftStream)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85


def philox(seed, rows, offset):
    """Philox4x32-10 blocks for the 64-bit counters (rows[i], offset) under the 64-bit key `seed`.
    rows: integers < 2^64 (any shape).  -> uint32 array (*rows.shape, 4) of the words (x, y, z, w)."""
    rows = np.asarray(rows, dtype=np.uint64)
    m = np.uint64(MASK32)
    c0, c1 = rows & m, rows >> np.uint64(32)
    c2 = np.full(rows.shape, offset & MASK32, np.uint64)
    c3 = np.full(rows.shape, offset >> 32, np.uint64)
    k0, k1 = seed & MASK32, (seed >> 32) & MASK32
    for _ in range(10):
        p0 = _M0 * c0            # 32 x 32 -> 64 bits: exact in uint64
        p1 = _M1 * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & m,
                          (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & m)
        k0, k1 = (k0 + _W0) & MASK32, (k1 + _W1) & MASK32
    return np.stack((c0, c1, c2, c3), -1).astype(np.uint32)


def u01(x):
    """Device u01: __uint2float_rz(x) * 2^-32, i.e. x rounded toward zero to 24 significant bits, over 2^32.  (The host
    branch of u01, (x >> 8) 2^-24, differs for x < 2^24.)  -> float32."""
    x = np.asarray(x, dtype=np.uint64)
    _, e = np.frexp(x.astype(np.float64))          # x < 2^e, exactly (e = bit length)
    sh = np.maximum(e - 24, 0).astype(np.uint64)
    return (((x >> sh) << sh).astype(np.float64) * 2.0 ** -32).astype(np.float32)


def sphere_from_uniforms(ua, ub):
    """Unit axis of sphere_from_uniforms in fp64: z = 1 - 2 ua, r = sqrt(4 ua (1 - ua)), azimuth 2 pi ub - pi."""
    ua, ub = np.asarray(ua, np.float64), np.asarray(ub, np.float64)
    r = np.sqrt(4.0 * ua * (1.0 - ua))
    ph = 2.0 * math.pi * ub - math.pi
    return np.stack((r * np.cos(ph), r * np.sin(ph), 1.0 - 2.0 * ua), -1)


def axis_u(block):
    """(fp64 unit axis from words x, y; float32 uniform from word z) of Philox blocks (..., 4)."""
    return sphere_from_uniforms(u01(block[..., 0]), u01(block[..., 1])), u01(block[..., 2])


def radius_uniform(w):
    """The Box-Muller radius uniforms ((w >> 8) + 1) 2^-24, in (0, 1]."""
    return ((np.asarray(w, np.uint64) >> np.uint64(8)) + np.uint64(1)).astype(np.float64) * 2.0 ** -24


def normal4(block):
    """normal4_from_u4 in fp64: radii from words x and z, azimuths from words y and w.  -> (..., 4), and the radial
    variates -2 ln u (..., 2) the error bound of the device's MUFU.LG2 needs."""
    ta, tb = -2.0 * np.log(radius_uniform(block[..., 0])), -2.0 * np.log(radius_uniform(block[..., 2]))
    pa = 2.0 * math.pi * u01(block[..., 1]).astype(np.float64) - math.pi
    pb = 2.0 * math.pi * u01(block[..., 3]).astype(np.float64) - math.pi
    ra, rb = np.sqrt(ta), np.sqrt(tb)
    return np.stack((ra * np.cos(pa), ra * np.sin(pa), rb * np.cos(pb), rb * np.sin(pb)), -1), np.stack((ta, tb), -1)


def count_le(table, rows, u):
    """#{j : table[rows[i], j] <= u[i]} -- the index of the inverse-CDF lookup, exact (np.searchsorted per fp32 row)."""
    rows = np.asarray(rows, np.int64)
    u = np.asarray(u, np.float32)
    out = np.empty(rows.shape, np.int64)
    for r in np.unique(rows):
        m = rows == r
        out[m] = np.searchsorted(table[r], u[m], side="right")
    return out


def angle_lookup(table, rows, u, loc):
    """The fp32 inverse-CDF angle of igso3_angle_lerp: i1 = min(count, 998), i0 = max(i1 - 1, 0),
    w = clamp((u - t0) / max(t1 - t0, 1e-6), 0, 1), then torch.lerp of the grid angles.  The clamps are fmaxf / fminf
    (a NaN operand gives the other one), as on the device.  The device contracts the lerp into one FMA, so it may
    differ from this two-rounding form by 1 ulp."""
    rows = np.asarray(rows, np.int64)
    u = np.asarray(u, np.float32)
    loc = np.asarray(loc, np.float32)
    n_cdf = table.shape[1]
    i1 = np.minimum(count_le(table, rows, u), n_cdf - 1)
    i0 = np.maximum(i1 - 1, 0)
    t0, t1 = table[rows, i0], table[rows, i1]
    with np.errstate(invalid="ignore"):
        diff = np.fmax(t1 - t0, np.float32(1e-6))
        w = np.fmin(np.fmax((u - t0) / diff, np.float32(0)), np.float32(1)).astype(np.float32)
    a0, a1 = loc[i0], loc[i1]
    d = (a1 - a0).astype(np.float32)
    return np.where(w < np.float32(0.5), a0 + w * d, a1 - d * (np.float32(1) - w)).astype(np.float32)


def ulp32(x):
    """Spacing of float32 at |x| (the smallest subnormal at 0)."""
    x = np.abs(np.asarray(x, np.float32))
    return (np.nextafter(x, np.float32(np.inf)) - x).astype(np.float64)


def rodrigues(axis, ang):
    return O.rodrigues(axis, np.asarray(ang, np.float64))


def igso3_draw(table, rows, loc, seed, offset, row_ids):
    """The table sampler's draw for global rows row_ids (row_offset + i) from table rows `rows`:
    -> dict(axis fp64, u f32, angle f32 (restated lookup), noise = Rodrigues(axis, angle) fp64)."""
    axis, u = axis_u(philox(seed, row_ids, offset))
    ang = angle_lookup(table, rows, u, loc)
    return dict(axis=axis, u=u, angle=ang, noise=rodrigues(axis, ang))


def score_g(angle, eps):
    """fp64 d log f / d omega of IGSO(3)(eps) at `angle` (3-image closed form: exact to fp64 for eps <= 1, the schedule's
    range; 0 at omega = 0)."""
    return O.igso3_closed_dlog(np.asarray(angle, np.float64), np.asarray(eps, np.float64))
