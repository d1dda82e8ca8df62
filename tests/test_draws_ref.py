"""CPU tier: the numpy restatement of the kernels' random draws (tests/draws_ref.py) against the Random123 known answers
and, bit for bit, against the host build of so3d_math.cuh's Philox; its conversions and lookup against their definitions."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import so3_oracle as O
from tests import draws_ref as D

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hm(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hm") / "host_math.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "host_math", "host_math.cpp")])
    return ctypes.CDLL(so)


def host_philox(hm, seed, row0, offset, n):
    out = np.empty(4 * n, np.uint32)
    hm.hm_philox(ctypes.c_ulonglong(seed), ctypes.c_ulonglong(row0), ctypes.c_ulonglong(offset),
                 out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), ctypes.c_long(n))
    return out.reshape(n, 4)


def test_philox_known_answers():
    """Random123's known answers for philox4x32-10 (counter = key = 0, and the digits of pi)."""
    assert [hex(x) for x in D.philox(0, [0], 0)[0]] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    seed = 0xa4093822 | (0x299f31d0 << 32)
    row = 0x243f6a88 | (0x85a308d3 << 32)
    off = 0x13198a2e | (0x03707344 << 32)
    assert [hex(x) for x in D.philox(seed, [row], off)[0]] == ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_philox_equals_host_build(hm):
    """Bit for bit the generator of so3d_math.cuh (host build) on random 64-bit (seed, row, offset), rows that cross 2^32
    and sit above 2^40 and near 2^64, and offsets with bit 63 set (the SE(3) translation stream)."""
    rng = np.random.default_rng(17)
    cases = [(0, 0, 0), (1234, 2**32 - 40, 7), (2**64 - 1, 2**40 + 5, 2**63 | 12345), (99, 2**64 - 300, 2**63),
             (0x1234_5678_9ABC, 2**40 - 100, 3)]
    cases += [(int(rng.integers(0, 2**63)) * 2 + 1, int(rng.integers(0, 2**62)), int(rng.integers(0, 2**63)) | (i % 2) << 63)
              for i in range(6)]
    for seed, row0, off in cases:
        n = 256
        want = host_philox(hm, seed, row0, off, n)
        got = D.philox(seed, row0 + np.arange(n, dtype=np.uint64), off)
        assert np.array_equal(got, want), (seed, row0, off)


def test_device_uniform_conversion():
    """u01 keeps the top 24 significant bits of the word (toward zero) over 2^32: for u >= 1/2 the host branch's
    (x >> 8) 2^-24, finer below it (and non-zero for x < 2^8, where the host branch gives 0)."""
    x = np.array([0, 1, 2**24 - 1, 2**24, 2**24 + 1, 2**25 + 3, 2**31, 2**32 - 1, 0x8000_0001, 0x0123_4567], np.uint64)
    got = D.u01(x)
    assert got.dtype == np.float32
    want = []
    for v in x.tolist():
        keep = max(v.bit_length() - 24, 0)
        want.append(((v >> keep) << keep) / 2.0 ** 32)
    assert np.array_equal(got.astype(np.float64), np.array(want))
    assert got[-3] == np.float32(1.0 - 2.0 ** -24) and got[-3] < 1.0
    assert got[1] == np.float32(2.0 ** -32)                      # the host branch would give 0
    w = np.random.default_rng(3).integers(0, 2**32, 10000, dtype=np.uint64)
    host = ((w >> np.uint64(8)).astype(np.float64) * 2.0 ** -24).astype(np.float32)
    top = w >= 2**31
    assert np.array_equal(D.u01(w)[top], host[top])
    assert np.all(D.u01(w)[~top] >= host[~top]) and np.any(D.u01(w)[~top] > host[~top])


def test_axis_and_normals_from_the_block():
    """The fp64 axis is a unit vector from words (x, y); the normals have the Box-Muller radius of words x and z."""
    blk = D.philox(5, np.arange(50000, dtype=np.uint64), 11)
    axis, u = D.axis_u(blk)
    assert np.max(np.abs(np.linalg.norm(axis, axis=-1) - 1)) < 1e-15
    assert np.array_equal(u, D.u01(blk[:, 2]))
    assert np.array_equal(axis[:, 2], 1.0 - 2.0 * D.u01(blk[:, 0]).astype(np.float64))
    z, t = D.normal4(blk)
    assert np.allclose(np.hypot(z[:, 0], z[:, 1]) ** 2, t[:, 0]) and np.allclose(np.hypot(z[:, 2], z[:, 3]) ** 2, t[:, 1])
    assert np.all(t <= 2 * 24 * math.log(2) + 1e-12) and np.all(t >= 0)
    assert abs(z.mean()) < 0.01 and abs(z.var() - 1) < 0.01


def test_lookup_index_and_lerp():
    """angle_lookup's index is #{trap <= u} on the fp32 row and its lerp is the oracle's (distributions.py:38-49) on
    finite rows; on a NaN row (a CDF of 0/0) it returns the first grid angle, as fmaxf / fminf make the device do."""
    eps = np.float32([0.0064, 0.05, 0.3, 1.0])
    trap, loc = O.igso3_cdf_table(eps)
    rng = np.random.default_rng(4)
    n = 4000
    rows = rng.integers(0, len(eps), n)
    u = rng.random(n).astype(np.float32)
    u[:8] = [0.0, 2.0 ** -24, 0.5, 1 - 2.0 ** -24, trap[rows[4], 500], trap[rows[5], 0], 2.0 ** -30, trap[rows[7], 100]]
    cnt = D.count_le(trap, rows, u)
    assert np.array_equal(cnt, (trap[rows] <= u[:, None]).sum(-1))
    got = D.angle_lookup(trap, rows, u, loc)
    want = np.concatenate([O.igso3_angle_from_uniform(u[i:i + 1], trap[rows[i]], loc) for i in range(n)])
    assert np.array_equal(got, want)
    nan_row = np.full((1, trap.shape[1]), np.nan, np.float32)
    assert np.array_equal(D.angle_lookup(nan_row, np.zeros(3, np.int64), np.float32([0.0, 0.5, 0.9]), loc), np.full(3, loc[0]))
