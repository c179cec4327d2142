"""include/sag_detmath.h against a higher-precision reference: glibc's long-double sinl / cosl / atan2l / logl (through
numpy's longdouble, 64-bit mantissa on x86-64), so that an error of the double routines is seen rather than compared
with glibc's own double rounding.  Parity cannot see an error in this file (the kernels and the oracle share it); the
device compiles the same header and is pinned to it by the parity tests.  Errors are in units of the last place of the
correctly rounded double result; next to the zeros of sin / cos only an absolute bound holds."""
import numpy as np
import pytest

import oracle as O

LD = np.longdouble
pytestmark = pytest.mark.skipif(np.finfo(LD).nmant < 63, reason="needs an 80-bit long double reference")


def _ulps(a, ref):
    """|a - ref| in ulps of the double nearest to the long-double reference"""
    return np.abs((a.astype(LD) - ref) / np.spacing(np.abs(ref.astype(np.float64))).astype(LD)).astype(np.float64)


def _abs(a, ref):
    return np.abs(a.astype(LD) - ref).astype(np.float64)


def test_sincos_against_long_double():
    rng = np.random.RandomState(0)
    x = np.concatenate([rng.uniform(-20, 20, 1000000), rng.normal(0, 1e-3, 100000)])
    s, c = O.detmath("sincos", x)
    rs, rc = np.sin(x.astype(LD)), np.cos(x.astype(LD))
    assert _ulps(s, rs).max() <= 1.5 and _ulps(c, rc).max() <= 1.5                       # measured 1.45 / 1.45
    # up to |x| = 7e4 (the argument reduction's range), away from the zeros
    x = rng.uniform(-7e4, 7e4, 1000000)
    s, c = O.detmath("sincos", x)
    rs, rc = np.sin(x.astype(LD)), np.cos(x.astype(LD))
    ms, mc = np.abs(rs) >= 1e-3, np.abs(rc) >= 1e-3
    assert _ulps(s[ms], rs[ms]).max() <= 3.0 and _ulps(c[mc], rc[mc]).max() <= 3.0         # measured 1.46 / 1.48
    assert _abs(s, rs).max() <= 1.2e-16 and _abs(c, rc).max() <= 1.2e-16
    # the doubles next to multiples of pi/2, where the result is ~1e-16 and a relative bound means nothing
    k = rng.randint(-44000, 44001, 400000)
    x = np.nextafter(k * (np.pi / 2), np.where(rng.uniform(size=k.size) < 0.5, -np.inf, np.inf))
    s, c = O.detmath("sincos", x)
    zs, zc = k % 2 == 0, k % 2 == 1                                                     # sin, cos vanish there
    assert _abs(s[zs], np.sin(x[zs].astype(LD))).max() <= 5e-22                           # measured 3.7e-22
    assert _abs(c[zc], np.cos(x[zc].astype(LD))).max() <= 5e-22
    x = np.arange(-64, 65) * (np.pi / 4)
    s, c = O.detmath("sincos", x)
    assert _abs(s, np.sin(x.astype(LD))).max() <= 1.2e-16 and _abs(c, np.cos(x.astype(LD))).max() <= 1.2e-16
    assert (s * s + c * c - 1.0).__abs__().max() < 5e-16


def test_atan2_within_2ulp_and_special_cases():
    rng = np.random.RandomState(1)
    y, x = rng.normal(0, 2, 1000000), rng.normal(0, 2, 1000000)
    a = O.detmath("atan2", y, x)
    assert _ulps(a, np.arctan2(y.astype(LD), x.astype(LD))).max() <= 1.5                 # measured 1.44
    ys = np.array([0.0, 0.0, 1.0, -1.0, 0.0, 1e-300, -1e-300])
    xs = np.array([1.0, -1.0, 0.0, 0.0, 0.0, -1.0, -1.0])
    np.testing.assert_allclose(O.detmath("atan2", ys, xs), np.arctan2(ys, xs), rtol=0, atol=1e-300)


def test_log_within_1ulp():
    rng = np.random.RandomState(2)
    u = 1.0 - rng.uniform(size=1000000)
    u[:8] = [1.0, 0.5, 2.0 ** -53, 1e-10, 0.999999999, 0.7071067811865475, 0.7071067811865476, 0.25]
    l = O.detmath("log", u)
    ref = np.log(u.astype(LD))
    m = ref != 0
    assert _ulps(l[m], ref[m]).max() <= 0.9 and l[0] == 0.0                              # measured 0.84


def test_folded_lidar_equals_literal_lidar():
    """sag_lidar_bin16 (one division, bin index from folds) vs the literal atan2 form of safe_adaptation_gym.py:204-223:
    random scenes, objects exactly on bin edges (every multiple of pi/8), on the axes, and at the robot's own position"""
    import oracle as O
    rng = np.random.RandomState(5)
    worst = 0.0
    for i in range(6000):
        n = rng.randint(1, 14)
        rx, ry = rng.uniform(-2, 2, 2)
        yaw = rng.uniform(-10, 10)
        xs, ys = rng.uniform(-3.5, 3.5, n), rng.uniform(-3.5, 3.5, n)
        if i % 5 == 0:   # bin edges in the ego frame
            yaw = 0.0
            k, d = rng.randint(0, 16, n), rng.uniform(0.05, 3.2, n)
            xs, ys = rx + d * np.cos(k * np.pi / 8), ry + d * np.sin(k * np.pi / 8)
        if i % 7 == 0:   # exactly on an axis / at the robot
            xs[0], ys[0] = rx, ry + (rng.randint(-1, 2)) * 0.5
        a, b = O.lidar(rx, ry, yaw, xs, ys), O.lidar(rx, ry, yaw, xs, ys, literal=True)
        worst = max(worst, float(np.abs(a - b).max()))
    assert worst < 1e-14, worst
