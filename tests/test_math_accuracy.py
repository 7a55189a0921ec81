"""Accuracy of the kernels' own exp/exp10/log/log10/atan/pow (aerobulk_b200/csrc/ab_math.cuh),
compiled for the host from the same source and compared with mpmath (50 digits).
Bound: 4 ulp (|rel err| <= 4.5e-16) over the argument ranges the physics uses; the GPU parity
tolerance is 1e-10, five orders of magnitude looser."""
import ctypes as C
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_abm_host.so")
ULP = 2.0 ** -52


@pytest.fixture(scope="module")
def abm():
    src = os.path.join(HERE, "abm_host_shim.cpp")
    deps = [src] + [os.path.join(HERE, "..", "aerobulk_b200", "csrc", f) for f in ("ab_math.cuh", "ab_math_tables.cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-ffp-contract=off", "-mfma", "-std=c++17", "-shared", "-fPIC",
                               "-o", SO, src])
    L = C.CDLL(SO)
    dp = C.POINTER(C.c_double)
    L.abm_eval.argtypes = [C.c_int, dp, dp, dp, C.c_long]

    def ev(fn, x, y=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = x if y is None else np.ascontiguousarray(y, dtype=np.float64)
        out = np.empty_like(x)
        L.abm_eval(fn, x.ctypes.data_as(dp), y.ctypes.data_as(dp), out.ctypes.data_as(dp), x.size)
        return out
    return ev


def _relerr(got, xs, f, ys=None):
    mp.mp.dps = 50
    worst = 0.0
    for i, x in enumerate(xs):
        ref = f(mp.mpf(float(x))) if ys is None else f(mp.mpf(float(x)), mp.mpf(float(ys[i])))
        if ref == 0:
            assert got[i] == 0.0
            continue
        worst = max(worst, float(abs((mp.mpf(float(got[i])) - ref) / ref)))
    return worst


RNG = np.random.default_rng(20251017)
N = 4000


def test_exp(abm):
    x = np.concatenate([RNG.uniform(-60, 60, N), RNG.uniform(-1, 1, N), RNG.uniform(-700, -600, 200), [0.0, -0.0, 1e-300]])
    assert _relerr(abm(0, x), x, mp.exp) <= 4 * ULP
    assert (abm(0, np.array([-701.0, -1500.0, -1e9])) == 0).all()     # flush (EXP(-zHwl/0.014) in WL_COARE)


def test_exp10(abm):
    x = np.concatenate([RNG.uniform(-10, 10, N), RNG.uniform(-0.2, 4.0, N)])   # e_sat uses [-0.2, 3.8]
    assert _relerr(abm(1, x), x, lambda v: mp.mpf(10) ** v) <= 4 * ULP


def test_log_log10(abm):
    x = np.concatenate([np.exp(RNG.uniform(-40, 40, N)), RNG.uniform(0.5, 2.0, N), [1.0, 2.0, 0.5, 1e-9, 10.0]])
    x = np.concatenate([x, 1.0 + RNG.uniform(-3e-3, 3e-3, N), np.nextafter(1.0, [0.0, 2.0])])
    mp.mp.dps = 50
    for xi, gi in zip(x, abm(2, x)):
        ref = mp.log(mp.mpf(float(xi)))
        err = abs(mp.mpf(float(gi)) - ref)
        assert err <= 4 * ULP * abs(ref), (xi, gi, float(ref))
    assert abm(2, np.array([1.0]))[0] == 0.0
    x = np.exp(RNG.uniform(-5, 5, N))
    assert _relerr(abm(3, x)[np.abs(np.log10(x)) > 1e-3], x[np.abs(np.log10(x)) > 1e-3], mp.log10) <= 5 * ULP


def test_atan(abm):
    x = np.concatenate([RNG.uniform(-20, 20, N), RNG.uniform(0.3, 3.0, N), np.exp(RNG.uniform(-20, 20, N)),
                        [0.0, 0.41421356237309503, 0.41421356237309515, 2.414213562373095, 2.4142135623730954, 1.0]])
    assert _relerr(abm(4, x), x, mp.atan) <= 4 * ULP
    assert np.signbit(abm(4, np.array([-0.0]))[0])


def test_atan_of_arguments_from_one_up(abm):
    """datan_ge1: the one-range atan the stability functions use (their arguments are >= 1): atan(c) + atan((x-c)/(1+cx))
    with c = tan(3 pi/8) keeps the inner argument inside the polynomial's range for every x in [1, inf)."""
    x = np.concatenate([RNG.uniform(1.0, 6.0, N), 1.0 + np.exp(RNG.uniform(-36, 3, N)), np.exp(RNG.uniform(0, 40, N)),
                        [1.0, np.nextafter(1.0, 2.0), 2.414213562373095, 2.4142135623730954, 1.7320508, 1e30]])
    assert _relerr(abm(16, x), x, mp.atan) <= 3 * ULP
    # and it agrees with the general-purpose version to rounding
    assert np.abs(abm(16, x) - abm(4, x)).max() <= 4 * ULP
    # around c the only rounding left is atan_hi(c) + (t + atan_lo(c)): correctly rounded (the low part decides it)
    x = 2.414213562373095 + np.arange(-300, 301) * np.spacing(2.414213562373095)
    got = abm(16, x)
    assert all(abs(mp.mpf(float(g)) - mp.atan(mp.mpf(float(v)))) <= np.spacing(g) / 2 for g, v in zip(got, x))


def test_guard_free_roots(abm):
    x = np.concatenate([np.exp(RNG.uniform(-60, 60, N)), RNG.uniform(1.0, 30.0, N), [1.0, 1e-30, 1e30]])
    mp.mp.dps = 50
    assert _relerr(abm(17, x), x, mp.sqrt) <= 2 * ULP
    assert _relerr(abm(18, x), x, lambda v: v ** mp.mpf(0.75)) <= 3 * ULP
    assert (abm(17, x) == abm(15, x)).all() and (abm(18, x) == abm(13, x)).all()    # the guarded versions, bit for bit


def test_powr_and_rcp(abm):
    x = np.exp(RNG.uniform(-12, 12, N))
    y = RNG.choice([0.25, 0.3333, 0.5, 0.6, 0.72, 0.75, 0.79, 1.5, -0.599, -3.935, 0.929, 2.0 / 3.0, 0.0], N)
    got = abm(5, x, y)
    mp.mp.dps = 50
    worst = 0.0
    for xi, yi, gi in zip(x, y, got):
        ref = mp.mpf(float(xi)) ** mp.mpf(float(yi))
        # exp(y log x): the error of log is amplified by |y log x|
        bound = (4 + 2 * abs(float(yi) * np.log(xi))) * ULP
        assert abs((mp.mpf(float(gi)) - ref) / ref) <= bound, (xi, yi)
    assert (abm(5, np.zeros(3), np.array([0.75, 0.79, 2.0 / 3.0])) == 0).all()   # 0**y = 0
    x = np.exp(RNG.uniform(-30, 30, N))
    assert _relerr(abm(6, x), x, lambda v: 1 / v) <= 2 * ULP


def test_fast_roots(abm):
    """x**(-1/2), x**(-1/3), x**(-1/4), x**0.75, x**(1/3): one seed (degraded to 2^-21 in the host build, the worst the
    device seeds may have) and one cubic-convergence step."""
    x = np.concatenate([np.exp(RNG.uniform(-60, 60, N)), RNG.uniform(0.5, 4.0, N), [1.0, 2.0, 8.0, 1e-29, 1e30]])
    mp.mp.dps = 50
    assert _relerr(abm(10, x), x, lambda v: 1 / mp.sqrt(v)) <= 2 * ULP
    assert _relerr(abm(11, x), x, lambda v: v ** (mp.mpf(-1) / 3)) <= 2 * ULP
    assert _relerr(abm(12, x), x, lambda v: v ** mp.mpf(-0.25)) <= 2 * ULP
    assert _relerr(abm(13, x), x, lambda v: v ** mp.mpf(0.75)) <= 3 * ULP
    assert _relerr(abm(14, x), x, lambda v: v ** (mp.mpf(1) / 3)) <= 3 * ULP
    assert _relerr(abm(15, x), x, mp.sqrt) <= 2 * ULP
    z = np.array([0.0, 1e-31, 1e-300])
    assert (abm(13, z) == 0).all() and (abm(14, z) == 0).all()     # documented flush below 1e-30
    assert (abm(15, np.array([0.0, 1e-300])) == 0).all()
    assert _relerr(abm(6, x), x, lambda v: 1 / v) <= 2 * ULP       # 3-instruction reciprocal refinement


def test_generated_tables_are_up_to_date():
    """aerobulk_b200/csrc/ab_math_tables.cuh is exactly what tools/gen_math_tables.py generates (mpmath, 50 digits)."""
    import sys
    root = os.path.dirname(HERE)
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gen_math_tables.py"), "--check"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
