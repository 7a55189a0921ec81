"""Per-function GPU unit tests (SURVEY.md 4): every __device__ building block of the hot path
(aerobulk_b200/csrc/ab_device.cuh, ab_math.cuh) evaluated by probe_kernel through the C ABI
(aerobulk_gpu_probe) against the matching abo_* export of the CPU oracle, i.e. against the restatement of
the reference function it replaces (file:line in the table below).

Tolerances, written here: the device functions use their own exp/log/atan/roots (<= 4 ulp each) and FMA
contraction, so a building block agrees with glibc arithmetic to a few 1e-16 relative per transcendental;
REL is the bound asserted per function on |gpu - oracle| / max(|oracle|, FLOOR).  The kernels' own math (MATH below) is
held to mpmath; the sea-ice building blocks are in tests/test_gpu_ice_functions.py."""
import mpmath as mp
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N = 4000
rng = np.random.default_rng(20251017)
U = lambda lo, hi, n=N: lo + (hi - lo) * rng.random(n)

T_AIR = U(240.0, 320.0)
T_SEA = U(271.0, 305.0)
Q_AIR = U(1e-4, 0.03)
P = U(80000.0, 110000.0)
ZETA = np.concatenate([U(-50.0, 0.0, N // 2), U(0.0, 50.0, N // 4), -10.0 ** U(-12, 0, N // 8), 10.0 ** U(-12, 0, N // 8)])
ZETA[:4] = (0.0, -0.0, 1e-300, -1e-300)      # psi(+0) = -4.524e-3 for COARE (SIGN(0.5, +0) selects the stable side)
WIND = U(0.3, 40.0)

# name -> (oracle callable on scalars, argument arrays, REL, FLOOR, reference file:line)
CASES = {
    "e_sat": (lambda L: L.abo_e_sat, (np.concatenate([T_AIR, U(150.0, 181.0, 50)]),), 2e-14, 1.0, "mod_phymbl.f90:777-800"),
    "q_sat": (lambda L: L.abo_q_sat, (T_AIR, P), 2e-14, 1e-6, "mod_phymbl.f90:881-904"),
    "theta_from_z_P0_T_q": (lambda L: L.abo_theta_from_z_P0_T_q, (U(1.0, 30.0), P, T_AIR, Q_AIR * 0.3), 1e-14, 1.0,
                            "mod_phymbl.f90:283-375"),
    "rho_air": (lambda L: L.abo_rho_air, (T_AIR, Q_AIR, P), 1e-14, 1.0, "mod_phymbl.f90:522-546"),
    "visc_air": (lambda L: L.abo_visc_air, (T_AIR,), 1e-14, 1e-6, "mod_phymbl.f90:549-563"),
    "L_vap": (lambda L: L.abo_L_vap, (T_SEA,), 1e-14, 1.0, "mod_phymbl.f90:579-598"),
    "cp_air": (lambda L: L.abo_cp_air, (Q_AIR,), 1e-14, 1.0, "mod_phymbl.f90:603-622"),
    "gamma_moist": (lambda L: L.abo_gamma_moist, (T_AIR, Q_AIR), 2e-14, 1e-3, "mod_phymbl.f90:627-649"),
    "alpha_sw": (lambda L: L.abo_alpha_sw, (np.concatenate([T_SEA, U(268.0, 271.0, 50)]),), 2e-14, 1e-6,
                 "mod_phymbl.f90:1267-1286"),
    "qlw_net": (lambda L: L.abo_qlw_net, (U(150.0, 500.0), T_SEA), 1e-13, 10.0, "mod_phymbl.f90:1291-1314"),
    "one_on_L": (lambda L: L.abo_one_on_L, (T_AIR, Q_AIR, 10.0 ** U(-4, 0.3), U(-1.0, 1.0), U(-1e-3, 1e-3)), 2e-14, 1e-3,
                 "mod_phymbl.f90:666-693"),
    # Ri_b = g z dtheta_v / (Tv Ub^2) with dtheta_v a DIFFERENCE of two ~300 K virtual temperatures: its rounding error is
    # ~1 ulp(300 K) whatever its size, so the error is measured against Ri_b of a unit virtual-temperature difference
    # (floor = g z / (280 Ub^2), filled in per point by the test)
    "Ri_bulk": (lambda L: L.abo_Ri_bulk, (U(2.0, 30.0), T_SEA, T_SEA + U(-8.0, 4.0), Q_AIR, Q_AIR * 0.8, U(0.2, 30.0)), 1e-12,
                "ri_bulk_scale", "mod_phymbl.f90:712-747"),
    "q_air_rh": (lambda L: L.abo_q_air_rh, (U(5.0, 100.0), T_AIR, P), 2e-14, 1e-6, "mod_phymbl.f90:963-985"),
    "q_air_dp": (lambda L: L.abo_q_air_dp, (T_AIR - 3.0, P), 2e-14, 1e-6, "mod_phymbl.f90:990-1000"),
    "cd_n10_ncar": (lambda L: L.abo_cd_n10_ncar, (np.concatenate([WIND, [32.999999, 33.0, 33.000001, 0.5]]),), 1e-14, 1e-4,
                    "mod_blk_ncar.f90:244-271"),
    "charn_coare3p0": (lambda L: L.abo_charn_coare3p0, (np.concatenate([WIND, [10.0, 18.0, 9.999999, 18.000001]]),), 1e-14, 1e-3,
                       "mod_blk_coare3p0.f90:420-447"),
    "charn_coare3p6": (lambda L: L.abo_charn_coare3p6, (np.concatenate([WIND, [0.0, 2.9, 19.5, 35.0]]),), 1e-14, 1e-3,
                       "mod_blk_coare3p6.f90:417-432"),
}
# psi: absolute floor 1 (psi is O(1..100)); COARE convective branch mixes 3 logs, 2 atans and a cube root.  The solvers take
# psi_h(zeta_u) from the paired psi_mh_*_unstable evaluators and psi_h(zeta_t) from the single ones: the psi_h probes
# return NaN where the two differ, which the finiteness check below catches
PSI = {"ncar": (3, 2e-14), "coare": (2, 1e-13), "ecmwf": (4, 5e-14), "andreas": (5, 1e-13)}


def _oracle_eval(fn, cols):
    return np.array([fn(*[float(c[i]) for c in cols]) for i in range(cols[0].size)])


@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    ab.reset()
    return ab


@pytest.fixture(scope="module")
def OL():
    from oracle import oracle
    return oracle.lib()


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_function_matches_oracle(ab, OL, name):
    get, cols, rel, floor, where = CASES[name]
    cols = [np.asarray(c, dtype=np.float64) for c in cols]
    got = ab.probe(name, *cols)
    ref = _oracle_eval(get(OL), cols)
    assert np.all(np.isfinite(got)), name
    if floor == "ri_bulk_scale":
        floor = 9.8 * cols[0] / (280.0 * cols[5] ** 2)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), floor)
    print(f"[function] {name:22s} ({where}): max rel err {err.max():.2e} over {ref.size} points")
    assert err.max() <= rel, (name, float(err.max()), [float(c[err.argmax()]) for c in cols])


@pytest.mark.parametrize("algo", sorted(PSI))
@pytest.mark.parametrize("which", ["m", "h"])
def test_psi_matches_oracle(ab, OL, algo, which):
    aid, rel = PSI[algo]
    z = ZETA if algo != "ecmwf" else np.clip(ZETA, -60.0, 10.0)
    got = ab.probe(f"psi_{which}_{algo}", z)
    fn = OL.abo_psi_m if which == "m" else OL.abo_psi_h
    ref = np.array([fn(aid, float(x)) for x in z])
    assert np.all(np.isfinite(got)), (algo, which)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)
    print(f"[function] psi_{which}_{algo}: max scaled err {err.max():.2e}; psi(+0) = {got[0]!r}, psi(-0) = {got[1]!r}")
    assert err.max() <= rel, (algo, which, float(err.max()), float(z[err.argmax()]))
    if algo == "coare":
        assert got[0] == pytest.approx(-4.524e-3, rel=2e-3) and abs(got[1]) < 1e-12   # SURVEY 8a a19: the +0 quirk is kept


@pytest.mark.parametrize("iflag", [1, 2])
def test_z0tq_lkb_matches_oracle(ab, OL, iflag):
    """Liu-Katsaros-Businger table (src/mod_phymbl.f90:1635-1701): every interval, the edges and both out-of-range sides."""
    rer = np.concatenate([10.0 ** U(-4, 3.2, N), [0.11, 0.825, 3.0, 10.0, 30.0, 100.0, 300.0, 1000.0, 0.0, -1.0, 2000.0]])
    z0 = 10.0 ** U(-6, -2.6, rer.size)
    got = ab.probe("z0tq_LKB", np.full(rer.size, float(iflag)), rer, z0)
    ref = np.array([OL.abo_z0tq_LKB(iflag, float(r), float(z)) for r, z in zip(rer, z0)])
    err = np.abs(got - ref) / np.abs(ref)
    print(f"[function] z0tq_LKB iflag={iflag}: max rel err {err.max():.2e}")
    assert err.max() <= 2e-13, (float(err.max()), float(rer[err.argmax()]))   # log-space evaluation: |log z0t| <= 21 amplifies the ulps


@pytest.mark.parametrize("coare", [True, False])
def test_cool_skin_matches_oracle(ab, OL, coare):
    """dT_cs of CS_COARE (src/mod_skin_coare.f90:48-93) / CS_ECMWF (src/mod_skin_ecmwf.f90:68-110) rebuilt from the
    oracle's delta_skin_layer (src/mod_phymbl.f90:2010-2046) with the loop of the reference."""
    n = 1500
    alpha = np.array([OL.abo_alpha_sw(float(t)) for t in U(272.0, 304.0, n)])
    Qsw = np.where(rng.random(n) < 0.4, 0.0, U(0.0, 900.0, n))
    Qns = U(-400.0, 60.0, n)
    us = 10.0 ** U(-3, 0.0, n)
    Qlat = U(-300.0, 20.0, n)
    got = ab.probe("cs_coare" if coare else "cs_ecmwf", alpha, Qsw, Qns, us, Qlat)
    ref = np.empty(n)
    for i in range(n):
        a, qs, qn, u, ql = (float(x[i]) for x in (alpha, Qsw, Qns, us, Qlat))
        d = OL.abo_delta_skin_layer(a, qn, u, int(coare), ql)
        zQabs = qn
        for _ in range(4):
            zfr = max((0.137 if coare else 0.065) + 11.0 * d - 6.6e-5 / d * (1.0 - np.exp(-d / 8.0e-4)), 0.01)
            zQabs = qn + zfr * qs
            d = OL.abo_delta_skin_layer(a, zQabs, u, int(coare), ql)
        ref[i] = zQabs * d / 0.6
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-2)
    print(f"[function] cool skin ({'COARE' if coare else 'ECMWF'}): max scaled err {err.max():.2e}")
    assert err.max() <= 1e-12, float(err.max())


ULP = 2.0 ** -52
TAN_PI8 = [0.41421356237309503, 0.41421356237309515]      # the doubles either side of tan(pi/8) and tan(3 pi/8)
TAN_3PI8 = [2.414213562373095, 2.4142135623730954]
_next = lambda x, d: np.atleast_1d(np.nextafter(np.asarray(x, dtype=np.float64), d))
_ATAN_EDGES = np.array(TAN_PI8 + TAN_3PI8 + [1.0])
_ATAN_EDGES = np.concatenate([_ATAN_EDGES, _next(_ATAN_EDGES, 0.0), _next(_ATAN_EDGES, 10.0)])
_GE1 = np.concatenate([U(1.0, 6.0), 1.0 + np.exp(U(-36.0, 3.0)), np.exp(U(0.0, 40.0)),
                       [1.0, np.nextafter(1.0, 2.0), 1.7320508, 1e30] + TAN_3PI8])
_L10 = np.exp(U(-5.0, 5.0))
_POWR_X = np.exp(U(-12.0, 12.0))
_POWR_Y = rng.choice([0.25, 0.3333, 0.5, 0.6, 0.72, 0.75, 0.79, 1.5, -0.599, -3.935, 0.929, 2.0 / 3.0, 1.4, 1.0 + 1.0 / 14.0, 0.0],
                     _POWR_X.size)
_P100 = 2.0 ** -100                               # the guard of pow075 / fast_cbrt: 0 below it

# name -> (mpmath function, [(label, arguments, bound)], arguments that must give exactly 0).  A bound is a relative error
# against mpmath (50 digits): "core" keeps the bound of the ranges checked since round 2; every other set takes the bound
# tests/test_math_accuracy.py proves for the host build of the same source (whose seeds are degraded to 2**-21), in ulp
# of 2**-52.  powr: (4 + 2 |y log x|) ulp, the error of the logarithm amplified by the exponent.
MATH = {
    "exp": (mp.exp, [("core", (U(-690.0, 690.0),), 4.5e-16),
                     ("near 0, flush threshold", (np.concatenate([U(-1.0, 1.0), U(-700.0, -690.0, 500), [-700.0, 0.0, -0.0],
                                                                  _next(-700.0, 0.0)]),), 4 * ULP)],
            (np.array([np.nextafter(-700.0, -800.0), -700.5, -701.0, -1500.0, -1e9]),)),
    "exp10": (lambda x: mp.mpf(10) ** x, [("core", (U(-300.0, 300.0),), 4.5e-16),
                                          ("e_sat range, flush threshold",
                                           (np.concatenate([U(-0.2, 4.0), U(-304.0, -300.0, 500), [-304.0, 0.0],
                                                            _next(-304.0, 0.0)]),), 4 * ULP)],
              (np.array([np.nextafter(-304.0, -400.0), -304.5, -305.0, -1e9]),)),
    "log": (mp.log, [("core", (10.0 ** U(-300, 300),), 4.5e-16),
                     ("near 1", (np.concatenate([1.0 + U(-3e-3, 3e-3), U(0.5, 2.0), _next(1.0, 0.0), _next(1.0, 2.0),
                                                 [2.0, 0.5, 1e-9, 10.0]]),), 4 * ULP)],
            (np.array([1.0]),)),
    "atan": (mp.atan, [("core", (np.concatenate([U(-50.0, 50.0), 10.0 ** U(-8, 8)]),), 4.5e-16),
                       ("range switches", (np.concatenate([U(0.3, 3.0), _ATAN_EDGES, -_ATAN_EDGES[_ATAN_EDGES > 0]]),), 4 * ULP)],
             (np.array([0.0]),)),
    "atan_ge1": (mp.atan, [("x >= 1", (_GE1,), 3 * ULP)], None),
    "log10": (mp.log10, [("|log10 x| > 1e-3", (np.concatenate([_L10[np.abs(np.log10(_L10)) > 1e-3], 10.0 ** U(-300, 300)]),),
                          5 * ULP)], (np.array([1.0]),)),
    "exp_b": (mp.exp, [("[-700, 700]", (np.concatenate([U(-700.0, 700.0), U(-1.0, 1.0), [-700.0, 700.0, 0.0]]),), 4 * ULP)],
              None),
    "exp10_b": (lambda x: mp.mpf(10) ** x, [("[-300, 300]", (np.concatenate([U(-300.0, 300.0), U(-0.2, 4.0), [-300.0, 300.0]]),),
                                            4 * ULP)], None),
    "sqrt": (mp.sqrt, [("core", (10.0 ** U(-280, 300),), 4.5e-16), ("e**[-60, 60]", (np.exp(U(-60.0, 60.0)),), 2 * ULP)],
             (np.array([0.0, 1e-300]),)),
    "rsqrt": (lambda x: 1 / mp.sqrt(x), [("core", (10.0 ** U(-30, 30),), 6e-16), ("e**[-60, 60]", (np.exp(U(-60.0, 60.0)),), 2 * ULP)],
              None),
    "cbrt": (mp.cbrt, [("core", (10.0 ** U(-28, 30),), 6e-16),
                       ("guard", (np.concatenate([[_P100, np.nextafter(_P100, 1.0), 2.0 * _P100, 1e-30], U(0.5, 4.0)]),), 3 * ULP)],
             (np.array([np.nextafter(_P100, 0.0), 1e-31, 1e-300, 0.0]),)),
    "rcbrt": (lambda x: 1 / mp.cbrt(x), [("core", (10.0 ** U(-28, 30),), 6e-16), ("e**[-60, 60]", (np.exp(U(-60.0, 60.0)),), 2 * ULP)],
              None),
    "pow075": (lambda x: x ** mp.mpf(0.75), [("core", (10.0 ** U(-28, 30),), 6e-16),
                                            ("guard", (np.concatenate([[_P100, np.nextafter(_P100, 1.0), 2.0 * _P100, 1e-30],
                                                                       U(0.5, 4.0)]),), 3 * ULP)],
               (np.array([np.nextafter(_P100, 0.0), 1e-31, 1e-300, 0.0]),)),
    "rcp": (lambda x: 1 / x, [("core", (10.0 ** U(-280, 280) * np.sign(U(-1, 1)),), 4.5e-16),
                              ("e**[-30, 30]", (np.exp(U(-30.0, 30.0)) * np.sign(U(-1, 1)),), 2 * ULP)], None),
    "powr": (lambda x, y: x ** y, [("e**[-12, 12] ** y", (_POWR_X, _POWR_Y),
                                    lambda x, y: (4 + 2 * np.abs(y * np.log(x))) * ULP)],
             (np.zeros(4), np.array([0.75, 0.79, 2.0 / 3.0, 1.4]))),
}


def _mp_relerr(f, got, cols):
    with mp.workdps(50):
        return np.array([float(abs((mp.mpf(float(g)) - r) / r))
                         for g, r in ((got[i], f(*[mp.mpf(float(c[i])) for c in cols])) for i in range(got.size))])


@pytest.mark.parametrize("name", sorted(MATH))
def test_own_math_on_device(ab, name):
    """ab_math.cuh as the device compiles it (MUFU seeds, FMA contraction) against mpmath, over the ranges the physics
    uses and the tails where the functions switch: the flush thresholds of exp / exp10, log near 1, atan's range switches
    at tan(pi/8) and tan(3 pi/8), the 2**-100 guard of pow075 / cbrt.  The host build of the same source is held to the
    same bounds in tests/test_math_accuracy.py; a device value outside them points at contraction or a seed."""
    f, sets, zeros = MATH[name]
    for label, cols, bound in sets:
        cols = [np.asarray(c, dtype=np.float64) for c in cols]
        got = ab.probe(name, *cols)
        err = _mp_relerr(f, got, cols)
        b = bound(*cols) if callable(bound) else np.full(err.size, bound)
        print(f"[function] abm::{name:8s} {label:28s}: max rel err {err.max():.2e} ({err.max() / ULP:.2f} ulp), "
              f"worst err/bound {(err / b).max():.2f}")
        assert (err <= b).all(), (name, label, float(err.max()), [float(c[(err / b).argmax()]) for c in cols])
    if zeros is not None:
        got = ab.probe(name, *zeros)
        assert (got == 0.0).all(), (name, got)
    if name == "atan":
        assert np.signbit(ab.probe("atan", np.array([-0.0]))[0])


def test_atan_ge1_correctly_rounded_at_its_expansion_point(ab):
    """datan_ge1(x) = atan_hi(c) + (t + atan_lo(c)), c = tan(3 pi/8), t = atan((x - c) / (1 + c x)).  For x within a few
    hundred ulp of c, t is a few ulp of the result and exact to ~1e-30, so the one rounding left is the final addition:
    the result must be correctly rounded.  The low part of atan(c) (0.12 ulp) decides the rounding of about one point in
    eight here; an error of 3 ulp elsewhere cannot show its loss."""
    c = TAN_3PI8[0]
    x = c + np.arange(-300, 301) * np.spacing(c)
    got = ab.probe("atan_ge1", x)
    with mp.workdps(50):
        err = np.array([float(abs(mp.mpf(float(g)) - mp.atan(mp.mpf(float(v))))) for g, v in zip(got, x)]) / np.spacing(got)
    print(f"[function] abm::atan_ge1 around tan(3 pi/8): max err {err.max():.4f} ulp of the result")
    assert err.max() <= 0.5, (float(err.max()), float(x[err.argmax()]))
