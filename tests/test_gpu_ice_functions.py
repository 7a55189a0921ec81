"""Per-function GPU unit tests of the sea-ice building blocks (aerobulk_b200/csrc/ab_ice.cuh), evaluated by probe_kernel
(aerobulk_gpu_probe ids 60-70) against a 50-digit mpmath restatement of each formula as the reference writes it
(src/mod_phymbl.f90, src/ice/mod_blk_ice_an05.f90, src/ice/mod_cdn_form_ice.f90).

The restatement uses the literal constants as written (each one the double the compiler makes of it) and takes every
decision -- SIGN, MAX, the clamps, the Andreas 1987 regime -- on the double value the reference computes; only the
magnitudes are evaluated in mpmath.  The CPU tests hold the restatement to the oracle's abo_* exports, so that a slip
in it shows up without a GPU; the GPU tests hold the device to it.

The solvers reach these functions only through solve_ice, where a branch is exercised only if the iteration happens to
go there; here every branch and every edge is taken on purpose: the sign of zero in psi_*_ice and f_*_louis, the
|zeta| = 50 clip, the 180 K clamp of e_sat_ice, LU13 as A -> 1 and the regime edges of rough_leng_tq."""
import ctypes as C
import functools
import math

import mpmath as mp
import numpy as np
import pytest

ULP = 2.0 ** -52
N = 1500
rng = np.random.default_rng(20261022)
U = lambda lo, hi, n=N: lo + (hi - lo) * rng.random(n)
LOGU = lambda lo, hi, n=N: 10.0 ** U(math.log10(lo), math.log10(hi), n)
F = lambda x: mp.mpf(float(x))                  # the double a literal or an argument is, exactly


def stable(x):                                   # 0.5 + SIGN(0.5, x) == 1: SIGN takes the sign bit, +0 is stable
    return not math.copysign(1.0, x) < 0


# ---------------------------------------------------------------- mpmath restatement (mp.workdps(50) by the callers)
RTT0, RDG_I, GRAV, RPI = 273.16, 0.7858350313586662, 9.8, 3.141592653589793   # mod_const.f90:38-61, mod_phymbl.f90:147
REPS0 = 287.05 / 461.495                                                         # R_dry / R_vap, folded in FP64
LU13_Y = 1. + 1. / (10. * 1.4)                  # rNu_0 + 1/(10 rbeta_0), mod_cdn_form_ice.f90:196, as gfortran folds it


def e_sat_ice(T):                                # mod_phymbl.f90:815-830
    zta = max(T, 180.)
    ztmp = F(RTT0) / zta
    zle = F(-9.09718) * (ztmp - 1) + F(-3.56654) * mp.log10(ztmp) + F(0.876793) * (1 - zta / F(RTT0)) + F(RDG_I)
    return 100 * mp.power(10, zle)


def q_sat_ice(T, p):                             # :881-904 with l_ice
    es = e_sat_ice(T)
    return F(REPS0) * es / (F(p) - (1 - F(REPS0)) * es)


def psi_ice(z, which):                           # mod_blk_ice_an05.f90:329-405
    if stable(z):
        z = F(z)
        return -(F(0.7) * z + F(0.75) * (z - F(14.3)) * mp.exp(F(-0.35) * z) + F(10.7))
    zx = mp.power(abs(1 - 16 * F(z)), F(0.25))
    if which == "h":
        return 2 * mp.log((1 + zx * zx) / 2)
    return mp.log((1 + zx * zx) / 2) + 2 * mp.log((1 + zx) / 2) - 2 * mp.atan(zx) + F(0.5) * F(RPI)


def f_louis(ra, zu, rib, cxn, z0):               # mod_phymbl.f90:1419-1479, rc_louis = 5
    R = F(rib)
    if stable(rib):
        return 1 / (1 + ra * R / mp.sqrt(abs(1 + R)))
    ztu = R / (1 + 3 * 25 * F(cxn) * mp.sqrt(abs(-R * (F(zu) / F(z0) + 1))))
    return 1 - ra * ztu


def rough_leng_m(us, nu):                        # mod_blk_ice_an05.f90:247-268
    zus = F(max(us, 1.E-9))
    zz = (zus - F(0.18)) / F(0.1)
    return F(0.135) * F(nu) / zus + F(0.035) * zus * zus / F(GRAV) * (5 * mp.exp(-zz * zz) + 1)


def an87_zre(z0, us, nu):                        # R* as the reference computes it in FP64 (:288)
    return max(max(us, 1.E-9) * z0 / nu, 0.)


def an87_regime(zre):                            # the three SIGN masks of :289-292; none of them in ]2.49999, 2.5[
    if zre <= 0.135:
        return "smooth"
    if zre <= 2.49999:
        return "trans"
    return "rough" if zre >= 2.5 else "stop"


AN87 = {"smooth": ((1.25, 0., 0.), (1.61, 0., 0.)), "trans": ((0.149, -0.550, 0.), (0.351, -0.628, 0.)),
        "rough": ((0.317, -0.565, -0.183), (0.396, -0.512, -0.180))}


def z0tq_an87(z0, us, nu, regime, iq):           # :298-323; iq 0: z0t, 1: z0q
    zlog = mp.log(F(max(us, 1.E-9)) * F(z0) / F(nu))
    b0, b1, b2 = AN87[regime][iq]
    return F(z0) * mp.exp(F(b0) + F(b1) * zlog + F(b2) * zlog * zlog)


def cdn10_lu13(A):                               # mod_cdn_form_ice.f90:170-208 (A**(mu-1) == 1)
    return F(2.23E-3) * mp.power(F(1. - A), F(LU13_Y))


def lg15_log_ratio(zu, z0w=4.54e-4):             # :322, on the host with glibc as make_ice_uniform computes it
    t = 1. / z0w
    return math.log(10. * t) / math.log(zu * t)


def cdn_lg15(lr, A):                             # :299-330 (Eq.46)
    return F(3.46e-3) * F(lr) * F(lr) * F(A) * mp.power(F(1. - A), F(1.4))


# ---------------------------------------------------------------- argument sets
def _pm(a):
    return np.concatenate([a, -a])


T_ICE = np.concatenate([U(150.0, 300.0), [180.0, 179.9, 273.16, 150.0, 300.0, np.nextafter(180.0, 0.0),
                                          np.nextafter(180.0, 300.0)]])
ZETA = np.concatenate([U(-50.0, 50.0), _pm(10.0 ** U(-12, 0, N // 4)), [0.0, -0.0, 1e-300, -1e-300],
                       _pm(np.array([50.0, np.nextafter(50.0, 0.0), np.nextafter(50.0, 100.0), 49.999999, 50.000001]))])
RIB = np.concatenate([U(-20.0, 20.0), _pm(10.0 ** U(-12, 0, N // 4)), [0.0, -0.0, 1e-300, -1e-300, 20.0, -20.0]])
US_M = np.concatenate([[0.0, 1e-12, 1e-9], U(1e-4, 2.0), 0.18 + U(-0.03, 0.03, N // 2), [0.18, 0.08, 0.28]])
A_LU13 = np.concatenate([U(0.0, 1.0), [0.0, 1.0, 0.5], 1.0 - 2.0 ** -np.arange(1.0, 51.0)])
A_LG15 = np.concatenate([U(0.0, 1.0), [0.0, 1.0, 0.5]])
ZU_LG15 = U(2.0, 10.0, A_LG15.size)
LR_LG15 = np.array([lg15_log_ratio(zu) for zu in ZU_LG15])

# name -> (restatement on the probe's arguments, oracle export on them, probe arguments, bound, floor, reference file:line)
# err = |x - ref| / max(|ref|, floor); floor 0 is relative and requires x == 0 where ref == 0.  A callable bound is per point.
CASES = {
    "e_sat_ice": (e_sat_ice, lambda L, T: L.abo_e_sat_ice(T), (T_ICE,), 2e-14, 0.0, "mod_phymbl.f90:815-830"),
    "q_sat_ice": (q_sat_ice, lambda L, T, p: L.abo_q_sat_ice(T, p), (T_ICE, U(60000.0, 110000.0, T_ICE.size)), 2e-14, 0.0,
                  "mod_phymbl.f90:881-904"),
    "psi_m_ice": (lambda z: psi_ice(z, "m"), lambda L, z: L.abo_psi_m_ice(z), (ZETA,), 2e-14, 1.0,
                  "mod_blk_ice_an05.f90:329-366"),
    "psi_h_ice": (lambda z: psi_ice(z, "h"), lambda L, z: L.abo_psi_h_ice(z), (ZETA,), 2e-14, 1.0,
                  "mod_blk_ice_an05.f90:368-405"),
    "f_m_louis": (lambda *a: f_louis(10, *a), lambda L, *a: L.abo_f_m_louis(*a),
                  (U(2.0, 10.0, RIB.size), RIB, LOGU(1e-4, 5e-3, RIB.size), LOGU(4.5e-4, 2e-3, RIB.size)), 1e-14, 0.0,
                  "mod_phymbl.f90:1419-1440"),
    "f_h_louis": (lambda *a: f_louis(15, *a), lambda L, *a: L.abo_f_h_louis(*a),
                  (U(2.0, 10.0, RIB.size), RIB, LOGU(1e-4, 5e-3, RIB.size), LOGU(4.5e-4, 2e-3, RIB.size)), 1e-14, 0.0,
                  "mod_phymbl.f90:1458-1479"),
    "rough_leng_m": (rough_leng_m, lambda L, us, nu: L.abo_rough_leng_m(us, nu), (US_M, U(1.2e-5, 1.8e-5, US_M.size)),
                     1e-14, 0.0, "mod_blk_ice_an05.f90:247-268"),
    # x**y on the device is exp(y log x): the error of the logarithm is amplified by |y log x| (the powr rule of
    # tests/test_math_accuracy.py), here up to 37 at A = 1 - 2**-50
    "CdN10_f_LU13": (cdn10_lu13, lambda L, A: L.abo_CdN10_f_LU13(A), (A_LU13,),
                     lambda A: (4 + 2 * np.abs(LU13_Y * np.log(np.maximum(1.0 - A, 1e-300)))) * ULP, 0.0,
                     "mod_cdn_form_ice.f90:170-208"),
    # the probe takes (log_ratio, A) and ignores zu; the oracle takes zu and computes the ratio itself
    "CdN_f_LG15_light": (lambda lr, A, zu: cdn_lg15(lr, A), lambda L, lr, A, zu: L.abo_CdN_f_LG15_light(zu, A, 4.54e-4),
                         (LR_LG15, A_LG15, ZU_LG15), 1e-14, 0.0, "mod_cdn_form_ice.f90:299-330"),
}


@functools.lru_cache(maxsize=None)
def _reference(name):
    ref_fn, _, cols, *_ = CASES[name]
    with mp.workdps(50):
        return [ref_fn(*[float(c[i]) for c in cols]) for i in range(cols[0].size)]


def _errors(got, ref, floor):
    err = np.empty(len(ref))
    for i, (g, r) in enumerate(zip(got, ref)):
        if r == 0 and floor == 0.0:
            err[i] = 0.0 if g == 0.0 else np.inf
        else:
            err[i] = float(abs(mp.mpf(float(g)) - r) / max(abs(r), floor))
    return err


def _bound(bound, cols):
    return bound(*cols) if callable(bound) else np.full(cols[0].size, bound)


@pytest.fixture(scope="module")
def OL():
    from oracle import oracle
    return oracle.lib()


@pytest.mark.parametrize("name", sorted(CASES))
def test_restatement_matches_oracle(OL, name):
    """CPU: the mpmath restatement against the oracle's glibc evaluation of the same formula (no GPU needed)."""
    _, get, cols, bound, floor, where = CASES[name]
    got = np.array([get(OL, *[float(c[i]) for c in cols]) for i in range(cols[0].size)])
    err = _errors(got, _reference(name), floor)
    b = _bound(bound, cols)       # the device's bound: glibc's pow / exp / log are within 1 ulp, the device's within 4
    print(f"[restatement] {name:18s} ({where}): oracle vs mpmath max err {err.max():.2e}, worst err/bound {(err / b).max():.2f}")
    assert (err <= b).all(), (name, float(err.max()), [float(c[(err / b).argmax()]) for c in cols])


def test_rough_leng_tq_restatement_matches_oracle(OL):
    """CPU: regime choice and z0t / z0q of the restatement against abo_rough_leng_tq, on the random and the edge sets."""
    z0t, z0q = C.c_double(), C.c_double()
    worst = 0.0
    for z0, us, nu in list(zip(*AN87_RANDOM)) + [p[:3] for p in AN87_EDGES]:
        bad = OL.abo_rough_leng_tq(z0, us, nu, C.byref(z0t), C.byref(z0q))
        regime = an87_regime(an87_zre(z0, us, nu))
        assert bad == (regime == "stop"), (z0, us, nu)
        if bad:
            continue
        with mp.workdps(50):
            for iq, v in enumerate((z0t.value, z0q.value)):
                r = z0tq_an87(z0, us, nu, regime, iq)
                worst = max(worst, float(abs(v - r) / r))
    print(f"[restatement] rough_leng_tq: oracle vs mpmath max rel err {worst:.2e}")
    assert worst <= 2e-14


# ---------------------------------------------------------------- Andreas 1987: random R* and the regime edges
def _an87_random():
    rstar = LOGU(1e-3, 1e3)
    us, nu = LOGU(1e-2, 1.0), U(1.2e-5, 1.8e-5)
    return rstar * nu / us, us, nu


AN87_RANDOM = _an87_random()
AN87_EDGE_VALUES = (0.135, 2.49999, 2.5)


def _ulp_steps(e, k):
    x = e
    for _ in range(abs(k)):
        x = np.nextafter(x, np.inf if k > 0 else -np.inf)
    return float(x)


def _an87_edges():
    """(z0, us, nu, edge, k, exact): points whose FP64 R* = us*z0/nu is k ulp from an edge.  `exact` marks a power-of-two
    us and nu (nu = 2**-16 = 1.53e-5, inside the range of visc_air): there fdiv(us*z0, nu) on the device is exact, so
    its R* is the reference's to the bit.  Elsewhere z0 is searched ulp by ulp; an offset the map z0 -> R* skips is left
    out."""
    pts = []
    for e in AN87_EDGE_VALUES:
        for k in range(-8, 9):
            t = _ulp_steps(e, k)
            pts.append((t * 2.0 ** -16 / 0.25, 0.25, 2.0 ** -16, e, k, True))
            for us, nu in ((0.21, 1.37e-5), (0.0437, 1.71e-5), (0.733, 1.23e-5)):
                z0 = t * nu / us
                for _ in range(64):
                    r = an87_zre(z0, us, nu)
                    if r == t:
                        pts.append((z0, us, nu, e, k, False))
                        break
                    z0 = float(np.nextafter(z0, np.inf if r < t else -np.inf))
    for r in (2.499991, 2.499995, 2.4999999, (2.49999 + 2.5) / 2):   # strictly inside the gap of the reference
        pts.append((r * 2.0 ** -16 / 0.25, 0.25, 2.0 ** -16, None, None, True))
        pts.append((r * 1.37e-5 / 0.21, 0.21, 1.37e-5, None, None, False))
    return pts


AN87_EDGES = _an87_edges()


def test_an87_edge_points_cover_every_offset():
    """CPU: the edge set reaches R* = e + k ulp for every edge and every |k| <= 8 (bit-exact points: all of them)."""
    for e in AN87_EDGE_VALUES:
        exact = {p[4] for p in AN87_EDGES if p[3] == e and p[5]}
        other = [p[4] for p in AN87_EDGES if p[3] == e and not p[5]]
        assert exact == set(range(-8, 9)), e
        assert len(other) >= 30 and {-4, 0, 4} & set(other), (e, sorted(other))
        for z0, us, nu, _, k, _ in (p for p in AN87_EDGES if p[3] == e):
            assert an87_zre(z0, us, nu) == _ulp_steps(e, k)


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    ab.reset()
    return ab


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_device_ice_function(ab, name):
    _, _, cols, bound, floor, where = CASES[name]
    got = ab.probe(name, *cols)
    assert np.isfinite(got).all(), name
    err = _errors(got, _reference(name), floor)
    b = _bound(bound, cols)
    print(f"[function] {name:18s} ({where}): max err {err.max():.2e} over {err.size} points "
          f"(bound {'per point' if callable(bound) else f'{bound:.0e}'}; worst err/bound {(err / b).max():.2f})")
    assert (err <= b).all(), (name, float(err.max()), [float(c[(err / b).argmax()]) for c in cols])


@pytest.mark.gpu
def test_device_ice_exact_values(ab):
    """The quirks the reference has at its branch points, held to the bit (to rounding for psi(+0))."""
    z = np.array([0.0, -0.0, 1e-300, -1e-300])
    for which in ("m", "h"):
        got = ab.probe(f"psi_{which}_ice", z)
        # SIGN(0.5, +0) selects the stable side: -(0.75 (0 - 14.3) + 10.7) = 0.025 up to the rounding of 10.725 - 10.7
        assert abs(got[0] - 0.025) <= 4 * np.spacing(10.7) and abs(got[2] - 0.025) <= 4 * np.spacing(10.7), (which, got)
        assert got[1] == 0.0 and got[3] == 0.0, (which, got)        # -0: the unstable side, x = 1, every term cancels
    rib = np.array([0.0, -0.0, 1e-300, -1e-300])
    for which in ("m", "h"):
        got = ab.probe(f"f_{which}_louis", np.full(4, 10.0), rib, np.full(4, 1.5e-3), np.full(4, 1e-3))
        assert (got == 1.0).all(), (which, got)
    assert (ab.probe("CdN10_f_LU13", np.array([1.0, 0.0])) == np.array([0.0, 2.23e-3])).all()
    assert (ab.probe("CdN_f_LG15_light", np.full(2, LR_LG15[0]), np.array([0.0, 1.0])) == 0.0).all()
    # e_sat_ice clamps at 180 K: every T below gives e_sat_ice(180) exactly
    t = np.array([180.0, 179.9, 150.0, np.nextafter(180.0, 0.0), 100.0])
    got = ab.probe("e_sat_ice", t)
    assert (got == got[0]).all(), got


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["z0t", "z0q"])
def test_device_rough_leng_tq(ab, OL, which):
    """Andreas 1987 (mod_blk_ice_an05.f90:270-325) as solve_ice evaluates it: log_rough_leng_tq(z0, dlog(z0), u*, nu).

    The device computes R* with fdiv (within 1.5 ulp of the IEEE quotient), so within a few ulp of a regime edge it may
    pick the other side.  Rules, with k the distance of the reference's FP64 R* from the nearest edge in ulp:
    - bit-exact points (power-of-two u* and nu: the device's R* is the reference's): the reference's regime, always;
    - |k| > 4: NaN exactly where abo_rough_leng_tq stops, otherwise the mpmath value of the reference's regime;
    - |k| <= 4: the mpmath value of the regime on either side of the edge, or NaN where that side is the stop window.
    Values within 2e-13 relative: the evaluation is in log space, where |LOG(z0t)| <= 21 amplifies the ulps (as
    z0tq_LKB)."""
    iq = 0 if which == "z0t" else 1
    z0r, usr, nur = AN87_RANDOM
    pts = [(float(a), float(b), float(c), None, None, False) for a, b, c in zip(z0r, usr, nur)] + AN87_EDGES
    z0, us, nu = (np.array([p[i] for p in pts]) for i in range(3))
    got = ab.probe(f"{which}_an87", z0, us, nu)
    zt, zq = C.c_double(), C.c_double()
    worst, n_near = 0.0, 0
    with mp.workdps(50):
        for i, (a, b, c, e, k, exact) in enumerate(pts):
            zre = an87_zre(a, b, c)
            regime = an87_regime(zre)
            assert (OL.abo_rough_leng_tq(a, b, c, C.byref(zt), C.byref(zq)) == 1) == (regime == "stop")
            dist = min(abs(zre - x) / np.spacing(x) for x in AN87_EDGE_VALUES)
            if exact or dist > 4:
                allowed = {regime}
            else:
                n_near += 1
                edge = min(AN87_EDGE_VALUES, key=lambda x: abs(zre - x))
                allowed = {an87_regime(float(np.nextafter(edge, -np.inf))), an87_regime(float(np.nextafter(edge, np.inf)))}
            g = float(got[i])
            ok, errs = False, []
            for r in allowed:
                if r == "stop":
                    ok |= math.isnan(g)
                    continue
                ref = z0tq_an87(a, b, c, r, iq)
                err = float(abs(mp.mpf(g) - ref) / ref) if math.isfinite(g) else math.inf
                errs.append(err)
                ok |= err <= 2e-13
            assert ok, (which, a, b, c, zre, e, k, exact, sorted(allowed), g, errs)
            if errs and min(errs) <= 2e-13:
                worst = max(worst, min(errs))
    print(f"[function] {which}_an87 (mod_blk_ice_an05.f90:270-325): max rel err {worst:.2e} over {len(pts)} points "
          f"({n_near} within 4 ulp of a regime edge)")
    assert n_near >= 50
