#!/usr/bin/env python
"""Generates aerobulk_b200/csrc/ab_math_tables.cuh: polynomial coefficients (FP64, in __constant__ memory)
of the kernel's own exp / log / atan and the piecewise polynomial of Goff's saturation vapour pressure.
Coefficients are Chebyshev-node interpolants computed with mpmath at 200 bits and rounded to double; the
script prints the worst error of each rounded polynomial.

Why own tables: ptxas materialises every FP64 literal of CUDA's libdevice math with two 32-bit moves
(UMOV/IMAD.MOV), ~35 % of all issued instructions of the flux kernels; coefficients read from the
constant bank cost 0.5 instruction each (LDCU.128 loads two).
"""
import os
import sys
import mpmath as mp

mp.mp.prec = 200
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "..", "aerobulk_b200", "csrc", "ab_math_tables.cuh")


def cheb_fit(f, a, b, deg):
    """Monomial coefficients (in x) of the degree-`deg` interpolant of f at Chebyshev nodes of [a,b]."""
    n = deg + 1
    xs = [(a + b) / 2 + (b - a) / 2 * mp.cos(mp.pi * (2 * k + 1) / (2 * n)) for k in range(n)]
    A = mp.matrix(n, n)
    y = mp.matrix(n, 1)
    for i, x in enumerate(xs):
        for j in range(n):
            A[i, j] = x ** j
        y[i] = f(x)
    c = mp.lu_solve(A, y)
    return [c[i] for i in range(n)]


def horner_double(cs, x):
    """Evaluate with FP64-rounded coefficients but exact arithmetic (isolates approximation error)."""
    r = mp.mpf(0)
    for c in reversed(cs):
        r = r * x + mp.mpf(float(c))
    return r


def max_err(f, cs, a, b, rel=True, n=4001):
    worst = mp.mpf(0)
    for k in range(n):
        x = a + (b - a) * k / (n - 1)
        fx = f(x)
        e = abs(horner_double(cs, x) - fx)
        if rel and fx != 0:
            e = e / abs(fx)
        worst = max(worst, e)
    return worst


def emit(name, cs, comment):
    s = f"// {comment}\nABM_TABLE double {name}[{len(cs)}] = {{\n"
    s += ",\n".join(f"    {float(c).hex()}  /* {float(c):+.17e} */" for c in cs)
    return s + "\n};\n\n"


# ---- unstable stability functions psi(zeta), zeta in [-PSI_ZMAX, 0], as piecewise polynomials of |zeta|.  Row 0 covers
# |zeta| < 2^PSI_E0 with a polynomial in u = |zeta| whose constant term is 0 (psi(-0) = 0, and absolute accuracy at the
# tiny zeta of the roughness heights); row 1 + 2^PSI_K (e - PSI_E0) + j covers [2^e (1 + j 2^-K), 2^e (1 + (j+1) 2^-K))
# with a polynomial in u = |zeta| - c, c its centre: the row index and c come from the high word of |zeta| and u is exact.
# The nearest singularities are branch points on the stable side (zeta = 1/34.15, 1/15, 1/10.15 for COARE, 1/16 for
# Paulson) and the poles of zeta^2/(1+zeta^2) at +-i; with 2^PSI_K intervals per binade every interval is at least
# 2^(K+1) + 1 of its half-widths away from them.  The COARE functions are written as mod_common_coare.f90 writes them, with
# its truncated literals (as doubles, like the reference build).
PSI_E0, PSI_K, PSI_DEG, PSI_ZMAX = -7, 2, 11, 50


def _lit(s):
    return mp.mpf(float(s))


def psi_coare_m(z):
    phi_m = mp.power(1 - 15 * z, mp.mpf(1) / 4)
    k = 2 * mp.log((1 + phi_m) / 2) + mp.log((1 + phi_m * phi_m) / 2) - 2 * mp.atan(phi_m) + mp.pi / 2
    return _coare_blend(z, k, _coare_conv(mp.power(1 - _lit("10.15") * z, _lit(".3333"))))


def psi_coare_h(z):
    k = 2 * mp.log((1 + mp.sqrt(1 - 15 * z)) / 2)
    return _coare_blend(z, k, _coare_conv(mp.power(1 - _lit("34.15") * z, _lit(".3333"))))


def _coare_conv(phi):
    return (mp.mpf("1.5") * mp.log((1 + phi + phi * phi) / 3) - _lit("1.7320508") * mp.atan((1 + 2 * phi) / _lit("1.7320508"))
            + _lit("1.813799447"))


def _coare_blend(z, k, c):
    f = z * z / (1 + z * z)
    return (1 - f) * k + f * c


def psi_paulson_m(z):
    x = mp.power(1 - 16 * z, mp.mpf(1) / 4)
    return 2 * mp.log((1 + x) / 2) + mp.log((1 + x * x) / 2) - 2 * mp.atan(x) + mp.pi / 2


def psi_paulson_h(z):
    return 2 * mp.log((1 + mp.sqrt(1 - 16 * z)) / 2)


PSI_FUNCS = {"COARE": (psi_coare_m, psi_coare_h), "PAULSON": (psi_paulson_m, psi_paulson_h)}


def psi_rows(e0, k):
    """[(lo, hi, centre)] of |zeta| for every row."""
    rows = [(mp.mpf(0), mp.mpf(2) ** e0, mp.mpf(0))]
    e = e0
    while rows[-1][1] < PSI_ZMAX:
        for j in range(2 ** k):
            lo = mp.mpf(2) ** e * (1 + mp.mpf(j) / 2 ** k)
            hi = lo + mp.mpf(2) ** (e - k)
            rows.append((lo, hi, (lo + hi) / 2))
            if hi > PSI_ZMAX:
                break
        e += 1
    return rows


def psi_fit(psi, row, deg):
    """FP64 coefficients c_0..c_deg of the row's polynomial in u (u = |zeta| - centre)."""
    lo, hi, c = row
    if c == 0:     # row 0: u * q(u), q of degree deg - 1
        q = cheb_fit(lambda u: psi(-u) / u, lo, hi, deg - 1)
        return [0.0] + [float(x) for x in q]
    return [float(x) for x in cheb_fit(lambda u: psi(-(c + u)), lo - c, hi - c, deg)]


def psi_err(psi, row, cs, n=61):
    """Worst |p(u) - psi| / max(|psi|, 1) over the row (FP64 coefficients, exact arithmetic), both ends included."""
    lo, hi, c = row
    worst = mp.mpf(0)
    for i in range(n):
        a = lo + (hi - lo) * i / (n - 1)
        ref = psi(-a) if a != 0 else mp.mpf(0)
        worst = max(worst, abs(horner_double(cs, a - c) - ref) / max(abs(ref), 1))
    return worst


def psi_tables(deg=PSI_DEG, e0=PSI_E0, k=PSI_K, quiet=False):
    """Header text of the psi tables and the worst error of each.  In a table, pair j = (c_2j, c_2j+1) of row r is
    double2 number j * PSI_ROWS + r (pair j of every row contiguous: lanes on different rows hit different banks), psi_m's
    pairs first, then psi_h's."""
    rows = psi_rows(e0, k)
    text = ("// unstable psi_m, psi_h for zeta in [-%d, 0] as piecewise polynomials of degree %d in u = |zeta| - c: row 0 is\n"
            "// |zeta| < 2^%d (c = 0, c_0 = 0), row 1 + %d (e - %d) + j is [2^e (1 + j/%d), 2^e (1 + (j+1)/%d)), c its centre\n"
            "constexpr int PSI_E0 = %d, PSI_K = %d, PSI_DEG = %d, PSI_ROWS = %d;\nconstexpr double PSI_ZMAX = %d.;\n"
            % (PSI_ZMAX, deg, e0, 2 ** k, e0, 2 ** k, 2 ** k, e0, k, deg, len(rows), PSI_ZMAX))
    worst = {}
    for fam, fns in PSI_FUNCS.items():
        tabs = []
        for name, psi in zip("mh", fns):
            coefs = [psi_fit(psi, r, deg) for r in rows]
            errs = [psi_err(psi, r, cs) for r, cs in zip(rows, coefs)]
            i = max(range(len(rows)), key=lambda i: errs[i])
            worst[fam + "_" + name] = errs[i]
            if not quiet:
                print("psi_%s %-7s deg %d, %d rows: worst |err| / max(|psi|, 1) %.3e (2^%.1f) on |zeta| in [%.4g, %.4g]"
                      % (name, fam, deg, len(rows), errs[i], mp.log(errs[i], 2), rows[i][0], rows[i][1]))
            tabs.append(coefs)
        text += ("// %s: worst |err| / max(|psi|, 1) of psi_m %.2e, psi_h %.2e (coefficients rounded, exact arithmetic)\n"
                 "alignas(16) ABM_GTABLE double PSI_%s_T[%d] = {\n"
                 % (fam, worst[fam + "_m"], worst[fam + "_h"], fam, 2 * len(rows) * (deg + 1)) +
                 ",\n".join(f"    {cs[2 * j].hex()}, {cs[2 * j + 1].hex()}"
                            for coefs in tabs for j in range((deg + 1) // 2) for cs in coefs) + "\n};\n")
    return text + "\n", worst


def main():
    parts = ["// GENERATED by tools/gen_math_tables.py -- do not edit.\n#pragma once\n\n"
             "#ifndef ABM_TABLE\n#define ABM_TABLE __constant__\n#endif\n"
             "#ifndef ABM_GTABLE\n#define ABM_GTABLE __device__ const\n#endif\n\nnamespace abm {\n\n"]
    ln2 = mp.log(2)

    # EXP_C, LOG_C and the MATH_K entries L2E, L2T, LG2_HI, LG2_LO belong to the polynomial exp / exp10 / log, which the
    # table-driven ones replaced: no code reads them.  They stay because ptxas pairs constant loads into LDCU.128 by their
    # offsets in constant bank 3, which follow from every table declared before them.  Deleting the tables re-pairs the loads
    # of every flux kernel; aligning every table to 16 bytes, which makes the deletion neutral, by itself changes the
    # registers and spills of 61 of the 126 kernels and made ANDREAS 3.9 % slower on a B200 (profiles/sass_compare_r03e.txt,
    # profiles/ptxas_align_r03e.txt, profiles/kbench_4320x2160_r03e.txt).
    # exp(r), |r| <= ln2/2, degree 11
    a = ln2 / 2 * mp.mpf("1.0001")
    cs = cheb_fit(mp.exp, -a, a, 11)
    e = max_err(mp.exp, cs, -a, a)
    print("exp  deg 11 rel err %.3e (2^%.1f)" % (e, mp.log(e, 2)))
    parts.append(emit("EXP_C", cs, "exp(r) on |r| <= ln2/2, c0..c11; max rel err %.2e (read by no kernel, kept for the bank layout)" % e))

    # log: P(z) = (2 atanh(s) - 2 s) / s^3 with z = s^2, s in [0, 0.1716]; log(m) = 2s + s*z*P(z)
    zmax = ((mp.sqrt(2) - 1) / (mp.sqrt(2) + 1)) ** 2 * mp.mpf("1.001")

    def P(z):
        if z == 0:
            return mp.mpf(2) / 3
        s = mp.sqrt(z)
        return (2 * mp.atanh(s) - 2 * s) / (s * z)
    for deg in (6, 7):
        cs = cheb_fit(P, mp.mpf(0), zmax, deg)
        e = max_err(P, cs, mp.mpf(0), zmax)
        # error contribution relative to log(m) ~ 2s: s*z*dP / (2s) = z*dP/2
        print("log  deg %d rel err of P %.3e -> rel err of log <= %.3e" % (deg, e, e * zmax / 2 * mp.mpf(2) / 3))
    cs = cheb_fit(P, mp.mpf(0), zmax, 6)
    parts.append(emit("LOG_C", cs, "(2 atanh(s) - 2s)/s^3 in z = s^2 on [0, 0.0295], c0..c6 (read by no kernel, kept for the bank layout)"))

    # atan(t) = t + t*z*Q(z), z = t^2, |t| <= tan(pi/8); Q(z) = (atan(t) - t)/t^3
    tmax = mp.tan(mp.pi / 8) * mp.mpf("1.0001")

    def Q(z):
        if z == 0:
            return -mp.mpf(1) / 3
        t = mp.sqrt(z)
        return (mp.atan(t) - t) / (t * z)
    for deg in (9, 10, 11, 12):
        cs = cheb_fit(Q, mp.mpf(0), tmax ** 2, deg)
        e = max_err(Q, cs, mp.mpf(0), tmax ** 2)
        print("atan deg %d rel err of Q %.3e -> rel err of atan <= %.3e" % (deg, e, e * tmax ** 2 / 3))
    cs = cheb_fit(Q, mp.mpf(0), tmax ** 2, 10)
    parts.append(emit("ATAN_C", cs, "(atan(t) - t)/t^3 in z = t^2 on [0, tan(pi/8)^2], c0..c10"))

    # ---- table-driven exp: exp(x) = 2^m * T[j] * exp(r), k = 64 m + j = rint(x 64/ln2), |r| <= ln2/128
    a = ln2 / 128 * mp.mpf("1.001")

    def QE(r):
        return mp.mpf(1) / 2 + r / 6 if abs(r) < mp.mpf(10) ** -20 else (mp.exp(r) - 1 - r) / (r * r)
    cs = cheb_fit(QE, -a, a, 3)
    e = max_err(QE, cs, -a, a)
    print("exp(table) q deg 3: rel err of q %.3e -> rel err of exp <= %.3e" % (e, e * a * a))
    parts.append(emit("EXPT_C", cs, "(exp(r) - 1 - r)/r^2 on |r| <= ln2/128, c0..c3"))
    tab = [mp.mpf(2) ** (mp.mpf(j) / 64) for j in range(64)]
    parts.append("// 2^(j/64), j = 0..63 (copied to shared memory by abm::load_tables)\nABM_GTABLE double EXP_T[64] = {\n" +
                 ",\n".join(f"    {float(t).hex()}" for t in tab) + "\n};\n\n")

    # ---- table-driven log: m in [0.708, 1.416) cut into 256 intervals of 4096 hi-word units; c_j = centre
    # (c_149 = 1 exactly), rc_j = fl(1/c_j), lc_j = fl(-log(rc_j)); log(m) = lc_j + log1p(m rc_j - 1)
    import struct
    BASE = 0x3fe6a800
    rows = []
    for j in range(256):
        hi = BASE + j * 4096 + 2048
        c = struct.unpack("<d", struct.pack("<Q", hi << 32))[0]
        rc = float(mp.mpf(1) / mp.mpf(c))
        lc = float(-mp.log(mp.mpf(rc)))
        rows.append((rc, lc))
    assert rows[149] == (1.0, 0.0) or rows[149] == (1.0, -0.0), rows[149]
    rmax = mp.mpf(2) ** -9 * mp.mpf("1.01")

    def QL(r):
        return -mp.mpf(1) / 2 + r / 3 if abs(r) < mp.mpf(10) ** -20 else (mp.log1p(r) - r) / (r * r)
    cs = cheb_fit(QL, -rmax, rmax, 4)
    e = max_err(QL, cs, -rmax, rmax)
    print("log(table) q deg 4: rel err of q %.3e -> rel err of log1p <= %.3e" % (e, e * rmax))
    parts.append(emit("LOGT_C", cs, "(log1p(r) - r)/r^2 on |r| <= 2^-9, c0..c4"))
    parts.append("// {1/c_j, -log(1/c_j)} for the 256 mantissa intervals (hi word 0x%x + 4096 j ...)\n"
                 "ABM_GTABLE double LOG_T[512] = {\n" % BASE +
                 ",\n".join(f"    {rc.hex()}, {(lc + 0.0).hex()}" for rc, lc in rows) + "\n};\n\n")

    # ---- Goff (1957) saturation vapour pressure over water [Pa], written as abd::e_sat writes it (rt0 = 273.15, the
    # reference's literals), as one degree-7 polynomial per interval of h = 2 K (a power of two: the argument reduction
    # is exact).  Interval m is centred on T_c = h m, so rint(T / h) selects it and x = (T - T_c) (2 / h) is in [-1, 1].
    # Rows m = 115..165 cover [229, 331); e_sat takes the table on [230, 330).  The table is four arrays of coefficient
    # pairs (c0 c1 | c2 c3 | c4 c5 | c6 c7) indexed by row, so a row is four 16-byte loads and lanes that read different
    # rows hit different shared-memory banks (with 64-byte rows side by side, every row maps onto one of two bank groups).
    rt0 = mp.mpf("273.15")

    def goff(T):
        z = rt0 / T
        r = T / rt0
        return 100 * mp.power(10, mp.mpf("10.79574") * (1 - z) - mp.mpf("5.028") * mp.log10(r)
                              + mp.mpf("1.50475e-4") * (1 - mp.power(10, mp.mpf("-8.2969") * (r - 1)))
                              + mp.mpf("0.42873e-3") * (mp.power(10, mp.mpf("4.76955") * (1 - z)) - 1)
                              + mp.mpf("0.78614"))
    ESAT_H, ESAT_DEG, ESAT_M0, ESAT_M1 = 2, 7, 115, 165
    rows, worst = [], (mp.mpf(0), 0)
    for m in range(ESAT_M0, ESAT_M1 + 1):
        Tc = mp.mpf(ESAT_H * m)
        g = lambda x, Tc=Tc: goff(Tc + x * ESAT_H / 2)
        cs = cheb_fit(g, mp.mpf(-1), mp.mpf(1), ESAT_DEG)
        worst = max(worst, (max_err(g, cs, mp.mpf(-1), mp.mpf(1), n=201), ESAT_H * m))
        rows.append(cs)
    print("e_sat table: %d x 2 K, deg %d: worst rel err %.3e (2^%.1f) in the interval centred on %d K"
          % (len(rows), ESAT_DEG, worst[0], mp.log(worst[0], 2), worst[1]))
    parts.append("// Goff (1957) e_sat [Pa] on [T_c - h/2, T_c + h/2], T_c = h m, m = %d..%d: c0..c%d in x = (T - T_c) (2 / h),\n"
                 "// pair j = (c_2j, c_2j+1) of row m - %d at [j][m - %d]; worst rel err %.2e (coefficients rounded, exact arithmetic)\n"
                 "constexpr double ESAT_H = %d.;\nconstexpr int ESAT_M0 = %d, ESAT_ROWS = %d;\n"
                 "alignas(16) ABM_GTABLE double ESAT_T[%d] = {\n"
                 % (ESAT_M0, ESAT_M1, ESAT_DEG, ESAT_M0, ESAT_M0, worst[0], ESAT_H, ESAT_M0, len(rows), len(rows) * (ESAT_DEG + 1)) +
                 ",\n".join(f"    {float(cs[2 * j]).hex()}, {float(cs[2 * j + 1]).hex()}"
                             for j in range((ESAT_DEG + 1) // 2) for cs in rows) + "\n};\n\n")

    parts.append(psi_tables()[0])

    def hilo(x):
        hi = float(x)
        # keep the low 21 bits of hi's mantissa free so that k*hi is exact for |k| < 2^11
        import struct
        b = struct.unpack("<Q", struct.pack("<d", hi))[0] & ~((1 << 21) - 1)
        hi = struct.unpack("<d", struct.pack("<Q", b))[0]
        lo = float(x - mp.mpf(hi))
        return hi, lo
    l2h, l2l = hilo(ln2)
    lg2h, lg2l = hilo(mp.log10(2))
    consts = {
        "LN2_HI": l2h, "LN2_LO": l2l, "L2E": float(1 / ln2),
        "L2E64": float(64 / ln2), "LN2_64_HI": hilo(ln2 / 64)[0], "LN2_64_LO": hilo(ln2 / 64)[1],
        "L2T64": float(64 * mp.log(10, 2)), "LG2_64_HI": hilo(mp.log10(2) / 64)[0], "LG2_64_LO": hilo(mp.log10(2) / 64)[1],
        "LG2_HI": lg2h, "LG2_LO": lg2l, "L2T": float(mp.log(10, 2)), "LN10": float(mp.log(10)),
        "LOG10E": float(1 / mp.log(10)),
        "PIO2_HI": float(mp.pi / 2), "PIO2_LO": float(mp.pi / 2 - mp.mpf(float(mp.pi / 2))),
        "PIO4_HI": float(mp.pi / 4), "PIO4_LO": float(mp.pi / 4 - mp.mpf(float(mp.pi / 4))),
        # atan range thresholds tan(3 pi/8), tan(pi/8) and the series coefficients of the root functions
        "TAN3PIO8": 2.414213562373095, "TANPIO8": 0.4142135623730950, "TWO_NINTHS": 2.0 / 9.0, "ONE_THIRD": 1.0 / 3.0,
        # datan_ge1: atan(x) = atan(c) + atan((x - c) / (1 + c x)) with c = the double TAN3PIO8 above; atan(c) as hi + lo
        "ATANC_HI": float(mp.atan(mp.mpf(2.414213562373095))),
        "ATANC_LO": float(mp.atan(mp.mpf(2.414213562373095)) - mp.mpf(float(mp.atan(mp.mpf(2.414213562373095))))),
    }
    parts.append("// scalar constants (hi parts of ln2 / log10(2) have 21 trailing zero bits: k*hi is exact)\n")
    parts.append("ABM_TABLE double MATH_K[%d] = {\n" % len(consts))
    parts.append(",\n".join(f"    {v.hex()}  /* {k} = {v:+.17e} */" for k, v in consts.items()))
    parts.append("\n};\nenum {" + ", ".join(f"K_{k} = {i}" for i, k in enumerate(consts)) + "};\n\n}  // namespace abm\n")
    text = "".join(parts)
    if "--check" in sys.argv:      # the committed header is what this script generates
        if open(OUT).read() != text:
            print("STALE:", os.path.normpath(OUT))
            sys.exit(1)
        print("up to date:", os.path.normpath(OUT))
        return
    with open(OUT, "w") as f:
        f.write(text)
    print("wrote", os.path.normpath(OUT))


if __name__ == "__main__":
    main()
