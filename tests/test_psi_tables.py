"""The unstable stability functions from the piecewise polynomials PSI_COARE_T / PSI_PAULSON_T (abm::psi_row, abm::psi_poly,
which the psi_*_unstable functions of ab_device.cuh take for zeta in [-50, 0]) against mpmath (50 digits) of the formulas as
the reference writes them: |p - psi| / max(|psi|, 1) <= 4 ulp of 1 everywhere, sampled densely inside every row, at both
ends of every row and a few ulp on either side, at -0, the smallest normals and -50.  The host build checks the polynomials
themselves; the GPU test checks the functions the kernels call at the edges of the table's range (below -50, and for NaN,
the formulas run), against the oracle at the tolerances of tests/test_gpu_functions.py.  The kernels read the COARE table
(COARE 3.0, 3.6 and the first guess of ECMWF) and the Paulson table (ECMWF); NCAR and ANDREAS keep their formulas."""
import ctypes as C
import functools
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ULP = 2.0 ** -52
ZMAX, E0, K = 50.0, -7, 2          # the table's range and rows (tools/gen_math_tables.py)
D = lambda s: mp.mpf(float(s))     # a literal as the reference build rounds it


def coare_conv(phi):
    return 1.5 * mp.log((1 + phi + phi * phi) / 3) - D("1.7320508") * mp.atan((1 + 2 * phi) / D("1.7320508")) + D("1.813799447")


def coare_blend(z, k, c):
    f = z * z / (1 + z * z)
    return (1 - f) * k + f * c


def psi_m_coare(z):      # mod_common_coare.f90:217-254, unstable side
    x = mp.power(1 - 15 * z, 0.25)
    k = 2 * mp.log((1 + x) / 2) + mp.log((1 + x * x) / 2) - 2 * mp.atan(x) + mp.pi / 2
    return coare_blend(z, k, coare_conv(mp.power(1 - D("10.15") * z, D(".3333"))))


def psi_h_coare(z):      # mod_common_coare.f90:305-344
    k = 2 * mp.log((1 + mp.sqrt(1 - 15 * z)) / 2)
    return coare_blend(z, k, coare_conv(mp.power(1 - D("34.15") * z, D(".3333"))))


def psi_m_paulson(z):    # mod_blk_ncar.f90:333-363 (ECMWF and ANDREAS: the same function)
    x = mp.power(1 - 16 * z, 0.25)
    return 2 * mp.log((1 + x) / 2) + mp.log((1 + x * x) / 2) - 2 * mp.atan(x) + mp.pi / 2


def psi_h_paulson(z):    # mod_blk_ncar.f90:379-407
    return 2 * mp.log((1 + mp.sqrt(1 - 16 * z)) / 2)


FUNCS = {("coare", "m"): (0, 0, psi_m_coare), ("coare", "h"): (0, 1, psi_h_coare),
         ("paulson", "m"): (1, 0, psi_m_paulson), ("paulson", "h"): (1, 1, psi_h_paulson)}


@pytest.fixture(scope="module")
def psi_host(tmp_path_factory):
    """abm::psi_row / abm::psi_poly compiled for the host (tests/psi_host_shim.cpp), built in a temporary directory."""
    so = str(tmp_path_factory.mktemp("psi_host") / "psi_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-ffp-contract=off", "-mfma", "-std=c++17", "-shared", "-fPIC",
                           "-o", so, os.path.join(HERE, "psi_host_shim.cpp")])
    L = C.CDLL(so)
    dp = C.POINTER(C.c_double)
    L.psi_table_eval.argtypes = [C.c_int, C.c_int, dp, dp, C.c_long]

    def ev(fam, which, z):
        z = np.ascontiguousarray(z, dtype=np.float64)
        out = np.empty_like(z)
        L.psi_table_eval(fam, which, z.ctypes.data_as(dp), out.ctypes.data_as(dp), z.size)
        return out
    return ev


def _around(x, k=3):
    """x and its k neighbours on either side, one ulp apart."""
    lo, hi = [x], [x]
    for _ in range(k):
        lo.append(np.nextafter(lo[-1], -np.inf))
        hi.append(np.nextafter(hi[-1], np.inf))
    return np.array(lo[:0:-1] + hi)


def row_edges():
    """The lower ends of rows 1, 2, ...: 2^e (1 + j 2^-K) below 50."""
    return [2.0 ** e * (1 + j / 2 ** K) for e in range(E0, 6) for j in range(2 ** K) if 2.0 ** e * (1 + j / 2 ** K) < ZMAX]


@functools.lru_cache(maxsize=None)
def arguments():
    """zeta in [-50, -0]: 33 points inside every row, every row edge +-3 ulp, -0, the smallest normals, -50."""
    edges = row_edges()
    bounds = [0.0] + edges + [ZMAX]
    a = [np.linspace(lo, hi, 33) for lo, hi in zip(bounds[:-1], bounds[1:])]
    a += [_around(e) for e in edges]
    a += [np.array([0.0, 5e-324, 2.2250738585072014e-308, np.nextafter(2.2250738585072014e-308, 1.0), 1e-300, 1e-12]),
          _around(ZMAX)[:4]]
    z = -np.unique(np.concatenate(a))
    z[0] = -0.0 if z[0] == 0.0 else z[0]
    return z


@functools.lru_cache(maxsize=None)
def reference(key):
    mp.mp.dps = 50
    fn = FUNCS[key][2]
    return np.array([float(fn(mp.mpf(float(x)))) if x != 0 else 0.0 for x in arguments()])


@pytest.mark.parametrize("key", sorted(FUNCS))
def test_table_matches_formula_host(psi_host, key):
    fam, which, fn = FUNCS[key]
    z = arguments()
    got = psi_host(fam, which, z)
    mp.mp.dps = 50
    err = np.array([float(abs(mp.mpf(float(g)) - fn(mp.mpf(float(x))))) if x != 0 else abs(g) for g, x in zip(got, z)])
    err /= np.maximum(np.abs(reference(key)), 1.0)
    i = int(err.argmax())
    print(f"[psi table] {key}: worst |p - psi| / max(|psi|, 1) = {err.max() / ULP:.2f} ulp of 1 at zeta = {z[i]!r}")
    assert err.max() <= 4 * ULP, (key, float(z[i]), float(err[i] / ULP))
    assert got[np.where(z == 0)[0]].tolist() == [0.0]                   # psi(-0) = 0 exactly


def test_table_rows_cover_the_range():
    """The rows the generator wrote are the rows this test samples: row 0, then 2^K per binade from 2^E0 to the one holding 50."""
    text = open(os.path.join(HERE, "..", "aerobulk_b200", "csrc", "ab_math_tables.cuh")).read()
    assert f"constexpr int PSI_E0 = {E0}, PSI_K = {K}," in text
    assert int(text.split("PSI_ROWS = ")[1].split(";")[0]) == 1 + len(row_edges())


@pytest.mark.gpu
def test_psi_edges_of_the_table_gpu():
    """The functions the solvers call, at -0, around -50 (table inside, formula below) and for NaN, against the oracle."""
    import aerobulk_b200 as ab
    from oracle import oracle
    OL = oracle.lib()
    z = np.concatenate([[-0.0, -1e-300, -2.2250738585072014e-308], _around(-ZMAX), [-50.5, -75.0, -200.0]])
    for algo, aid, rel in (("ncar", 3, 2e-14), ("coare", 2, 1e-13), ("ecmwf", 4, 5e-14), ("andreas", 5, 1e-13)):
        zz = np.clip(z, -60.0, 10.0) if algo == "ecmwf" else z
        for which in "mh":
            got = ab.probe(f"psi_{which}_{algo}", zz)
            fn = OL.abo_psi_m if which == "m" else OL.abo_psi_h
            ref = np.array([fn(aid, float(x)) for x in zz])
            assert np.all(np.isfinite(got)), (algo, which)
            err = np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)
            assert err.max() <= rel, (algo, which, float(err.max()), float(zz[err.argmax()]))
            assert abs(got[0]) < 1e-12, (algo, which)
    # a NaN with the sign bit set takes the unstable branch and, outside the table, the formula: NaN for COARE (the
    # Paulson formulas' MAX(..., 1) and the ECMWF cap turn NaN into a number, as the reference's MAX / MIN do)
    for which in "mh":
        assert np.isnan(ab.probe(f"psi_{which}_coare", np.array([-np.nan]))).all(), which
