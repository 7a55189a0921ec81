"""Goff's saturation vapour pressure from the piecewise polynomial ESAT_T (abm::esat_table, which abd::e_sat takes on
[230, 330) K) against mpmath (50 digits) of the formula as e_sat writes it: <= 2 ulp everywhere, including at every
interval edge (odd kelvins) and a few ulp on either side, and no step across an edge beyond that.  The host build
checks the polynomial itself, the GPU probe checks e_sat as the kernels run it; outside the table's range e_sat keeps
the formula (checked against the oracle at the tolerance of tests/test_gpu_functions.py)."""
import ctypes as C
import functools
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ULP = 2.0 ** -52
RT0 = "273.15"


@pytest.fixture(scope="module")
def esat_host(tmp_path_factory):
    """abm::esat_table compiled for the host (tests/esat_host_shim.cpp), built in a temporary directory."""
    so = str(tmp_path_factory.mktemp("esat_host") / "esat_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-ffp-contract=off", "-mfma", "-std=c++17", "-shared", "-fPIC",
                           "-o", so, os.path.join(HERE, "esat_host_shim.cpp")])
    L = C.CDLL(so)
    dp = C.POINTER(C.c_double)
    L.esat_table_eval.argtypes = [dp, dp, C.c_long]

    def ev(T):
        T = np.ascontiguousarray(T, dtype=np.float64)
        out = np.empty_like(T)
        L.esat_table_eval(T.ctypes.data_as(dp), out.ctypes.data_as(dp), T.size)
        return out
    return ev


def goff(T):
    mp.mp.dps = 50
    T = mp.mpf(float(T))
    rt0 = mp.mpf(RT0)
    z, r = rt0 / T, T / rt0
    return 100 * mp.power(10, mp.mpf("10.79574") * (1 - z) - mp.mpf("5.028") * mp.log10(r)
                          + mp.mpf("1.50475e-4") * (1 - mp.power(10, mp.mpf("-8.2969") * (r - 1)))
                          + mp.mpf("0.42873e-3") * (mp.power(10, mp.mpf("4.76955") * (1 - z)) - 1)
                          + mp.mpf("0.78614"))


EDGES = np.arange(231.0, 330.0, 2.0)                 # the row boundaries inside [230, 330)


def _around(x, k=4):
    """x and its k neighbours on either side, one ulp apart."""
    lo, hi = [x], [x]
    for _ in range(k):
        lo.append(np.nextafter(lo[-1], -np.inf))
        hi.append(np.nextafter(hi[-1], np.inf))
    return np.array(lo[:0:-1] + hi)


@functools.lru_cache(maxsize=None)
def sweep():
    """Temperatures and the mpmath reference: a dense sweep of [230, 330), each edge +-4 ulp, both ends."""
    T = np.unique(np.concatenate([np.linspace(230.0, 330.0, 5001)[:-1],
                                  np.random.default_rng(20261020).uniform(230.0, 330.0, 2000),
                                  np.concatenate([_around(e) for e in EDGES]), _around(230.0)[4:],
                                  _around(np.nextafter(330.0, 0.0))[:5]]))
    return T, [goff(t) for t in T]


def _ulp_err(got, ref):
    return np.array([float((mp.mpf(float(g)) - r) / r) for g, r in zip(got, ref)]) / ULP


def _check_sweep(got):
    T, ref = sweep()
    err = _ulp_err(got, ref)
    i = int(np.abs(err).argmax())
    assert np.abs(err).max() <= 2.0, (float(T[i]), float(err[i]))
    # across each edge: the two rows' errors differ by <= 2 ulp, and the function still rises with every ulp of T
    # (one ulp of T moves e_sat by 2-3 of its own ulp)
    for e in EDGES:
        idx = np.where(np.abs(T - e) <= 4e-13)[0]
        idx = idx[np.argsort(T[idx])]
        assert np.ptp(err[idx]) <= 2.0, (e, err[idx])
        assert (np.diff(got[idx]) > 0).all(), e


def test_table_matches_goff_host(esat_host):
    T, _ = sweep()
    _check_sweep(esat_host(T))


@pytest.mark.gpu
def test_e_sat_matches_goff_gpu():
    import aerobulk_b200 as ab
    from oracle import oracle

    T, _ = sweep()
    _check_sweep(ab.probe("e_sat", T))
    # outside the table: the formula, as before
    out = np.array([229.99, np.nextafter(230.0, 0.0), 330.0, 335.0, 180.0, 150.0])
    got = ab.probe("e_sat", out)
    ref = np.array([oracle.lib().abo_e_sat(float(t)) for t in out])
    assert (np.abs(got - ref) / np.abs(ref)).max() <= 2e-14
