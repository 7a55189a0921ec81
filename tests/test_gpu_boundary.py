"""Boundary behaviour of the C ABI on the GPU: session semantics of AEROBULK_MODEL
(sticky globals, optional arguments, fail-stop conditions), the two C++-bridge symbols and
size-independent properties at BASELINE's full grid sizes."""
import ctypes as C

import numpy as np
import pytest

from aerobulk_b200 import synth

pytestmark = pytest.mark.gpu
IN_KEYS = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")


@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    return ab


def _ins(f):
    return [f[k] for k in IN_KEYS]


def test_sticky_globals_and_optionals(ab):
    f = synth.fields(64, 32)
    ab.reset()
    assert ab.nb_iter() == 5 and not ab.use_skin() and ab.humidity_type() == "sh"
    o = ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(f))
    assert "T_s" not in o                                  # T_s only with rad_sw & rad_lw
    ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(f), Niter=8)
    assert ab.nb_iter() == 8                                # Niter is sticky (mod_aerobulk.f90:236)
    o8 = ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(f))
    o8b = ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(f), Niter=8)
    assert np.array_equal(o8["QL"], o8b["QL"])
    # radiation given but skin not requested: bulk SST is returned as T_s
    o = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, *_ins(f), rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
    assert np.array_equal(o["T_s"], f["sst"]) and not ab.use_skin()
    o = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, *_ins(f), l_use_skin=True, rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
    assert ab.use_skin() and not np.array_equal(o["T_s"], f["sst"])
    # l_use_skin_schemes is sticky (mod_aerobulk.f90:74): a later call without the flag still uses the skin
    o2 = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, *_ins(f), rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
    assert np.array_equal(o2["T_s"], o["T_s"])
    # ... while ncar ignores it
    o3 = ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(f), rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
    assert np.array_equal(o3["T_s"], f["sst"])


def test_fail_stop_conditions(ab):
    f = synth.fields(32, 16)
    ab.reset()
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model(0, 1, "ncar", 2.0, 10.0, *_ins(f))
    assert e.value.code == 1
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model(1, 1, "bogus", 2.0, 10.0, *_ins(f))
    assert e.value.code == 7
    with pytest.raises(ab.AerobulkError) as e:                # skin only for coare*/ecmwf
        ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(f), l_use_skin=True, rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
    assert e.value.code == 2
    ab.reset()
    with pytest.raises(ab.AerobulkError) as e:                # skin needs radiation
        ab.aerobulk_model(1, 1, "ecmwf", 2.0, 10.0, *_ins(f), l_use_skin=True)
    assert e.value.code == 3
    ab.reset()
    g = dict(f)
    g["sst"] = f["sst"] - 273.15                              # deg C instead of K: everything masked
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(g))
    assert e.value.code == 4
    g = dict(f)
    g["slp"] = f["slp"].copy()
    g["slp"][3, 3] = 1013.0                                   # one point in hPa: masked, not fatal
    ab.reset()
    ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(g))
    g = dict(f)
    g["hum_zt"] = f["hum_zt"] * 1000.0 + 110.0                # neither sh, rh nor dp
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, *_ins(g))
    assert e.value.code == 5
    g = dict(f)
    g["U_zu"] = f["U_zu"] * 0.0 + 48.0                         # |U| <= 50 passes the mask, tau > 10 N/m2 stops
    g["V_zu"] = f["V_zu"] * 0.0
    ab.reset()
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, *_ins(g))
    assert e.value.code == 8 and "wind stress too strong" in e.value.message
    # double jt==1 of a skin session before jt==Nt: the reference's ALLOCATE fails
    ab.reset()
    kw = dict(l_use_skin=True, rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
    ab.aerobulk_model(1, 3, "coare3p0", 2.0, 10.0, *_ins(f), **kw)
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model(1, 3, "coare3p6", 2.0, 10.0, *_ins(f), **kw)   # 3.0 and 3.6 share mod_skin_coare's arrays
    assert e.value.code == 9
    ab.reset()


def test_public_aerobulk_init(ab):
    """AEROBULK_INIT called directly (it is PUBLIC in the reference, src/mod_aerobulk.f90:20): same decisions and
    fail-stops as the initialisation AEROBULK_MODEL runs at jt == 1."""
    f = synth.fields(64, 32, humidity="dp")
    ab.reset()
    ab.aerobulk_init(2, "ecmwf", *_ins(f), l_use_skin=True, prsw=f["rad_sw"], prlw=f["rad_lw"])
    assert ab.use_skin() and ab.humidity_type() == "dp"
    for jt in (1, 2):     # AEROBULK_MODEL(jt == 1) initialises again on its own arguments, as in the reference
        o = ab.aerobulk_model(jt, 2, "ecmwf", 2.0, 10.0, *_ins(f), l_use_skin=True, rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
        assert "T_s" in o and np.isfinite(o["T_s"]).all()
    assert ab.get_state(0, 64 * 32) is None                 # the session ended at jt == nitend
    ab.reset()
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_init(1, "ncar", *_ins(f), l_use_skin=True, prsw=f["rad_sw"], prlw=f["rad_lw"])
    assert e.value.code == 2                                # skin asked for an algorithm without skin schemes
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_init(1, "coare3p6", *_ins(f), l_use_skin=True)
    assert e.value.code == 3 and not ab.use_skin()          # no radiation given; the flag was rolled back
    g = dict(f)
    g["slp"] = f["slp"] / 100.0                             # hPa: every point masked
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_init(1, "coare3p6", *_ins(g))
    assert e.value.code == 4
    ab.aerobulk_bye()


def test_empty_and_tiny_inputs(ab):
    ab.reset()
    z = np.zeros((0,), dtype=np.float64)
    with pytest.raises(ab.AerobulkError):      # the reference divides by SUM(mask)=0 -> "whole domain is masked"
        ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, z, z, z, z, z, z)
    f = synth.fields(1, 1)
    ab.reset()
    o = ab.aerobulk_model(1, 1, "andreas", 2.0, 10.0, *_ins(f))
    assert o["QL"].shape == (1, 1) and np.isfinite(o["QL"]).all()
    f = synth.fields(129, 7)                   # ragged: not a multiple of the block size
    ab.reset()
    o = ab.aerobulk_model(1, 1, "ecmwf", 2.0, 10.0, *_ins(f))
    assert np.isfinite(o["QH"]).all()


def test_c_ordered_2d_inputs_give_the_same_fields(ab):
    """ADVICE r1: numpy's default C-ordered 2-D arrays, mixed with Fortran-ordered ones, give index-for-index the same
    result as all-Fortran inputs (the mirror normalises the layout; outputs come back (Ni,Nj) column-major)."""
    Ni, Nj = 37, 23
    f = synth.fields(Ni, Nj)
    kw = dict(Niter=5, l_use_skin=True)
    ab.reset()
    want = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, *_ins(f), rad_sw=f["rad_sw"], rad_lw=f["rad_lw"], **kw)
    c = {k: np.ascontiguousarray(v) for k, v in f.items()}
    assert c["sst"].flags.c_contiguous and not c["sst"].flags.f_contiguous
    ab.reset()
    got = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, c["sst"], f["t_zt"], c["hum_zt"], c["U_zu"], f["V_zu"], c["slp"],
                            rad_sw=c["rad_sw"], rad_lw=f["rad_lw"], **kw)
    for k in want:
        assert got[k].shape == (Ni, Nj) and np.array_equal(got[k], want[k]), k
    # the TURB_* mirror too
    ab.reset()
    qs = np.full((Ni, Nj), 0.015)
    a = ab.turb("ncar", 1, 2.0, 10.0, f["sst"], f["t_zt"], qs, f["hum_zt"], np.hypot(f["U_zu"], f["V_zu"]))
    b = ab.turb("ncar", 1, 2.0, 10.0, c["sst"], c["t_zt"], np.ascontiguousarray(qs), c["hum_zt"],
                np.ascontiguousarray(np.hypot(f["U_zu"], f["V_zu"])))
    for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu"):
        assert np.array_equal(a[k], b[k]), k


def test_calm_points_have_zero_stress(ab):
    f = synth.fields(512, 256)
    calm = (f["U_zu"] == 0) & (f["V_zu"] == 0)
    assert calm.sum() > 0
    ab.reset()
    o = ab.aerobulk_model(1, 1, "coare3p0", 2.0, 10.0, *_ins(f))
    assert (o["Tau_x"][calm] == 0).all() and (o["Tau_y"][calm] == 0).all()   # zWzu <= 1e-3, mod_aerobulk_compute.f90:191
    assert np.isfinite(o["QL"][calm]).all()


def test_cxx_bridge_symbols(ab):
    """aerobulk_cxx_skin / aerobulk_cxx_no_skin exactly as src/aerobulk.cpp:105-108,135-137 calls them."""
    L = ab.lib()
    ab.reset()
    m = 2
    rt0 = 273.15
    arr = lambda *v: np.array(v, dtype=np.float64)
    sst, t, q, U, V, slp = arr(22 + rt0, 22 + rt0), arr(20 + rt0, 25 + rt0), arr(.012, .012), arr(4., 4.), arr(9., 9.), arr(101000., 101000.)
    rsw, rlw = arr(0., 0.), arr(350., 350.)
    outs = [np.zeros(m) for _ in range(6)]
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ci = lambda v: C.byref(C.c_int(v))
    cd = lambda v: C.byref(C.c_double(v))
    algo = b"coare3p6"
    L.aerobulk_cxx_skin(ci(1), ci(1), algo, cd(2.0), cd(10.0), p(sst), p(t), p(q), p(U), p(V), p(slp),
                        *[p(o) for o in outs[:5]], ci(8), C.byref(C.c_bool(True)), p(rsw), p(rlw), p(outs[5]),
                        ci(len(algo)), ci(m))
    ref = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, sst, t, q, U, V, slp, Niter=8, l_use_skin=True, rad_sw=rsw, rad_lw=rlw)
    for o, k in zip(outs, ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")):
        assert np.array_equal(o, ref[k]), k
    assert outs[5][0] < 22 + rt0          # cool skin at night
    algo = b"ncar"
    outs2 = [np.zeros(m) for _ in range(5)]
    L.aerobulk_cxx_no_skin(ci(1), ci(1), algo, cd(2.0), cd(10.0), p(sst), p(t), p(q), p(U), p(V), p(slp),
                           *[p(o) for o in outs2], ci(8), ci(len(algo)), ci(m))
    ref = ab.aerobulk_model(1, 1, "ncar", 2.0, 10.0, sst, t, q, U, V, slp, Niter=8)
    for o, k in zip(outs2, ("QL", "QH", "Tau_x", "Tau_y", "Evap")):
        assert np.array_equal(o, ref[k]), k


@pytest.mark.parametrize("algo,skin", [("ecmwf", True), ("andreas", False), ("coare3p0", False)])
def test_full_size_properties_4320x2160(ab, algo, skin):
    """BASELINE configs 3/4 at full size (9.3 M points): size-independent properties instead of the oracle.
    (a) a strided sample of the big grid equals the same points computed alone (independence of points,
    chunking/pipelining does not leak between points); (b) outputs finite; (c) rotating the wind by 90 deg
    rotates the stress and leaves the scalar fluxes bit-identical."""
    Ni, Nj = 4320, 2160
    f = synth.fields(Ni, Nj)
    kw = dict(l_use_skin=True, rad_sw=f["rad_sw"], rad_lw=f["rad_lw"]) if skin else {}
    ab.reset()
    big = ab.aerobulk_model(1, 1, algo, 2.0, 10.0, *_ins(f), **kw)
    for k, v in big.items():
        assert np.isfinite(v).all(), k
    sl = (slice(7, None, 97), slice(3, None, 89))
    sub = {k: np.asfortranarray(v[sl]) for k, v in f.items()}
    kws = dict(l_use_skin=True, rad_sw=sub["rad_sw"], rad_lw=sub["rad_lw"]) if skin else {}
    ab.reset()
    small = ab.aerobulk_model(1, 1, algo, 2.0, 10.0, *_ins(sub), **kws)
    for k in small:
        assert np.array_equal(small[k], big[k][sl]), k
    rot = dict(f)
    rot["U_zu"], rot["V_zu"] = np.asfortranarray(-f["V_zu"]), f["U_zu"]
    ab.reset()
    r = ab.aerobulk_model(1, 1, algo, 2.0, 10.0, *_ins(rot), **kw)
    assert np.array_equal(r["QL"], big["QL"]) and np.array_equal(r["QH"], big["QH"]) and np.array_equal(r["Evap"], big["Evap"])
    assert np.array_equal(r["Tau_x"], -big["Tau_y"]) and np.array_equal(r["Tau_y"], big["Tau_x"])


def test_cpp_example_matches_oracle(ab, tmp_path):
    """tests/cpp/example_call_aerobulk.cpp (the reference's C++ example, same inputs: U=(4,9), 8 iterations)
    built against include/aerobulk.hpp + libaerobulk_gpu.so, compared with the CPU oracle."""
    import os, subprocess
    from aerobulk_b200.model import _SO
    from oracle.oracle import OracleSession
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "example_call_aerobulk_cxx.x")
    subprocess.check_call(["/usr/bin/g++", "-std=c++11", "-O1", "-I", os.path.join(root, "include"),
                           os.path.join(root, "tests", "cpp", "example_call_aerobulk.cpp"), "-o", exe,
                           "-L", os.path.dirname(_SO), "-laerobulk_gpu", "-Wl,-rpath," + os.path.dirname(_SO)])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = {l.split()[1]: np.array(l.split()[2:], dtype=float) for l in r.stdout.splitlines() if l.startswith("RESULT")}
    assert set(rows) == {"coare3p0", "coare3p6", "ecmwf", "ncar", "andreas"}
    rt0 = 273.15
    arr = lambda *v: np.array(v, dtype=np.float64)
    ins = [arr(22 + rt0, 22 + rt0), arr(20 + rt0, 25 + rt0), arr(.012, .012), arr(4., 4.), arr(9., 9.), arr(101000., 101000.)]
    for algo, got in rows.items():
        kw = dict(Niter=8)
        if algo in ("coare3p0", "coare3p6", "ecmwf"):
            kw.update(l_use_skin=True, rad_sw=arr(0., 0.), rad_lw=arr(350., 350.))
        ref = OracleSession().model(1, 1, algo, 2.0, 10.0, *ins, **kw)
        want = np.concatenate([ref["QH"], ref["QL"], ref["Evap"], ref["Tau_x"], ref["Tau_y"], ref.get("T_s", ins[0])])
        scale = np.repeat([10.0, 10.0, 1e-5, 1e-2, 1e-2, 1.0], 2)
        assert (np.abs(got - want) / (np.abs(want) + scale)).max() <= 1e-10, algo


def test_sharded_init_on_device(ab):
    """aerobulk_gpu_init_local_stats on two row blocks + init_from_stats == one-shot AEROBULK_INIT."""
    import torch
    from aerobulk_b200 import model as abm
    Ni, Nj = 96, 64
    keys = IN_KEYS
    full = synth.fields(Ni, Nj, humidity="rh")
    ops = abm.stats_reduce_ops()
    parts = []
    for j0, j1 in ((0, 20), (20, 64)):
        b = synth.fields(Ni, Nj, j0=j0, j1=j1, humidity="rh")
        dev = {k: torch.from_numpy(np.ravel(v, order="F").copy()).cuda() for k, v in b.items()}
        parts.append(abm.init_local_stats(*[dev[k] for k in keys], rad_lw=dev["rad_lw"]))
    g = np.where(ops == 0, parts[0] + parts[1], np.where(ops == 1, np.minimum(parts[0], parts[1]), np.maximum(parts[0], parts[1])))
    dev = {k: torch.from_numpy(np.ravel(v, order="F").copy()).cuda() for k, v in full.items()}
    one = abm.init_local_stats(*[dev[k] for k in keys], rad_lw=dev["rad_lw"])
    assert g[0] == one[0] == Ni * Nj and g[1] == one[1]
    for k in range(9):
        bse = 2 + 5 * k
        assert g[bse] == pytest.approx(one[bse], rel=1e-13)
        assert np.array_equal(g[bse + 1:bse + 5], one[bse + 1:bse + 5])
        assert one[bse + 3] == np.ravel([full["sst"], full["t_zt"], full["slp"], full["U_zu"], full["V_zu"],
                                         np.hypot(full["U_zu"], full["V_zu"]), full["hum_zt"], full["rad_lw"], full["rad_lw"]][k]).min() \
            or k == 5
    ab.reset()
    abm.init_from_stats(2, "ecmwf", True, True, g)
    assert ab.humidity_type() == "rh" and ab.use_skin()
    # the following jt==1 call skips its local AEROBULK_INIT and computes with the global decisions
    b = synth.fields(Ni, Nj, j0=0, j1=20, humidity="rh")
    o = ab.aerobulk_model(1, 2, "ecmwf", 2.0, 10.0, *[b[k] for k in keys], l_use_skin=True, rad_sw=b["rad_sw"], rad_lw=b["rad_lw"])
    ab.reset()
    ref = ab.aerobulk_model(1, 2, "ecmwf", 2.0, 10.0, *[full[k] for k in keys], l_use_skin=True, rad_sw=full["rad_sw"], rad_lw=full["rad_lw"])
    for k in o:
        assert np.array_equal(o[k], ref[k][:, 0:20]), k
    ab.reset()


@pytest.mark.parametrize("rad", [True, False])
def test_stats_vector_with_masked_points_matches_numpy(ab, rad):
    """The AEROBULK_INIT statistics pass (stats_fast_kernel + stats_fix_kernel + stats_final): blocks without a masked
    point take the 27-accumulator fast path, blocks with one are redone with the full set -- the 64-double vector must be
    what numpy computes from the mask of src/mod_aerobulk.f90:104-124 (counts and extrema exactly, sums to rounding),
    whichever blocks the masked points fall in."""
    import torch
    from aerobulk_b200 import model as abm
    Ni, Nj = 700, 301                                   # 210 700 points: 824 blocks, the last one ragged
    f = synth.fields(Ni, Nj)
    rng = np.random.default_rng(5)
    flat = {k: np.ravel(v, order="F").copy() for k, v in f.items()}
    n = Ni * Nj
    hit = rng.choice(n, size=12, replace=False)
    flat["sst"][hit[0:3]] -= 273.15                     # deg C
    flat["t_zt"][hit[3]] = 400.0
    flat["slp"][hit[4:6]] /= 100.0                      # hPa
    flat["U_zu"][hit[6]], flat["V_zu"][hit[6]] = 40.0, 40.0   # |U| = 56.6 > 50
    flat["rad_lw"][hit[7]] = 900.0                      # inside the long-wave range, outside the short-wave one (prsw=rad_lw)
    flat["rad_lw"][hit[8]] = -1.0
    flat["sst"][n - 1] = 100.0                          # the ragged last block
    dev = {k: torch.from_numpy(v).cuda() for k, v in flat.items()}
    got = abm.init_local_stats(*[dev[k] for k in IN_KEYS], rad_lw=dev["rad_lw"] if rad else None)
    wnd = np.sqrt(flat["U_zu"] * flat["U_zu"] + flat["V_zu"] * flat["V_zu"])
    lw = flat["rad_lw"] if rad else np.zeros(n)
    m = (flat["sst"] >= 270.) & (flat["sst"] <= 320.) & (flat["t_zt"] >= 180.) & (flat["t_zt"] <= 330.) \
        & (flat["slp"] >= 80000.) & (flat["slp"] <= 110000.) & (wnd <= 50.)
    if rad:
        m &= (lw >= 0.) & (lw <= 750.)
    assert got[0] == m.sum() and got[1] == n and m.sum() == n - (10 if rad else 8)
    fields = [flat["sst"], flat["t_zt"], flat["slp"], flat["U_zu"], flat["V_zu"], wnd, flat["hum_zt"], lw, lw]
    for k, v in enumerate(fields):
        b = 2 + 5 * k
        assert got[b] == pytest.approx(v[m].sum(), rel=1e-12, abs=1e-9), k
        assert got[b + 1] == v[m].min() and got[b + 2] == v[m].max(), k
        assert got[b + 3] == v.min() and got[b + 4] == v.max(), k
    # no masked point at all: the same numbers from the fast path alone
    clean = {k: torch.from_numpy(np.ravel(v, order="F").copy()).cuda() for k, v in f.items()}
    got = abm.init_local_stats(*[clean[k] for k in IN_KEYS], rad_lw=clean["rad_lw"] if rad else None)
    assert got[0] == n and got[1] == n
    for k, key in enumerate(("sst", "t_zt", "slp", "U_zu", "V_zu")):
        v = np.ravel(f[key], order="F")
        b = 2 + 5 * k
        assert got[b] == pytest.approx(v.sum(), rel=1e-12)
        assert got[b + 1] == got[b + 3] == v.min() and got[b + 2] == got[b + 4] == v.max()
    ab.reset()


def test_flux_kernels_keep_their_occupancy(ab):
    """The launch configuration DESIGN.md 3.1 measured: kernels without skin 4 blocks of 256 threads per SM (<= 64
    registers), skin kernels 3 (<= 85 registers) -- a change that silently costs a resident block fails here."""
    for algo in ("ncar", "andreas", "coare3p0", "coare3p6", "ecmwf"):
        for zteq in (False, True):
            k = ab.kernel_info(algo, False, zteq)
            assert k["registers"] <= 64 and k["blocks_per_sm"] == 4, (algo, zteq, k)
    for algo in ("coare3p0", "coare3p6", "ecmwf"):
        for zteq in (False, True):
            k = ab.kernel_info(algo, True, zteq)
            assert k["registers"] <= 85 and k["blocks_per_sm"] == 3, (algo, zteq, k)
            assert k["local_bytes"] <= 160, (algo, zteq, k)          # a few spilled doubles outside the loop, no more
    assert ab.kernel_info("ncar", True) == ab.kernel_info("ncar", False)    # no skin variant of NCAR
    with pytest.raises(ab.AerobulkError):
        ab.kernel_info("lg15")


def test_deferred_wind_stress_error_on_device_api(ab):
    """Device-resident calls are asynchronous for jt>1: tau > 10 N/m2 surfaces at synchronize()."""
    import torch
    Ni, Nj = 64, 16
    f = synth.fields(Ni, Nj)
    dev = {k: torch.from_numpy(np.ravel(v, order="F").copy()).cuda() for k, v in f.items()}
    out = {k: torch.empty(Ni * Nj, dtype=torch.float64, device="cuda") for k in ("QL", "QH", "Tau_x", "Tau_y", "Evap")}
    ab.reset()
    ins = [dev[k] for k in IN_KEYS]
    ab.aerobulk_model_device(1, 3, "coare3p6", 2.0, 10.0, *ins, out=out, shape=(Ni, Nj))
    storm = dev["U_zu"] * 0 + 48.0
    ins2 = [dev["sst"], dev["t_zt"], dev["hum_zt"], storm, dev["V_zu"] * 0, dev["slp"]]
    ab.aerobulk_model_device(2, 3, "coare3p6", 2.0, 10.0, *ins2, out=out, shape=(Ni, Nj))
    with pytest.raises(ab.AerobulkError) as e:
        ab.synchronize()
    assert e.value.code == 8
    ab.reset()


def test_fields_in_one_slab_use_pitched_copies_and_agree(ab):
    """A caller that keeps its fields equally spaced in one slab gets one pitched copy per pipeline chunk
    (Transport::copy in ab_api.cu); results are bit-identical to separate arrays -- pageable and pinned slabs."""
    import torch
    Ni, Nj = 640, 400                      # 256 000 points: 1 chunk; plus a 3-chunk case below
    for (ni, nj) in ((Ni, Nj), (1440, 500)):
        n = ni * nj
        f = synth.fields(ni, nj)
        keys = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp", "rad_lw")
        ab.reset()
        ref = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, *[f[k] for k in keys[:6]], Niter=5, l_use_skin=True,
                                rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
        for pinned in (False, True):
            slab = torch.empty((7, n), dtype=torch.float64)
            oslab = torch.empty((6, n), dtype=torch.float64)
            if pinned:
                slab, oslab = slab.pin_memory(), oslab.pin_memory()
            view = {}
            for i, k in enumerate(keys):
                slab[i].numpy()[:] = np.ravel(f[k], order="F")
                view[k] = slab[i].numpy().reshape((ni, nj), order="F")
            names = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")
            out = {k: oslab[i].numpy().reshape((ni, nj), order="F") for i, k in enumerate(names)}
            ab.reset()
            got = ab.aerobulk_model(1, 1, "coare3p6", 2.0, 10.0, *[view[k] for k in keys[:6]], Niter=5, l_use_skin=True,
                                    rad_sw=f["rad_sw"], rad_lw=view["rad_lw"], out=out)
            for k in names:
                assert np.array_equal(got[k], ref[k]), (ni, pinned, k)
                assert np.array_equal(out[k], ref[k]), (ni, pinned, k)


def test_flux_diagnostics_match_numpy_and_combine_like_one_domain(ab):
    """aerobulk_gpu_flux_diagnostics: device sums / minima / maxima of the flux fields; two row blocks combined with
    aerobulk_gpu_diag_reduce_op equal the whole domain (min / max exactly, sums to rounding)."""
    Ni, Nj = 300, 200
    f = synth.fields(Ni, Nj)
    keys = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
    ab.reset()
    r = ab.aerobulk_model(1, 1, "ecmwf", 2.0, 10.0, *[f[k] for k in keys], Niter=4, l_use_skin=True,
                          rad_sw=f["rad_sw"], rad_lw=f["rad_lw"])
    st = ab.flux_diagnostics(r)
    ops = ab.diag_reduce_ops()
    assert st[0] == Ni * Nj and list(ops[:4]) == [0, 0, 1, 2]
    for i, k in enumerate(("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")):
        assert st[1 + 3 * i] == pytest.approx(r[k].sum(), rel=1e-12)
        assert st[2 + 3 * i] == r[k].min() and st[3 + 3 * i] == r[k].max()
    assert np.array_equal(ab.flux_diagnostics(r), st)                     # deterministic
    half = Nj // 2
    a = ab.flux_diagnostics({k: v[:, :half] for k, v in r.items()})
    b = ab.flux_diagnostics({k: v[:, half:] for k, v in r.items()})
    comb = np.where(ops == 0, a + b, np.where(ops == 1, np.minimum(a, b), np.maximum(a, b)))
    assert np.allclose(comb, st, rtol=1e-12, atol=0) and np.array_equal(comb[ops != 0], st[ops != 0])
    s = ab.diagnostics_summary(comb)
    assert s["n"] == Ni * Nj and s["QH"]["min"] == r["QH"].min() and abs(s["T_s"]["mean"] - r["T_s"].mean()) < 1e-9
    # a subset of the fields, on the device
    import torch
    t = {"QL": torch.from_numpy(np.ravel(r["QL"], order="F").copy()).cuda()}
    d = ab.flux_diagnostics(t)
    assert d[1] == pytest.approx(r["QL"].sum(), rel=1e-12) and d[4] == 0.0 and d[5] > 1e300 and d[6] < -1e300
    assert "QH" not in ab.diagnostics_summary(d)


def test_pinned_arrays_take_the_zero_copy_path_and_agree(ab):
    """When every array of a host-array call is pinned, the kernel reads / writes the caller's arrays directly (zero-copy,
    no stability sort); pageable arrays go through the library's pinned slab (copy threads).  Bit-identical over a state-carrying session."""
    import torch
    Ni, Nj, Nt = 512, 300, 4
    n = Ni * Nj
    f = synth.fields(Ni, Nj)
    keys = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp", "rad_lw", "rad_sw")
    names = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")

    def run(pinned):
        src, out = {}, {}
        hold = []
        for k in keys:
            t = torch.empty(n, dtype=torch.float64)
            t = t.pin_memory() if pinned else t
            t.numpy()[:] = np.ravel(f[k], order="F")
            hold.append(t)
            src[k] = t.numpy().reshape((Ni, Nj), order="F")
        for k in names:
            t = torch.zeros(n, dtype=torch.float64)
            t = t.pin_memory() if pinned else t
            hold.append(t)
            out[k] = t.numpy().reshape((Ni, Nj), order="F")
        ab.reset()
        res, launches = [], []
        for jt in range(1, Nt + 1):
            ab.lib().aerobulk_gpu_reset_launch_count()
            ab.aerobulk_model(jt, Nt, "coare3p6", 2.0, 10.0, *[src[k] for k in keys[:6]], Niter=5, l_use_skin=True,
                              rad_sw=src["rad_sw"], rad_lw=src["rad_lw"], out=out)
            res.append({k: out[k].copy() for k in names})
            launches.append(ab.launch_count())
        return res, launches

    a, la = run(False)
    b, lb = run(True)
    for jt in range(Nt):
        for k in names:
            assert np.array_equal(a[jt][k], b[jt][k]), (jt, k)
    # jt == 1 is staged either way (AEROBULK_INIT needs the statistics): three statistics kernels (fast pass, fix-up of
    # the blocks with masked points, final reduction), classify, flux.
    # Afterwards no classify: pinned arrays are used in place (ONE flux launch), pageable ones of this size go through
    # the library's pinned slab in row-block chunks (one flux launch per chunk; one chunk here)
    assert la[1:] == [1] * (Nt - 1) and lb[1:] == [1] * (Nt - 1) and la[0] == lb[0] == 5
    ab.reset()


@pytest.mark.parametrize("ni,nj", [(96, 50), (512, 300), (1031, 257)])
def test_host_register_gives_plain_arrays_the_pinned_path(ab, ni, nj):
    """aerobulk_gpu_host_register on ordinary numpy arrays: same results as the pageable path (driver-staged copies for
    the small grid, the library's copy threads + pinned slab for the larger ones), and the arrays can be released and
    used again."""
    f = synth.fields(ni, nj, seed=77)
    names = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp", "rad_sw", "rad_lw")
    arrs = {k: np.array(f[k], order="F") for k in names}
    outs = {k: np.zeros((ni, nj), order="F") for k in ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")}

    def session():
        ab.reset()
        for jt in (1, 2, 3):
            ab.aerobulk_model(jt, 3, "ecmwf", 2., 10., *[arrs[k] for k in names[:6]], Niter=6, l_use_skin=True,
                              rad_sw=arrs["rad_sw"], rad_lw=arrs["rad_lw"], out=outs)
        return {k: v.copy() for k, v in outs.items()}

    plain = session()
    for v in list(arrs.values()) + list(outs.values()):
        ab.host_register(v)
    try:
        pinned = session()
    finally:
        for v in list(arrs.values()) + list(outs.values()):
            ab.host_unregister(v)
    again = session()
    for k in plain:
        assert np.array_equal(plain[k], pinned[k]), k
        assert np.array_equal(plain[k], again[k]), k
    with pytest.raises(ab.AerobulkError):
        ab.host_unregister(arrs["sst"])  # not registered any more
