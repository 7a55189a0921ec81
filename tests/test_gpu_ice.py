"""SURVEY.md 8f row 4: sea-ice bulk algorithms (aerobulk_gpu_turb_ice) and the ice + leads computation
(aerobulk_gpu_oce_ice) against the oracle's restatement of src/ice/mod_blk_ice_*.f90."""
import numpy as np
import pytest

import parity_util as pu
from aerobulk_b200 import synth

pytestmark = pytest.mark.gpu
TOL = 1e-10   # scaled metric of tests/test_gpu_parity.py: |gpu-ref| / (|ref| + S_f)
OPT = ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10", "CdN_frm")
SCALE = pu.ICE_SCALE


@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    return ab


def _prove(tag, worst_pt, inputs, run_oracle, scale):
    """Every point above TOL must sit where the oracle itself moves under ulp-level input nudges, or where such a nudge
    trips the reference's rough_leng_tq fail-stop (parity_util.prove_flips)."""
    bad = np.flatnonzero(worst_pt > TOL)
    print(f"[parity] {tag}: n={worst_pt.size} max {worst_pt.max():.3e} points>1e-10: {bad.size}")
    if bad.size:
        proven = pu.prove_flips(bad, worst_pt[bad], inputs, run_oracle, tag, scale=scale, failstop=10)
        assert proven.all(), (tag, "points above 1e-10 where the oracle is NOT sensitive to ulp-level input nudges",
                              bad[~proven].tolist(), worst_pt[bad][~proven].tolist())


def _compare(tag, got, ref, keys, flux_of, inputs, run_oracle):
    """At most 2e-5 of the points above TOL (near-calm / vanishing-difference points amplify rounding noise), and each
    of them proven by _prove.  Ch and Ce are 0/0 at a vanishing air-surface difference: only compared where |dtheta|,
    |dq| is sizeable."""
    worst = 0.0
    worst_pt = np.zeros(np.size(got[keys[0]]))
    for k in keys:
        g, r = np.ravel(got[k]), np.ravel(ref[k])
        base = k[:-2] if k.endswith(("_i", "_w")) else k
        if base in ("xL", "L"):
            g, r = 1.0 / g, 1.0 / r
        e = np.abs(g - r) / (np.abs(r) + SCALE[base])
        if flux_of is not None and base in ("Ch", "Ce"):
            e = np.where(flux_of[base + k[len(base):]], e, 0.0)
        assert np.all(np.isfinite(g)), (tag, k)
        bad = int((e > TOL).sum())
        assert bad <= max(1, int(2e-5 * e.size)), (tag, k, bad, float(e.max()))
        worst = max(worst, float(np.sort(e)[-2]))
        worst_pt = np.maximum(worst_pt, e)
    _prove(tag, worst_pt, inputs, run_oracle, pu.ice_scale(keys))
    return worst


def _both(gpu_call, ref_call, f, AbErr, OrErr):
    """Runs the GPU and the oracle on the fields `f`.  AN05's rough_leng_tq stops for a roughness Reynolds number in
    ]2.49999, 2.5[ (about one evaluation in 5e5 lands there): a point that trips it on either side is replaced by its
    neighbour and the pair is run again."""
    import re
    for _ in range(6):
        try:
            return gpu_call(f), ref_call(f), f
        except (AbErr, OrErr) as e:
            if e.code != 10:
                raise
            i = int(re.search(r"point (\d+)", str(e)).group(1)) - 1
            f = {k: v.copy() for k, v in f.items()}
            for v in f.values():
                v[i] = v[i - 1 if i > 0 else 1]
    raise AssertionError("rough_leng_tq fail-stop keeps firing")


def _turb_inputs(n, zt):
    from oracle import oracle
    f = synth.ice_fields(n)
    L = oracle.lib()
    siq = np.array([L.abo_q_sat_ice(t, p) for t, p in zip(f["sit"], f["slp"])])
    tha = f["t_zt"] + 0.0098 * zt
    return f, siq, tha


@pytest.mark.parametrize("algo", ["nemo", "easy", "an05", "lu12", "lg15", "lg15_io"])
@pytest.mark.parametrize("zt,nb_iter", [(2.0, 5), (10.0, 20)])
def test_turb_ice_matches_oracle(ab, algo, zt, nb_iter):
    from oracle.oracle import OracleSession
    n = 40000
    f, siq, tha = _turb_inputs(n, zt)
    cxn = [1.4e-3, 1.3e-3, 1.2e-3] if algo == "easy" else None
    ab.reset()
    ab.set_nb_iter(nb_iter)
    o = OracleSession(threads=8)
    o.set_nb_iter(nb_iter)
    from oracle.oracle import OracleError
    f = dict(f, siq=siq, tha=tha)
    got, ref, f = _both(lambda d: ab.turb_ice(algo, zt, 10.0, d["sit"], d["tha"], d["siq"], d["hum_zt"], d["wind"], frice=d["frice"], cxn=cxn, want=OPT),
                        lambda d: o.turb_ice(algo, zt, 10.0, d["sit"], d["tha"], d["siq"], d["hum_zt"], d["wind"], frice=d["frice"], cxn=cxn, want=OPT),
                        f, ab.AerobulkError, OracleError)
    siq = f["siq"]
    dth, dq = np.abs(ref["t_zu"] - f["sit"]) > 0.05, np.abs(ref["q_zu"] - siq) > 2e-5
    inputs = dict(Ts_i=f["sit"], t_zt=f["tha"], qs_i=siq, q_zt=f["hum_zt"], U_zu=f["wind"], frice=f["frice"])
    last = {k: v[-1] for k, v in inputs.items()} if algo.startswith("lg15") else None
    worst = _compare(f"turb_ice {algo}", got, ref, ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu") + OPT, {"Ch": dth, "Ce": dq},
                     inputs, pu.turb_ice_runner(OracleSession, algo, zt, 10.0, nb_iter, cxn, last))
    assert worst <= TOL
    if algo.startswith("lg15"):   # reference behaviour: one form drag for all, from the last point
        assert np.all(got["CdN_frm"] == got["CdN_frm"][0])


def test_lg15_per_point_form_drag(ab):
    from oracle.oracle import OracleSession
    n = 20000
    f, siq, tha = _turb_inputs(n, 2.0)
    ab.reset()
    ab.set_ice_form_drag_per_point(True)
    got = ab.turb_ice("lg15", 2.0, 10.0, f["sit"], tha, siq, f["hum_zt"], f["wind"], frice=f["frice"], want=OPT)
    ab.set_ice_form_drag_per_point(False)
    o = OracleSession(threads=8)
    ref = o.turb_ice("lg15", 2.0, 10.0, f["sit"], tha, siq, f["hum_zt"], f["wind"], frice=f["frice"], per_point_form_drag=True, want=OPT)
    dth, dq = np.abs(ref["t_zu"] - f["sit"]) > 0.05, np.abs(ref["q_zu"] - siq) > 2e-5
    inputs = dict(Ts_i=f["sit"], t_zt=tha, qs_i=siq, q_zt=f["hum_zt"], U_zu=f["wind"], frice=f["frice"])
    assert _compare("lg15 per point", got, ref, ("Cd", "Ch", "Ce", "t_zu", "q_zu") + OPT, {"Ch": dth, "Ce": dq}, inputs,
                    pu.turb_ice_runner(OracleSession, "lg15", 2.0, 10.0, o.nb_iter, per_point_form_drag=True)) <= TOL
    assert len(np.unique(got["CdN_frm"])) > 100


@pytest.mark.parametrize("ice,oce,hum", [("an05", "ecmwf", "q"), ("lg15_io", "ecmwf", "rh"), ("nemo", "ncar", "dp"),
                                         ("lu12", "coare3p6", "q"), ("easy", "andreas", "rh"), ("lg15", "coare3p0", "q"),
                                         ("an05", None, "q")])
def test_oce_ice_matches_oracle(ab, ice, oce, hum):
    from oracle.oracle import OracleSession
    n = 30000
    f = synth.ice_fields(n, humidity=hum)
    cxn = [1.4e-3, 1.3e-3, 1.2e-3] if ice == "easy" else None
    ab.reset()
    ab.set_nb_iter(20)                 # the programs use 20 (src/ice/test_aerobulk_oce+ice.f90:67)
    o = OracleSession(threads=8)
    o.set_nb_iter(20)
    from oracle.oracle import OracleError
    got, ref, f = _both(lambda d: ab.oce_ice(ice, oce, 2.0, 10.0, **d, hum_kind=hum, cxn=cxn),
                        lambda d: o.oce_ice(ice, oce, 2.0, 10.0, d["sit"], d["sst"], d["t_zt"], d["hum_zt"], d["wind"], d["slp"],
                                            d["frice"], hum_kind={"q": 0, "dp": 1, "rh": 2}[hum], cxn=cxn),
                        f, ab.AerobulkError, OracleError)
    keys = [k for k in ab.OCE_ICE_OUT if oce is not None or k.endswith("_i")]
    sizeable = {"Ch_i": np.abs(ref["QH_i"]) > 1.0, "Ce_i": np.abs(ref["QL_i"]) > 1.0,
                "Ch_w": np.abs(ref["QH_w"]) > 1.0, "Ce_w": np.abs(ref["QL_w"]) > 1.0}
    inputs = {k: f[k] for k in ("sit", "sst", "t_zt", "hum_zt", "wind", "slp", "frice")}
    last = {k: v[-1] for k, v in inputs.items()} if ice.startswith("lg15") else None
    run = pu.oce_ice_runner(OracleSession, ice, oce, 2.0, 10.0, 20, {"q": 0, "dp": 1, "rh": 2}[hum], cxn, last)
    assert _compare(f"oce_ice {ice}+{oce}", got, ref, keys, sizeable, inputs, run) <= TOL
    if oce is None:
        assert np.all(got["QH_w"] == 0.0) and np.all(got["Tau"] == 0.0)
    else:
        A = f["frice"]
        assert np.allclose(got["QH"], A * got["QH_i"] + (1 - A) * got["QH_w"], rtol=1e-14, atol=1e-12)
    assert np.all(got["Evap_i"] <= 0.0)


def test_oce_ice_subset_of_outputs_and_scenario(ab):
    """Only the cell means requested (the ice fluxes then live in scratch memory); test_ice.sh scenario."""
    from oracle.oracle import OracleSession
    f = synth.ice_fields(5000)
    ab.reset()
    ab.set_nb_iter(20)
    full = ab.oce_ice("an05", "ecmwf", 2.0, 10.0, **f)
    part = ab.oce_ice("an05", "ecmwf", 2.0, 10.0, **f, want=("Tau", "QH", "QL", "Evap"))
    for k in ("Tau", "QH", "QL", "Evap"):
        assert np.array_equal(full[k], part[k])
    one = lambda v: np.array([v])
    got = ab.oce_ice("lg15_io", "ecmwf", 2.0, 10.0, one(270.15), one(271.35), one(276.15), one(0.004), one(3.0), one(101000.0), one(0.8))
    o = OracleSession()
    o.set_nb_iter(20)
    ref = o.oce_ice("lg15_io", "ecmwf", 2.0, 10.0, one(270.15), one(271.35), one(276.15), one(0.004), one(3.0), one(101000.0), one(0.8))
    for k in ("Cd_i", "Ch_i", "QH_i", "QL_i", "Tau_i", "QH_w", "Tau_w", "QH"):
        assert got[k][0] == pytest.approx(ref[k][0], rel=1e-11)


def test_ice_errors(ab):
    f = synth.ice_fields(16)
    ab.reset()
    with pytest.raises(ab.AerobulkError) as e:
        ab.oce_ice("best", "ecmwf", 2.0, 10.0, **f)
    assert e.value.code == 7
    with pytest.raises(ab.AerobulkError) as e:
        ab.oce_ice("an05", "coare9", 2.0, 10.0, **f)
    assert e.value.code == 7
    with pytest.raises(ab.AerobulkError) as e:
        ab.turb_ice("easy", 2.0, 10.0, f["sit"], f["t_zt"], f["hum_zt"], f["hum_zt"], f["wind"])
    assert e.value.code == 101
    # the reference's rough_leng_tq fail-stop (roughness Reynolds number in ]2.49999, 2.5[), same inputs as the CPU test
    one = lambda v: np.array([v])
    with pytest.raises(ab.AerobulkError) as e:
        ab.turb_ice("an05", 2.0, 10.0, one(263.15), one(265.15), one(0.0018), one(0.0015), one(3.239102012771403))
    assert e.value.code == 10 and "zsmoot" in e.value.message
    r = ab.turb_ice("an05", 2.0, 10.0, one(263.15), one(265.15), one(0.0018), one(0.0015), one(3.3))
    assert np.isfinite(r["Cd"][0])
    f["wind"][3] = 300.0
    with pytest.raises(ab.AerobulkError) as e:
        ab.oce_ice("nemo", None, 2.0, 10.0, **f)
    assert e.value.code == 8


@pytest.mark.parametrize("algo,zt,hum", [("nemo", 2.0, "q"), ("an05", 2.0, "rh"), ("lu12", 10.0, "dp"), ("lg15", 2.0, "q"),
                                         ("lg15", 10.0, "rh"), ("an05", 10.0, "q")])
def test_series_ice_matches_oracle(ab, algo, zt, hum):
    """aerobulk_gpu_series_ice against the oracle's restatement of src/ice/test_aerobulk_buoy_series_ice.f90:326-470:
    all 21 series, records without ice read 0 on both sides."""
    from oracle.oracle import OracleSession, OracleError
    n = 40000
    f = synth.ice_fields(n, seed=314, humidity=hum)
    rng = np.random.default_rng(7)
    f = dict(sic=f["frice"], sit=f["sit"], t_zt=f["t_zt"], hum_zt=f["hum_zt"], wind=f["wind"], slp=f["slp"],
             rad_sw=np.maximum(0.0, 400.0 * rng.random(n) - 80.0), rad_lw=170.0 + 140.0 * rng.random(n))
    ab.reset()
    ab.set_nb_iter(20)                 # src/ice/test_aerobulk_buoy_series_ice.f90:77
    o = OracleSession(threads=8)
    o.set_nb_iter(20)
    hk = {"q": 0, "dp": 1, "rh": 2}[hum]
    got, ref, f = _both(lambda d: ab.series_ice(algo, zt, 10.0, **d, hum_kind=hum),
                        lambda d: o.series_ice(algo, zt, 10.0, **d, hum_kind=hk), f, ab.AerobulkError, OracleError)
    ice = f["sic"] > 0.01
    assert 0 < (~ice).sum() < n
    ren = {"Cd_i": "Cd", "Ch_i": "Ch", "Ce_i": "Ce", "TAU": "Tau", "SBLM": "Evap", "Ublk": "Ub", "RiB_zt": "RiB", "RiB_zu": "RiB",
           "Qlw": "QH", "QNS": "QH", "Qsw": "QH"}
    worst = 0.0
    worst_pt = np.zeros(n)
    for k in ab.SERIES_ICE_OUT:
        g, r = got[k], ref[k]
        assert np.all(np.isfinite(g)), k
        if k not in ("Qsw", "RiB_zt"):
            assert np.all(g[~ice] == 0.0) and np.all(r[~ice] == 0.0), k
        base = ren.get(k, k)
        if base == "L":
            g, r = 1.0 / np.where(ice, g, 1.0), 1.0 / np.where(ice, r, 1.0)
        e = np.abs(g - r) / (np.abs(r) + SCALE[base])
        if k == "Ch_i":
            e = np.where(np.abs(ref["QH"]) > 1.0, e, 0.0)
        if k == "Ce_i":
            e = np.where(np.abs(ref["QL"]) > 1.0, e, 0.0)
        bad = int((e > TOL).sum())
        assert bad <= max(1, int(2e-5 * n)), (algo, k, bad, float(e.max()))
        worst = max(worst, float(np.sort(e)[-2]))
        worst_pt = np.maximum(worst_pt, e)
    _prove(f"series_ice {algo} zt={zt} {hum}", worst_pt, f, pu.series_ice_runner(OracleSession, algo, zt, 10.0, 20, hk),
           pu.ice_scale(ab.SERIES_ICE_OUT))
    assert worst <= TOL
    # a subset of outputs gives the same bits
    part = ab.series_ice(algo, zt, 10.0, **f, hum_kind=hum, want=("QNS", "TAU"))
    assert np.array_equal(part["QNS"], got["QNS"]) and np.array_equal(part["TAU"], got["TAU"])
    with pytest.raises(ab.AerobulkError) as e:
        ab.series_ice("easy", zt, 10.0, **f, hum_kind=hum)
    assert e.value.code == 7


def test_series_cli_ice(ab, tmp_path):
    """python -m aerobulk_b200.series_cli --ice: CSV with the ERA5 column names of test_aerobulk_buoy_series_ice.f90:179-211
    (deg C temperatures, RH, u10/v10) -> the program's 14 series, equal to a direct aerobulk_gpu_series_ice call."""
    import os, subprocess, sys
    n = 48
    f = synth.ice_fields(n, seed=8, humidity="rh")
    rng = np.random.default_rng(2)
    ang = rng.uniform(0, 2 * np.pi, n)
    u10, v10 = f["wind"] * np.cos(ang), f["wind"] * np.sin(ang)
    rsw, rlw = 250.0 * rng.random(n), 180.0 + 90.0 * rng.random(n)
    fin, fout = tmp_path / "ice.csv", tmp_path / "out.csv"
    with open(fin, "w") as fh:
        fh.write("# synthetic ice station\ntime, siconc, istl1, t2m, rh_air, u10, v10, msl, ssrd, strd\n")
        for i in range(n):
            row = [f["frice"][i], f["sit"][i] - 273.15, f["t_zt"][i] - 273.15, f["hum_zt"][i], u10[i], v10[i], f["slp"][i], rsw[i], rlw[i]]
            fh.write(f"2019-02-{1 + i // 24:02d} {i % 24:02d}:00," + ",".join(repr(float(x)) for x in row) + "\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "aerobulk_b200.series_cli", str(fin), str(fout), "--ice", "--algo", "lu12"],
                       cwd=root, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = open(fout).read().strip().splitlines()
    hdr = lines[0].split(",")
    assert hdr[:5] == ["time", "Wind", "A", "rho_a", "Qlat"] and len(lines) == n + 1
    got = np.array([[float(x) for x in l.split(",")[1:]] for l in lines[1:]])
    ab.reset()
    ab.set_nb_iter(20)
    # the CLI converted the temperatures back to K and u10, v10 to a speed: feed the API the same values
    ref = ab.series_ice("lu12", 2.0, 10.0, f["frice"], (f["sit"] - 273.15) + 273.15, (f["t_zt"] - 273.15) + 273.15, f["hum_zt"],
                        np.hypot(u10, v10), f["slp"], rsw, rlw, hum_kind="rh")
    for j, k in enumerate(("rho_zu", "QL", "QH", "Qlw", "QNS", "Qsw", "TAU", "SBLM", "Cd_i", "Ch_i", "z0", "RiB_zt", "RiB_zu", "CdN")):
        assert np.array_equal(got[:, 2 + j], ref[k]), k
    r = subprocess.run([sys.executable, "-m", "aerobulk_b200.series_cli", str(fin), str(fout), "--ice", "--algo", "ncar"],
                       cwd=root, capture_output=True, text=True)
    assert r.returncode == 2
