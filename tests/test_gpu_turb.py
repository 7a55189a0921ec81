"""SURVEY.md 8f row 1: the direct TURB_* entry (aerobulk_gpu_turb) against the oracle's TURB_* restatement:
real isecday_utc / longitudes (dawn reset of the COARE warm layer), cool-skin and warm-layer switched
independently, optional outputs (CdN, ChN, CeN, z0, u*, L, UN10, dT_cs, dT_wl, Hz_wl)."""
import numpy as np
import pytest

import parity_util as pu
from aerobulk_b200 import synth

pytestmark = pytest.mark.gpu
TOL = 1e-10
WANT = ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10")


@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    return ab


def _inputs(Ni, Nj):
    f = synth.fields(Ni, Nj)
    tc = f["sst"] - 273.15
    es = 611.2 * np.exp(17.67 * tc / (tc + 243.5))
    ssq = 0.98 * 0.622 * es / (f["slp"] - 0.378 * es)
    theta = f["t_zt"] + 0.0098 * 2.0
    wnd = np.hypot(f["U_zu"], f["V_zu"])
    lon = np.asfortranarray(np.broadcast_to(np.linspace(0.0, 360.0, Ni, endpoint=False)[:, None], (Ni, Nj)).copy())
    return f, np.asfortranarray(ssq), np.asfortranarray(theta), np.asfortranarray(wnd), lon


def _cmp(tag, got, ref, keys, n, inputs, run_oracle):
    """Scaled error per output (S_f: parity_util.TURB_SCALE; L compared as 1/L).  A non-finite output fails; at most
    max(1, 2e-5 n) points of an output above TOL, and every point above TOL must be proven to sit where the oracle
    itself is sensitive to ulp-level input nudges (parity_util.prove_flips with run_oracle)."""
    g, r = pu.metric_view({k: got[k] for k in keys}), pu.metric_view({k: ref[k] for k in keys})
    worst = np.zeros(n)
    for k in keys:
        assert np.all(np.isfinite(g[k])), (tag, k, "non-finite output")
        e = pu.scaled_error(g[k], r[k], pu.TURB_SCALE[k])
        bad = int((e > TOL).sum())
        assert bad <= max(1, int(2e-5 * n)), (tag, k, bad, float(e.max()))
        worst = np.maximum(worst, e)
    bad = np.flatnonzero(worst > TOL)
    if bad.size:
        proven = pu.prove_flips(bad, worst[bad], inputs, run_oracle, tag, scale={k: pu.TURB_SCALE[k] for k in keys})
        assert proven.all(), (tag, "points above 1e-10 where the oracle is NOT sensitive to ulp-level input nudges",
                              bad[~proven].tolist(), worst[bad][~proven].tolist())


@pytest.mark.parametrize("algo", ["ncar", "andreas", "coare3p0", "coare3p6", "ecmwf"])
def test_turb_noskin_with_optional_outputs(ab, algo):
    from oracle.oracle import OracleSession
    Ni, Nj = 192, 96
    f, ssq, theta, wnd, _ = _inputs(Ni, Nj)
    ab.reset()
    ab.set_nb_iter(8)
    got = ab.turb(algo, 1, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, want=WANT)
    o = OracleSession(threads=8)
    o.set_nb_iter(8)
    ref = o.turb(algo, 1, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, want=WANT)
    assert np.array_equal(got["T_s"], f["sst"]) and np.array_equal(got["q_s"], ssq)   # untouched without skin
    inputs = dict(T_s=f["sst"], t_zt=theta, q_s=ssq, q_zt=f["hum_zt"], U_zu=wnd)
    _cmp(f"turb {algo}", got, ref, ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu") + WANT, Ni * Nj, inputs,
         pu.turb_runner(OracleSession, algo, 2.0, 10.0, 8))


@pytest.mark.parametrize("algo,cs,wl", [("coare3p6", True, False), ("coare3p6", False, True), ("coare3p6", True, True),
                                        ("coare3p0", True, True), ("ecmwf", True, True), ("ecmwf", False, True)])
def test_turb_skin_day_cycle_with_real_solar_time(ab, algo, cs, wl):
    """24 hourly steps with isecday_utc = 3600 (kt-1) and longitudes 0..360: every point crosses its local dawn
    (solar hour in ]4, 6.5]) at a different step, where WL_COARE resets its state (mod_skin_coare.f90:159-163)."""
    from oracle.oracle import OracleSession
    Ni, Nj, Nt = 96, 24, 24
    f, ssq, theta, wnd, lon = _inputs(Ni, Nj)
    ab.reset()
    ab.set_nb_iter(5)
    ab.set_nitend(Nt)
    o = OracleSession(threads=8)
    o.set_nb_iter(5)
    o.set_nitend(Nt)
    want = ("xu_star",) + (("pdT_cs",) if cs else ()) + (("pdT_wl", "pHz_wl") if wl else ())
    resets = 0
    prev_dT = None
    qsw_all = []
    for kt in range(1, Nt + 1):
        isd = 3600 * (kt - 1)
        # net solar flux following the LOCAL solar hour of each longitude
        hr = (isd / 3600.0 + lon / 15.0) % 24.0
        qsw = np.asfortranarray(np.maximum(0.0, 800.0 * np.sin(np.pi * (hr - 6.0) / 12.0)))
        qsw_all.append(qsw)
        kw = dict(l_use_cs=cs, l_use_wl=wl, Qsw=qsw, rad_lw=f["rad_lw"], slp=f["slp"], isecday_utc=isd, plong=lon, want=want)
        got = ab.turb(algo, kt, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, **kw)
        ref = o.turb(algo, kt, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, **kw)
        inputs = dict(T_s=f["sst"], t_zt=theta, q_s=ssq, q_zt=f["hum_zt"], U_zu=wnd, Qsw=list(qsw_all), rad_lw=f["rad_lw"],
                      slp=f["slp"], plong=lon)
        run = pu.turb_runner(OracleSession, algo, 2.0, 10.0, 5, cs, wl, isecday=[3600 * (j - 1) for j in range(1, kt + 1)],
                             nitend=Nt)
        _cmp(f"turb {algo} cs={cs} wl={wl} kt={kt}", got, ref, ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu", "T_s", "q_s") + want,
             Ni * Nj, inputs, lambda pi: run(pi)[-1:])
        if wl and algo != "ecmwf":
            dT = np.ravel(got["pdT_wl"], order="F")
            if prev_dT is not None:
                resets += int(((prev_dT > 1e-3) & (dT == 0.0)).sum())
            prev_dT = dT
    if wl and algo != "ecmwf":
        assert resets > 0            # the dawn reset did fire somewhere
    assert ab.get_state(0, Ni * Nj) is None   # *_EXIT at kt == nitend


def test_turb_argument_errors(ab):
    f, ssq, theta, wnd, lon = _inputs(16, 8)
    ab.reset()
    with pytest.raises(ab.AerobulkError) as e:
        ab.turb("ncar", 1, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, l_use_cs=True, Qsw=f["rad_sw"], rad_lw=f["rad_lw"], slp=f["slp"])
    assert e.value.code == 2
    with pytest.raises(ab.AerobulkError) as e:
        ab.turb("coare3p6", 1, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, l_use_cs=True)
    assert e.value.code == 3
    with pytest.raises(ab.AerobulkError) as e:     # warm layer needs the longitudes
        ab.turb("coare3p6", 1, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, l_use_wl=True, Qsw=f["rad_sw"], rad_lw=f["rad_lw"], slp=f["slp"])
    assert e.value.code == 3
    with pytest.raises(ab.AerobulkError) as e:     # kt > 1 without its kt == 1
        ab.turb("coare3p6", 2, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, l_use_wl=True, Qsw=f["rad_sw"], rad_lw=f["rad_lw"], slp=f["slp"], plong=lon)
    assert e.value.code == 9
    ab.reset()


def test_turb_and_turb_ice_with_pinned_arrays_zero_copy(ab):
    """Pinned arrays: aerobulk_gpu_turb / aerobulk_gpu_turb_ice work on the caller's memory directly; same bits."""
    import ctypes as C
    import torch
    Ni, Nj = 160, 90
    n = Ni * Nj
    f, ssq, theta, wnd, lon = _inputs(Ni, Nj)
    ab.reset()
    ab.set_nb_iter(6)
    ab.set_nitend(1)
    ref = ab.turb("coare3p6", 1, 2.0, 10.0, f["sst"], theta, ssq, f["hum_zt"], wnd, l_use_cs=True, l_use_wl=True,
                  Qsw=0.934 * f["rad_sw"], rad_lw=f["rad_lw"], slp=f["slp"], isecday_utc=43200, plong=lon, want=("xu_star", "pdT_cs"))
    pin = lambda a: torch.from_numpy(np.ravel(a, order="F").copy()).pin_memory()
    t = {k: pin(v) for k, v in dict(Ts=f["sst"], qs=ssq, th=theta, q=f["hum_zt"], w=wnd, Qsw=0.934 * f["rad_sw"],
                                     rlw=f["rad_lw"], slp=f["slp"], lon=lon).items()}
    o = {k: torch.zeros(n, dtype=torch.float64).pin_memory() for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu", "us", "dTcs")}
    opt = (C.c_void_p * 10)(None, None, None, None, o["us"].data_ptr(), None, None, o["dTcs"].data_ptr(), None, None)
    ab.reset()
    ab.set_nb_iter(6)
    ab.set_nitend(1)
    p = lambda x: x.data_ptr()
    rc = ab.lib().aerobulk_gpu_turb(b"coare3p6", 1, 2.0, 10.0, Ni, Nj, p(t["Ts"]), p(t["th"]), p(t["qs"]), p(t["q"]), p(t["w"]),
                                    1, 1, p(o["Cd"]), p(o["Ch"]), p(o["Ce"]), p(o["t_zu"]), p(o["q_zu"]), p(o["Ubzu"]),
                                    p(t["Qsw"]), p(t["rlw"]), p(t["slp"]), 43200, p(t["lon"]), C.cast(opt, C.c_void_p), 0)
    assert rc == 0, ab.last_error()
    flat = lambda a: np.ravel(a, order="F")
    for k, r in (("Cd", "Cd"), ("Ch", "Ch"), ("Ce", "Ce"), ("t_zu", "t_zu"), ("q_zu", "q_zu"), ("Ubzu", "Ubzu"),
                 ("us", "xu_star"), ("dTcs", "pdT_cs")):
        assert np.array_equal(o[k].numpy(), flat(ref[r])), k
    assert np.array_equal(t["Ts"].numpy(), flat(ref["T_s"])) and np.array_equal(t["qs"].numpy(), flat(ref["q_s"]))
    ab.reset()
