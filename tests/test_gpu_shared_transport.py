"""Every host-array entry point shares one transport and one pair of slabs per session (Transport in
aerobulk_b200/csrc/ab_api.cu): a pinned slab the copy threads fill and a device slab for staged copies, both grow-only
and shared by FP64 and FP32 calls.  These tests hold what that sharing must not change.

  - A coare3p6 + skin aerobulk_model session (Nt = 3, 1031 x 450 pageable arrays) with other entry points on larger
    pageable arrays between its steps: an NCAR turb without skin, an oce_ice with leads and a float32 NCAR
    aerobulk_model on an odd number of points, each large enough to regrow both slabs.  The session's outputs and its
    warm-layer state must be those of the same steps run alone on device tensors, and every interleaved call's outputs
    those of the same call on device tensors.
  - aerobulk_init and flux_diagnostics on pageable, pinned and device arrays (device: aerobulk_gpu_init_local_stats +
    aerobulk_gpu_init_from_stats, the same AEROBULK_INIT on device pointers) must agree: statistics, humidity type, the
    jt == 1 model outputs that follow, and the code and message of an error for fields in the wrong units.
Every output array starts filled with a sentinel."""
import ctypes as C

import numpy as np
import pytest

from aerobulk_b200 import synth

pytestmark = pytest.mark.gpu
SENTINEL = 7.25
NT = 3
NI, NJ = 1031, 450
N_BIG = 700_001        # turb and oce_ice: more bytes than the session's slabs hold
N_F32 = 1_300_001      # float32, odd: 11 arrays of it need more than the session's 14 FP64 rows
IN = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
OUT = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")
TURB_OUT = ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")


def _flat(a, dtype=np.float64):
    return np.ascontiguousarray(np.ravel(a, order="F"), dtype=dtype)


def _modes(mode):
    """(make input, make sentinel-filled output, pointer, back to numpy) for arrays in `mode`."""
    if mode == "pageable":
        return (lambda a: a.copy(), lambda n, dt=np.float64: np.full(n, SENTINEL, dtype=dt),
                lambda x: None if x is None else x.ctypes.data, lambda x: x.copy())
    import torch
    tdt = lambda dt: torch.float32 if dt == np.float32 else torch.float64
    if mode == "pinned":
        return (lambda a: torch.from_numpy(a.copy()).pin_memory(),
                lambda n, dt=np.float64: torch.full((n,), SENTINEL, dtype=tdt(dt)).pin_memory(),
                lambda x: None if x is None else x.data_ptr(), lambda x: x.numpy().copy())
    return (lambda a: torch.from_numpy(a.copy()).cuda(),
            lambda n, dt=np.float64: torch.full((n,), SENTINEL, dtype=tdt(dt), device="cuda"),
            lambda x: None if x is None else x.data_ptr(), lambda x: x.cpu().numpy().copy())


def _sync(mode):
    if mode == "device":
        import torch
        torch.cuda.synchronize()   # inputs and sentinels are written on torch's stream; device-pointer calls are asynchronous


# ---- the interleaved calls, each in "pageable" or "device" mode; outputs as numpy arrays
def _turb_inputs():
    f = synth.ice_fields(N_BIG, seed=11)
    tc = f["sit"] - 273.15
    es = 611.2 * np.exp(17.67 * tc / (tc + 243.5))
    return dict(T_s=_flat(f["sit"] + 2.0), q_s=_flat(0.98 * 0.622 * es / (f["slp"] - 0.378 * es)), t_zt=_flat(f["t_zt"]),
                q_zt=_flat(f["hum_zt"]), U_zu=_flat(f["wind"]))


def turb(mode):
    import aerobulk_b200 as ab
    mk, full, ptr, back = _modes(mode)
    d = {k: mk(v) for k, v in _turb_inputs().items()}
    o = {k: full(N_BIG) for k in TURB_OUT + ("CdN", "xL")}
    opt = (C.c_void_p * 10)(*[ptr(o.get(k)) for k in ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10", "pdT_cs",
                                                      "pdT_wl", "pHz_wl")])
    _sync(mode)
    rc = ab.lib().aerobulk_gpu_turb(b"ncar", 1, 2.0, 10.0, N_BIG, 1, ptr(d["T_s"]), ptr(d["t_zt"]), ptr(d["q_s"]),
                                    ptr(d["q_zt"]), ptr(d["U_zu"]), 0, 0, *[ptr(o[k]) for k in TURB_OUT], None, None, None,
                                    43200, None, C.cast(opt, C.c_void_p), int(mode == "device"))
    _sync(mode)
    assert rc == 0, ("turb", mode, ab.last_error())
    return {**{k: back(v) for k, v in o.items()}, "T_s": back(d["T_s"]), "q_s": back(d["q_s"])}


def oce_ice(mode):
    import aerobulk_b200 as ab
    from aerobulk_b200.model import OCE_ICE_OUT
    mk, full, ptr, back = _modes(mode)
    f = synth.ice_fields(N_BIG, seed=12)
    d = {k: mk(_flat(f[k])) for k in ("sit", "sst", "t_zt", "hum_zt", "wind", "slp", "frice")}
    # Tau_i, QL_i, Evap_i not asked for: the cell means read them from device scratch
    o = {k: full(N_BIG) for k in ("QH_i", "Cd_i", "Cd_w", "QH_w", "Tau_w", "Tau", "QH", "QL", "Evap")}
    arr = (C.c_void_p * len(OCE_ICE_OUT))(*[ptr(o.get(k)) for k in OCE_ICE_OUT])
    _sync(mode)
    rc = ab.lib().aerobulk_gpu_oce_ice(b"nemo", b"ecmwf", 2.0, 10.0, N_BIG, *[ptr(d[k]) for k in ("sit", "sst", "t_zt",
                                       "hum_zt")], 0, ptr(d["wind"]), ptr(d["slp"]), ptr(d["frice"]), None,
                                       C.cast(arr, C.c_void_p), int(mode == "device"))
    _sync(mode)
    assert rc == 0, ("oce_ice", mode, ab.last_error())
    return {k: back(v) for k, v in o.items()}


def model_f32(mode):
    """jt == 1 of an NCAR session of the same Nt: it leaves nitend, the sticky skin flag (NCAR has no skin scheme) and
    the humidity type as the coare3p6 session set them."""
    import aerobulk_b200 as ab
    mk, full, ptr, back = _modes(mode)
    f = synth.fields(N_F32, 1, seed=13)
    d = {k: mk(_flat(f[k], np.float32)) for k in IN}
    o = {k: full(N_F32, np.float32) for k in OUT[:5]}
    entry = ab.lib().aerobulk_gpu_model_device_f32 if mode == "device" else ab.lib().aerobulk_gpu_model_f32
    _sync(mode)
    rc = entry(1, NT, b"ncar", 2.0, 10.0, N_F32, 1, *[ptr(d[k]) for k in IN], *[ptr(o[k]) for k in OUT[:5]],
               C.byref(C.c_int(5)), None, None, None, None)
    _sync(mode)
    assert rc == 0, ("model_f32", mode, ab.last_error())
    return {k: back(v) for k, v in o.items()}


OTHERS = {"turb": turb, "oce_ice": oce_ice, "model_f32": model_f32}


def session(mode, between=None):
    """The coare3p6 + skin session on arrays in `mode`: per step the outputs and, before the last step, the warm-layer
    state.  `between(jt)` runs after step jt < NT."""
    import aerobulk_b200 as ab
    mk, full, ptr, back = _modes(mode)
    f = synth.fields(NI, NJ, seed=606)
    ins = {k: mk(_flat(f[k])) for k in IN + ("rad_lw",)}
    entry = ab.lib().aerobulk_gpu_model_device if mode == "device" else ab.lib().aerobulk_gpu_model
    steps = []
    for jt in range(1, NT + 1):
        rsw = mk(_flat(synth.rad_sw_hour(NI, NJ, 10 + 2 * jt)))
        o = {k: full(NI * NJ) for k in OUT}
        _sync(mode)
        rc = entry(jt, NT, b"coare3p6", 2.0, 10.0, NI, NJ, *[ptr(ins[k]) for k in IN], *[ptr(o[k]) for k in OUT[:5]],
                   C.byref(C.c_int(5)), C.byref(C.c_int(1)), ptr(rsw), ptr(ins["rad_lw"]), ptr(o["T_s"]))
        _sync(mode)
        assert rc == 0, ("session", mode, jt, ab.last_error())
        res = {k: back(v) for k, v in o.items()}
        for k, v in res.items():
            assert not np.any(v == SENTINEL), ("session", mode, jt, k, "not written everywhere")
        if jt == NT - 1:
            for w in range(4):
                res[f"state{w}"] = ab.get_state(w, NI * NJ)
                assert res[f"state{w}"] is not None, (mode, w)
        steps.append(res)
        if between and jt < NT:
            between(jt)
    return steps


def _same(got, ref, what):
    assert set(got) == set(ref), what
    for k in got:
        assert got[k].tobytes() == ref[k].tobytes(), (what, k)


@pytest.fixture
def fresh():
    import aerobulk_b200 as ab
    ab.reset()
    ab.set_sort(1)
    ab.set_verbose(False)
    yield ab
    ab.reset()


def test_entry_points_interleaved_in_a_session_share_the_slabs(fresh):
    ab = fresh
    alone = session("device")
    ref = {}
    for name, call in OTHERS.items():
        ab.reset()
        ab.set_verbose(False)
        ref[name] = call("device")
    ab.reset()
    ab.set_sort(1)
    ab.set_verbose(False)
    got = {}

    def between(jt):
        for name, call in OTHERS.items():
            got[(name, jt)] = call("pageable")
    steps = session("pageable", between)
    for jt, (g, r) in enumerate(zip(steps, alone), start=1):
        _same(g, r, ("session step", jt))
    for (name, jt), res in got.items():
        _same(res, ref[name], (name, "after step", jt))
        assert any(not np.all(v == SENTINEL) for v in res.values()), (name, jt)


N_INIT = 70_000   # above the 65 536-point bounce threshold


def _init_fields(celsius=False):
    f = synth.fields(N_INIT, 1, seed=21)
    d = {k: _flat(f[k]) for k in IN + ("rad_lw", "rad_sw")}
    d["rad_sw"] = _flat(synth.rad_sw_hour(N_INIT, 1, 12))
    if celsius:   # every point falls outside the sanity ranges: the reference's error for fields in the wrong units
        d["sst"] = d["sst"] - 273.15
    return d


def _init(mode, d):
    """AEROBULK_INIT on arrays in `mode`: (return code, error message, humidity type)."""
    import aerobulk_b200 as ab
    L = ab.lib()
    mk, _, ptr, _ = _modes(mode)
    a = {k: mk(v) for k, v in d.items()}
    _sync(mode)
    if mode == "device":
        st = np.zeros(64)
        rc = L.aerobulk_gpu_init_local_stats(N_INIT, 1, *[ptr(a[k]) for k in IN], ptr(a["rad_lw"]),
                                             st.ctypes.data_as(C.POINTER(C.c_double)))
        assert rc == 0, ab.last_error()
        rc = L.aerobulk_gpu_init_from_stats(NT, b"coare3p6", C.byref(C.c_int(1)), 1, st.ctypes.data_as(C.POINTER(C.c_double)))
    else:
        rc = L.aerobulk_gpu_init(NT, b"coare3p6", N_INIT, 1, *[ptr(a[k]) for k in IN], C.byref(C.c_int(1)), ptr(a["rad_sw"]),
                                 ptr(a["rad_lw"]))
    return rc, ab.last_error() if rc else "", ab.humidity_type()


def test_aerobulk_init_on_every_kind_of_array(fresh):
    import torch
    ab = fresh
    d = _init_fields()
    res = {}
    for mode in ("pageable", "pinned", "device"):
        ab.reset()
        ab.set_verbose(False)
        rc, msg, hum = _init(mode, d)
        assert rc == 0, (mode, msg)
        # the jt == 1 call that follows, on device tensors
        t = {k: torch.from_numpy(v).cuda() for k, v in d.items()}
        out = {k: torch.full((N_INIT,), SENTINEL, dtype=torch.float64, device="cuda") for k in OUT}
        ab.aerobulk_model_device(1, NT, "coare3p6", 2.0, 10.0, *[t[k] for k in IN], out, Niter=5, l_use_skin=True,
                                 rad_sw=t["rad_sw"], rad_lw=t["rad_lw"])
        torch.cuda.synchronize()
        res[mode] = (hum, {k: v.cpu().numpy() for k, v in out.items()})
    for mode in ("pinned", "device"):
        assert res[mode][0] == res["pageable"][0], mode
        _same(res[mode][1], res["pageable"][1], mode)
    bad = _init_fields(celsius=True)
    errs = {}
    for mode in ("pageable", "pinned", "device"):
        ab.reset()
        ab.set_verbose(False)
        errs[mode] = _init(mode, bad)[:2]
    assert errs["pageable"][0] == 4 and "check unit consistency" in errs["pageable"][1], errs   # AEROBULK_GPU_ERR_ALL_MASKED
    assert errs["pinned"] == errs["pageable"] and errs["device"] == errs["pageable"], errs


def test_flux_diagnostics_on_every_kind_of_array(fresh):
    ab = fresh
    rng = np.random.default_rng(31)
    n = N_INIT
    fields = {k: rng.normal(size=n) * 100.0 for k in OUT}
    fields["Tau_y"] = None   # absent fields are skipped
    L = ab.lib()
    stats = {}
    for mode in ("pageable", "pinned", "device"):
        mk, _, ptr, _ = _modes(mode)
        a = {k: None if v is None else mk(v) for k, v in fields.items()}
        _sync(mode)
        st = np.full(19, SENTINEL)
        rc = L.aerobulk_gpu_flux_diagnostics(n, *[ptr(a[k]) for k in OUT], st.ctypes.data_as(C.POINTER(C.c_double)),
                                             int(mode == "device"))
        assert rc == 0, (mode, ab.last_error())
        stats[mode] = st
    assert stats["pageable"][0] == n
    for mode in ("pinned", "device"):
        assert stats[mode].tobytes() == stats["pageable"].tobytes(), mode
