"""How the caller's arrays reach the kernel must not change what the turb, series and sea-ice entry points compute.

Every case runs on 80 000 points (above the 65 536-point bounce threshold) through each transport of
aerobulk_b200/csrc/ab_api.cu (Transport):
  - pageable numpy arrays: the copy threads and the pinned bounce slab;
  - pinned torch tensors: device aliases of the caller's memory (zero-copy);
  - CUDA tensors with on_device = 1: the caller's device pointers;
  - pageable numpy arrays in a process with AEROBULK_GPU_BOUNCE=0: staged cudaMemcpyAsync (compared by hash).
All outputs must be bit-identical.  Every output array starts filled with a sentinel, so the outputs the reference
leaves alone (turb's T_s, q_s without the skin schemes; oce_ice's over-water outputs and cell means without leads) are
seen to be untouched, not merely written with the same value."""
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from aerobulk_b200 import synth

pytestmark = pytest.mark.gpu
NI, NJ = 400, 200
N = NI * NJ
SENTINEL = 7.25
TURB_OUT = ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")


def _turb_inputs():
    f = synth.fields(NI, NJ, seed=4242)
    tc = f["sst"] - 273.15
    es = 611.2 * np.exp(17.67 * tc / (tc + 243.5))
    flat = lambda a: np.ravel(a, order="F").astype(np.float64)
    lon = np.broadcast_to(np.linspace(0.0, 360.0, NI, endpoint=False)[:, None], (NI, NJ))
    return dict(T_s=flat(f["sst"]), q_s=flat(0.98 * 0.622 * es / (f["slp"] - 0.378 * es)), t_zt=flat(f["t_zt"] + 0.0196),
                q_zt=flat(f["hum_zt"]), U_zu=flat(np.hypot(f["U_zu"], f["V_zu"])), Qsw=flat(f["rad_sw"]),
                rad_lw=flat(f["rad_lw"]), slp=flat(f["slp"]), plong=flat(lon))


def _ice_inputs():
    f = synth.ice_fields(N, seed=99)
    tc = f["sit"] - 273.15
    f["qs_i"] = 0.622 * 611.2 * np.exp(22.46 * tc / (tc + 272.62)) / f["slp"]
    rng = np.random.default_rng(1)
    f["rad_sw"], f["rad_lw"] = 300.0 * rng.random(N), 180.0 + 100.0 * rng.random(N)
    return f


def _series_inputs():
    d = synth.station_series(20, N // 20, seed=5)
    return {k: np.ascontiguousarray(v, dtype=np.float64 if k != "isecday_utc" else np.int32) for k, v in d.items()}


def _turb(algo, skin, opt):
    def call(L, p, on_device):
        arr = (C.c_void_p * 10)(*[p(k) for k in ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10", "pdT_cs", "pdT_wl",
                                                  "pHz_wl")])
        sk = dict(Qsw=p("Qsw"), rad_lw=p("rad_lw"), slp=p("slp"), plong=p("plong")) if skin else \
            dict(Qsw=None, rad_lw=None, slp=None, plong=None)
        return L.aerobulk_gpu_turb(algo.encode(), 1, 2.0, 10.0, NI, NJ, p("T_s"), p("t_zt"), p("q_s"), p("q_zt"), p("U_zu"),
                                   int(skin), int(skin), *[p(k) for k in TURB_OUT], sk["Qsw"], sk["rad_lw"], sk["slp"],
                                   43200, sk["plong"], C.cast(arr, C.c_void_p), on_device)
    ins = ("t_zt", "q_zt", "U_zu") + (("Qsw", "rad_lw", "slp", "plong") if skin else ())
    # T_s, q_s are INTENT(inout): without the skin schemes they keep the caller's values
    return dict(inputs=_turb_inputs, ins=ins, inout=("T_s", "q_s"), outs=TURB_OUT + opt, untouched=(), call=call,
                inout_untouched=not skin)


def _turb_ice():
    opt = ("CdN", "xu_star")

    def call(L, p, on_device):
        arr = (C.c_void_p * 8)(*[p(k) for k in ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10", "CdN_frm")])
        return L.aerobulk_gpu_turb_ice(b"lu12", 2.0, 10.0, NI, NJ, p("sit"), p("t_zt"), p("qs_i"), p("hum_zt"), p("wind"),
                                       p("frice"), None, *[p(k) for k in TURB_OUT], C.cast(arr, C.c_void_p), on_device)
    return dict(inputs=_ice_inputs, ins=("sit", "t_zt", "qs_i", "hum_zt", "wind", "frice"), inout=(), outs=TURB_OUT + opt,
                untouched=(), call=call)


def _oce_ice(oce):
    from aerobulk_b200.model import OCE_ICE_OUT
    # with leads: Tau_i, QL_i, Evap_i not asked for, so the cell means read them from scratch
    outs = OCE_ICE_OUT if oce is None else ("QH_i", "Cd_i", "Cd_w", "QH_w", "Tau_w", "Tau", "QH", "QL", "Evap")
    untouched = tuple(k for k in OCE_ICE_OUT[17:]) if oce is None else ()

    def call(L, p, on_device):
        arr = (C.c_void_p * len(OCE_ICE_OUT))(*[p(k) for k in OCE_ICE_OUT])
        return L.aerobulk_gpu_oce_ice(b"nemo", None if oce is None else oce.encode(), 2.0, 10.0, N, p("sit"), p("sst"),
                                      p("t_zt"), p("hum_zt"), 0, p("wind"), p("slp"), p("frice"), None,
                                      C.cast(arr, C.c_void_p), on_device)
    return dict(inputs=_ice_inputs, ins=("sit", "sst", "t_zt", "hum_zt", "wind", "slp", "frice"), inout=(), outs=outs,
                untouched=untouched, call=call)


def _series():
    from aerobulk_b200.model import SERIES_OUT

    def call(L, p, on_device):
        d = p.inputs
        Nt, S = d["isecday_utc"].shape[0], d["lon"].shape[0]
        arr = (C.c_void_p * len(SERIES_OUT))(*[p(k) for k in SERIES_OUT])
        return L.aerobulk_gpu_series(b"coare3p6", Nt, S, 2.0, 10.0, d["isecday_utc"].ctypes.data, p("lon"), p("sst"),
                                     p("t_zt"), p("hum_zt"), 0, p("wind"), p("slp"), p("rad_sw"), p("rad_lw"), 1,
                                     C.cast(arr, C.c_void_p), on_device)
    return dict(inputs=_series_inputs, ins=("lon", "sst", "t_zt", "hum_zt", "wind", "slp", "rad_sw", "rad_lw"), inout=(),
                outs=SERIES_OUT, untouched=(), call=call)


def _series_ice():
    from aerobulk_b200.model import SERIES_ICE_OUT

    def call(L, p, on_device):
        return L.aerobulk_gpu_series_ice(b"lg15", 2.0, 10.0, N, p("frice"), p("sit"), p("t_zt"), p("hum_zt"), 0, p("wind"),
                                         p("slp"), p("rad_sw"), p("rad_lw"),
                                         C.cast((C.c_void_p * len(SERIES_ICE_OUT))(*[p(k) for k in SERIES_ICE_OUT]),
                                                C.c_void_p), on_device)
    return dict(inputs=_ice_inputs, ins=("frice", "sit", "t_zt", "hum_zt", "wind", "slp", "rad_sw", "rad_lw"), inout=(),
                outs=SERIES_ICE_OUT, untouched=(), call=call)


CASES = {
    "turb-coare3p6-skin": lambda: _turb("coare3p6", True, ("CdN", "xu_star", "pdT_cs", "pdT_wl")),
    "turb-ncar": lambda: _turb("ncar", False, ("CdN", "xL")),
    "turb_ice-lu12": _turb_ice,
    "oce_ice-nemo-ecmwf": lambda: _oce_ice("ecmwf"),
    "oce_ice-nemo": lambda: _oce_ice(None),
    "series-coare3p6-skin": _series,
    "series_ice-lg15": _series_ice,
}


def run(name, mode):
    """Outputs (and in/out arrays) of case `name` as numpy arrays, with the caller's arrays in `mode`:
    "pageable" (numpy), "pinned" (pinned torch tensors) or "device" (CUDA tensors, on_device = 1)."""
    import aerobulk_b200 as ab
    case = CASES[name]()
    d = case["inputs"]()
    if mode == "pageable":
        mk = lambda a: a.copy()
        full = lambda n: np.full(n, SENTINEL)
        ptr = lambda x: x.ctypes.data
        back = lambda x: x
    else:
        import torch
        if mode == "pinned":
            mk = lambda a: torch.from_numpy(a.copy()).pin_memory()
            full = lambda n: torch.full((n,), SENTINEL, dtype=torch.float64).pin_memory()
        else:
            mk = lambda a: torch.from_numpy(a).cuda()
            full = lambda n: torch.full((n,), SENTINEL, dtype=torch.float64, device="cuda")
        ptr = lambda x: x.data_ptr()
        back = lambda x: x.cpu().numpy()
    bufs = {k: mk(d[k]) for k in case["ins"] + case["inout"]}
    bufs.update({k: full(N) for k in case["outs"]})

    class P:
        inputs = d

        def __call__(self, k):
            return ptr(bufs[k]) if k in bufs else None
    L = ab.lib()
    ab.reset()
    if mode == "device":
        import torch
        torch.cuda.synchronize()   # the inputs and sentinels are written on torch's stream
    rc = case["call"](L, P(), int(mode == "device"))
    if mode == "device":
        torch.cuda.synchronize()   # aerobulk_gpu_turb on device pointers is asynchronous
    assert rc == 0, (name, mode, rc, ab.last_error())
    res = {k: back(bufs[k]) for k in case["outs"] + case["inout"]}
    for k in case["untouched"]:
        assert np.all(res[k] == SENTINEL), (name, mode, k)
    for k in set(case["outs"]) - set(case["untouched"]):
        assert not np.all(res[k] == SENTINEL), (name, mode, k, "not written")
    if case.get("inout_untouched"):
        for k in case["inout"]:
            assert res[k].tobytes() == d[k].tobytes(), (name, mode, k)
    return res


def digest(res):
    h = hashlib.sha256()
    for k in sorted(res):
        h.update(k.encode())
        h.update(np.ascontiguousarray(res[k]).tobytes())
    return h.hexdigest()


@pytest.fixture(scope="module")
def pageable():
    return {name: run(name, "pageable") for name in CASES}


@pytest.mark.parametrize("mode", ["pinned", "device"])
@pytest.mark.parametrize("name", list(CASES))
def test_transport_gives_the_same_bits(pageable, name, mode):
    got = run(name, mode)
    assert set(got) == set(pageable[name])
    for k in got:
        assert got[k].tobytes() == pageable[name][k].tobytes(), (name, mode, k)


def test_staged_copies_give_the_same_bits(pageable):
    """AEROBULK_GPU_BOUNCE=0 is read once per process: the staged copies run in a subprocess."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = ("import sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]\n"
              "import test_gpu_host_transport as t\n"
              "for name in t.CASES: print('HASH', name, t.digest(t.run(name, 'pageable')))\n")
    r = subprocess.run([sys.executable, "-c", script, root, os.path.join(root, "tests")], cwd=root,
                       env={**os.environ, "AEROBULK_GPU_BOUNCE": "0"}, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    staged = dict(l.split()[1:] for l in r.stdout.splitlines() if l.startswith("HASH"))
    assert staged == {name: digest(res) for name, res in pageable.items()}
