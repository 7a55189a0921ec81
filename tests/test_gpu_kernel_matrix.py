"""Every template instantiation of libaerobulk_gpu.so against the oracle.

The hot path is template code: each (kernel, template arguments) pair is its own machine code, and `if (!ZTEQ)`,
`if (SKIN)`, CS / WL keep or drop whole blocks of the solvers.  MATRIX below names, for each instantiation the library
holds, one call that launches it.  The CPU census test reads the instantiations out of the built library
(`cuobjdump -symbols`) and fails when one has no entry, so a new template parameter or algorithm cannot ship without a
parity case.  The GPU tests run each entry at two point counts and gate it like the model path (parity_util).

Which instantiation a call launches: each launch_* function picks it through pick_ocean (ab_kernels.cuh) or pick_ice
(ab_ice.cu), from the flags ab_api.cu derives with zt_eq_zu and has_skin_schemes:
  - ZTEQ = |zu - zt| < 0.01, for every kernel;
  - flux_kernel<ALGO, SKIN, ZTEQ> (aerobulk_model): SKIN = l_use_skin for COARE 3.0 / 3.6 and ECMWF, false otherwise;
  - turb_kernel<ALGO, CS, WL, ZTEQ> (TURB_*): CS = l_use_cs, WL = l_use_wl (NCAR and ANDREAS take neither);
  - series_kernel<ALGO, SKIN, ZTEQ> (station series): SKIN as for flux_kernel;
  - ice_turb_kernel / ice_flux_kernel / ice_series_kernel<IALGO, ZTEQ>: lg15_io runs as ICE_LG15;
  - leads_kernel<OALGO, ZTEQ>: OALGO = calgo_oce of the ice + leads call.
Enum values: Algo in ab_device.cuh, IceAlgo in ab_ice.cuh.
"""
from __future__ import annotations

import ctypes as C
import os
import re
import shutil
import subprocess
from typing import NamedTuple, Optional

import numpy as np
import pytest

import parity_util as pu
from aerobulk_b200 import synth

TOL = pu.TOL
ALGO = {"coare3p0": 1, "coare3p6": 2, "ncar": 3, "ecmwf": 4, "andreas": 5}          # abd::Algo
ICE = {"nemo": 1, "easy": 2, "an05": 3, "lu12": 4, "lg15": 5, "lg15_io": 5}          # abd::IceAlgo
SKIN_ALGOS = ("coare3p0", "coare3p6", "ecmwf")
HUM = {"q": 0, "dp": 1, "rh": 2}
CXN_EASY = [1.4e-3, 1.3e-3, 1.2e-3]


def zteq(zt: float, zu: float) -> bool:
    return abs(zu - zt) < 0.01


class Case(NamedTuple):
    entry: str                 # model | turb | series | turb_ice | oce_ice | series_ice
    algo: str
    zt: float
    zu: float = 10.0
    skin: bool = False         # l_use_skin of model / series
    cs: bool = False           # l_use_cs of turb
    wl: bool = False           # l_use_wl of turb
    oce: Optional[str] = None  # calgo_oce of oce_ice
    hum: str = "q"

    def keys(self) -> list:
        z = int(zteq(self.zt, self.zu))
        if self.entry in ("model", "series"):
            k = "flux_kernel" if self.entry == "model" else "series_kernel"
            return [(k, (ALGO[self.algo], int(self.skin and self.algo in SKIN_ALGOS), z))]
        if self.entry == "turb":
            return [("turb_kernel", (ALGO[self.algo], int(self.cs), int(self.wl), z))]
        if self.entry == "turb_ice":
            return [("ice_turb_kernel", (ICE[self.algo], z))]
        if self.entry == "series_ice":
            return [("ice_series_kernel", (ICE[self.algo], z))]
        return [("ice_flux_kernel", (ICE[self.algo], z))] + ([("leads_kernel", (ALGO[self.oce], z))] if self.oce else [])

    def __str__(self):
        opts = "".join(f" {o}" for o, on in (("skin", self.skin), ("cs", self.cs), ("wl", self.wl)) if on)
        oce = f"+{self.oce}" if self.oce else ""
        return f"{self.entry} {self.algo}{oce}{opts} zt={self.zt} zu={self.zu} {self.hum}"


# zt == zu cases run at 10/10; once per kernel family at zt = 9.995: equal by the 0.01 rule, but log(zt) != log(zu)
CASES = [
    Case("model", "coare3p0", 2.0), Case("model", "coare3p0", 10.0),
    Case("model", "coare3p0", 2.0, skin=True), Case("model", "coare3p0", 10.0, skin=True),
    Case("model", "coare3p6", 2.0), Case("model", "coare3p6", 10.0),
    Case("model", "coare3p6", 2.0, skin=True), Case("model", "coare3p6", 10.0, skin=True),
    Case("model", "ecmwf", 2.0), Case("model", "ecmwf", 10.0),
    Case("model", "ecmwf", 2.0, skin=True), Case("model", "ecmwf", 10.0, skin=True),
    Case("model", "ncar", 2.0), Case("model", "ncar", 9.995),
    Case("model", "andreas", 2.0), Case("model", "andreas", 10.0),

    Case("turb", "coare3p0", 2.0), Case("turb", "coare3p0", 10.0),
    Case("turb", "coare3p0", 2.0, cs=True), Case("turb", "coare3p0", 10.0, cs=True),
    Case("turb", "coare3p0", 2.0, wl=True), Case("turb", "coare3p0", 10.0, wl=True),
    Case("turb", "coare3p0", 2.0, cs=True, wl=True), Case("turb", "coare3p0", 10.0, cs=True, wl=True),
    Case("turb", "coare3p6", 2.0), Case("turb", "coare3p6", 10.0),
    Case("turb", "coare3p6", 2.0, cs=True), Case("turb", "coare3p6", 10.0, cs=True),
    Case("turb", "coare3p6", 2.0, wl=True), Case("turb", "coare3p6", 10.0, wl=True),
    Case("turb", "coare3p6", 2.0, cs=True, wl=True), Case("turb", "coare3p6", 9.995, cs=True, wl=True),
    Case("turb", "ecmwf", 2.0), Case("turb", "ecmwf", 10.0),
    Case("turb", "ecmwf", 2.0, cs=True), Case("turb", "ecmwf", 10.0, cs=True),
    Case("turb", "ecmwf", 2.0, wl=True), Case("turb", "ecmwf", 10.0, wl=True),
    Case("turb", "ecmwf", 2.0, cs=True, wl=True), Case("turb", "ecmwf", 10.0, cs=True, wl=True),
    Case("turb", "ncar", 2.0), Case("turb", "ncar", 10.0),
    Case("turb", "andreas", 2.0), Case("turb", "andreas", 10.0),

    Case("series", "coare3p0", 2.0), Case("series", "coare3p0", 10.0),
    Case("series", "coare3p0", 2.0, skin=True), Case("series", "coare3p0", 10.0, skin=True),
    Case("series", "coare3p6", 2.0), Case("series", "coare3p6", 10.0),
    Case("series", "coare3p6", 2.0, skin=True), Case("series", "coare3p6", 10.0, skin=True),
    Case("series", "ecmwf", 2.0), Case("series", "ecmwf", 10.0),
    Case("series", "ecmwf", 2.0, skin=True), Case("series", "ecmwf", 9.995, skin=True),
    Case("series", "ncar", 2.0), Case("series", "ncar", 10.0),
    Case("series", "andreas", 2.0), Case("series", "andreas", 10.0),

    Case("turb_ice", "nemo", 2.0), Case("turb_ice", "nemo", 10.0),
    Case("turb_ice", "easy", 2.0), Case("turb_ice", "easy", 10.0),
    Case("turb_ice", "an05", 2.0), Case("turb_ice", "an05", 9.995),
    Case("turb_ice", "lu12", 2.0), Case("turb_ice", "lu12", 10.0),
    Case("turb_ice", "lg15", 2.0), Case("turb_ice", "lg15_io", 10.0),

    Case("oce_ice", "nemo", 2.0, oce="coare3p0"), Case("oce_ice", "nemo", 10.0, oce="andreas", hum="dp"),
    Case("oce_ice", "easy", 2.0, oce="coare3p6", hum="rh"), Case("oce_ice", "easy", 10.0, oce="ncar"),
    Case("oce_ice", "an05", 2.0, oce="ncar", hum="dp"), Case("oce_ice", "an05", 10.0, oce="coare3p6", hum="rh"),
    Case("oce_ice", "lu12", 2.0, oce="ecmwf"), Case("oce_ice", "lu12", 9.995, oce="coare3p0", hum="dp"),
    Case("oce_ice", "lg15", 2.0, oce="andreas", hum="rh"), Case("oce_ice", "lg15_io", 10.0, oce="ecmwf"),

    Case("series_ice", "nemo", 2.0), Case("series_ice", "nemo", 10.0, hum="rh"),
    Case("series_ice", "an05", 2.0, hum="dp"), Case("series_ice", "an05", 10.0),
    Case("series_ice", "lu12", 2.0, hum="rh"), Case("series_ice", "lu12", 10.0, hum="dp"),
    Case("series_ice", "lg15", 2.0), Case("series_ice", "lg15", 9.995, hum="rh"),
]


def _matrix() -> dict:
    m = {}
    for c in CASES:
        for k in c.keys():
            assert k not in m, (k, str(c), str(m[k]))   # one call per instantiation
            m[k] = c
    return m


MATRIX = _matrix()


# ---------------------------------------------------------------------------------------------------------------------
# census (CPU)
# ---------------------------------------------------------------------------------------------------------------------
_SYM = re.compile(r"_ZN3abk\d+(\w+?_kernel)I((?:Li\d+E|Lb[01]E)+)E")


def _instantiations(lib_path: str) -> set:
    from aerobulk_b200 import build
    cuobjdump = os.path.join(os.path.dirname(os.path.realpath(build._nvcc())), "cuobjdump")
    if not os.path.exists(cuobjdump):
        cuobjdump = shutil.which("cuobjdump")
    assert cuobjdump, "cuobjdump not found next to nvcc"
    out = subprocess.run([cuobjdump, "-symbols", lib_path], capture_output=True, text=True, check=True).stdout
    found = set()
    for name, args in _SYM.findall(out):
        found.add((name, tuple(int(v) for v in re.findall(r"L[ib](\d+)E", args))))
    return found


def test_every_kernel_instantiation_has_a_parity_case():
    from aerobulk_b200 import build
    lib = build.build()
    found = _instantiations(lib)
    assert len(found) > 0, "no templated kernel found in the library"
    missing = sorted(found - set(MATRIX))
    stale = sorted(set(MATRIX) - found)
    assert not missing, ("kernel instantiations without a parity case in MATRIX", missing)
    assert not stale, ("MATRIX entries the library does not instantiate", stale)


# ---------------------------------------------------------------------------------------------------------------------
# inputs: synthetic fields plus an appended block of edge points
# ---------------------------------------------------------------------------------------------------------------------
N_BIG = 3 * 2048 + 777     # synthetic points: a multiple of neither the block (256) nor the sort window (2048)
N_SMALL = 201              # one partial block, one partial sort window
NB_ITER = 6                # MOD(nb_iter, jit) commits the warm layer at jit = 1, 2, 3, 6 (SURVEY 8a quirk 1)
NB_ICE = 10
TAIL = 37                  # sentinel values past n in every device output
SENTINEL = -1.2345e300
STATE_SCALE = (1.0, 20.0, 1e7, 1e3)   # dT_wl [K], Hz_wl [m], Qnt_ac [J/m2], Tau_ac [N s/m2] (test_gpu_parity.py)


def _magnus(t):
    tc = t - 273.15
    return 611.2 * np.exp(17.67 * tc / (tc + 243.5))


def _ocean_edge() -> dict:
    """Exact calm, 0.3-1 m/s and 28-34 m/s winds, air-sea dT from -15 to +10 K, SST at -1.8 and 33 degC, slp 87 000 and
    108 000 Pa, humidity near saturation, Qsw 0 / 1100 and rad_lw 150 / 500 W/m2; then very dry polar air (q < 1e-6,
    where the COARE first guess floors q_zu and COARE 3.0 at zt == zu does not, ab_device.cuh first_guess_coare)."""
    g = np.array(np.meshgrid([0.0, 0.3, 0.6, 1.0, 28.0, 31.0, 34.0], [-15.0, -5.0, 2.0, 10.0], [271.35, 306.15],
                             [87000.0, 108000.0], [0.98, 0.6], [0.0, 1.0], indexing="ij")).reshape(6, -1)
    wind, dT, sst, slp, frac, rad = g
    dry = np.array(np.meshgrid([0.6, 5.0, 15.0], [-10.0, 0.5, 5.0], [1e-7, 8e-7], indexing="ij")).reshape(3, -1)
    m = dry.shape[1]
    wind = np.r_[wind, dry[0]]
    t_zt = np.r_[sst + dT, 271.35 + dry[1]]
    sst = np.r_[sst, np.full(m, 271.35)]
    slp = np.r_[slp, np.full(m, 101000.0)]
    q = np.r_[frac * 0.622 * _magnus(t_zt[:-m]) / slp[:-m], dry[2]]
    rad = np.r_[rad, np.zeros(m)]
    ang = 0.7 * np.arange(wind.size)
    return dict(sst=sst, t_zt=t_zt, hum_zt=q, U_zu=wind * np.cos(ang), V_zu=wind * np.sin(ang), slp=slp,
                rad_sw=1100.0 * rad, rad_lw=150.0 + 350.0 * rad)


def _ocean(size: str):
    """(flat fields, number of synthetic points): 1-D arrays, the edge block after the synthetic points."""
    if size == "small":
        f = synth.fields(67, 3, seed=synth.SEED + 1)
        return {k: np.ravel(v, order="F") for k, v in f.items()}, 201
    f = synth.fields(769, 9)          # 769 x 9 = N_BIG
    f = {k: np.ravel(v, order="F") for k, v in f.items()}
    e = _ocean_edge()
    return {k: np.r_[f[k], e[k]] for k in f}, N_BIG


def _ice_edge(hum: str) -> dict:
    """Air down to 225 K (the humidity conversion evaluates e_sat on both sides of its table's 230 K edge), air-ice dT
    from -15 to +10 K, calm, 0.3-1 and 28-34 m/s winds, rh 60 / 99 %, slp 87 000 / 108 000 Pa, leads at -1.8 degC."""
    g = np.array(np.meshgrid([225.0, 229.99, 230.0, 230.01, 235.0, 250.0, 270.0], [-15.0, -3.0, 10.0],
                             [0.0, 0.3, 1.0, 28.0, 31.0, 34.0], [60.0, 99.0], [87000.0, 108000.0],
                             indexing="ij")).reshape(5, -1)
    t_zt, dT, wind, rh, slp = g
    n = t_zt.size
    i = np.arange(n)
    sit = np.clip(t_zt - dT, 200.0, 273.15)
    esat = _magnus(t_zt)
    hum = {"q": 0.01 * rh * 0.622 * esat / slp, "rh": rh}.get(hum)
    if hum is None:
        ln = np.log(0.01 * rh * esat / 611.2)
        hum = 273.15 + 243.5 * ln / (17.67 - ln)
    return dict(sit=sit, sst=np.where(i % 2 == 0, 271.35, 273.65), t_zt=t_zt, hum_zt=hum, wind=wind, slp=slp,
                frice=np.array([0.0, 0.5, 1.0])[i % 3], rad_sw=np.where(i % 4 < 2, 0.0, 1100.0),
                rad_lw=np.where(i % 3 == 0, 150.0, 500.0))


def _ice(size: str, hum: str):
    if size == "small":
        f = synth.ice_fields(N_SMALL, seed=synth.SEED + 1, humidity=hum)
        n0 = N_SMALL
    else:
        f = dict(synth.ice_fields(N_BIG, humidity=hum))
        n0 = N_BIG
    rng = np.random.default_rng(11)
    f["rad_sw"] = np.maximum(0.0, 400.0 * rng.random(n0) - 80.0)
    f["rad_lw"] = 170.0 + 140.0 * rng.random(n0)
    if size == "small":
        return f, n0
    e = _ice_edge(hum)
    return {k: np.r_[f[k], e[k]] for k in f}, n0


# ---------------------------------------------------------------------------------------------------------------------
# device-pointer calls with sentinel tails
# ---------------------------------------------------------------------------------------------------------------------
class Dev:
    """Device copies of the inputs; every output (and in/out) array is the head of a buffer of n + TAIL values that
    starts filled with SENTINEL, so a write past n shows up in the tail."""

    def __init__(self, n: int):
        import torch
        self.torch, self.n, self.bufs = torch, n, []

    def inp(self, a):
        return None if a is None else self.torch.from_numpy(np.ascontiguousarray(np.ravel(a), dtype=np.float64)).cuda()

    def out(self, init=None):
        b = self.torch.full((self.n + TAIL,), SENTINEL, dtype=self.torch.float64, device="cuda")
        if init is not None:
            b[:self.n] = self.inp(init)
        self.bufs.append(b)
        return b[:self.n]

    def run(self, ab, call):
        self.torch.cuda.synchronize()
        try:
            call()
        finally:
            ab.synchronize()
            self.torch.cuda.synchronize()
        for b in self.bufs:
            tail = b[self.n:].cpu().numpy()
            assert np.all(tail == SENTINEL), ("write past n", self.n, np.flatnonzero(tail != SENTINEL)[:5].tolist())


def _p(t):
    return None if t is None else t.data_ptr()


def _host(d: dict) -> dict:
    return {k: v.cpu().numpy().copy() for k, v in d.items()}


# ---------------------------------------------------------------------------------------------------------------------
# the gate
# ---------------------------------------------------------------------------------------------------------------------
REPORT = {}


def _gate(tag, family, worst, n_syn, inputs, run_oracle, scale, failstop=None):
    """Every point <= TOL or proven (parity_util.assert_parity); the synthetic points keep the 2e-5 cap on proven
    points, the appended edge points have no count cap."""
    uncapped = np.arange(worst.size) >= n_syn
    rep = pu.assert_parity(tag, worst, inputs, run_oracle, scale=scale, failstop=failstop, uncapped=uncapped)
    r = REPORT.setdefault(family, [0.0, 0.0, 0])
    r[0] = max(r[0], rep["max_unproven"])
    r[1] = max(r[1], rep["max_proven"])
    r[2] += rep["proven"]
    print(f"[parity] family {family}: worst unproven {r[0]:.3e}, worst proven {r[1]:.3e}, proven points so far {r[2]}")


def _worst(tag, got, ref, scale, masks=None):
    g, r = pu.metric_view(got), pu.metric_view(ref)
    worst = None
    for k in scale:
        assert np.all(np.isfinite(g[k])), (tag, k, "non-finite output", np.flatnonzero(~np.isfinite(g[k]))[:5].tolist())
        e = pu.scaled_error(g[k], r[k], scale[k])
        if masks and k in masks:
            e = np.where(masks[k], e, 0.0)
        worst = e if worst is None else np.maximum(worst, e)
    return worst


def _state_check(tag, ab, osess, algo, n, worst_state):
    for which in range(1 if algo == "ecmwf" else 4):
        sg, so = ab.get_state(which, n), osess.state(which, n)
        assert sg is not None and so is not None, (tag, which)
        worst_state[:] = np.maximum(worst_state, np.abs(sg - so) / (np.abs(so) + STATE_SCALE[which]))


def _state_gate(tag, worst_state, worst):
    """As test_gpu_parity._session: the state may differ only where the outputs were proven to sit on a branch."""
    bad_state = np.flatnonzero(worst_state > 1e-9)
    print(f"[parity] {tag}: warm-layer state max scaled err {worst_state.max():.3e}, points>1e-9: {bad_state.size}")
    flux_bad = set(np.flatnonzero(worst > TOL).tolist())
    unexplained = [int(i) for i in bad_state if int(i) not in flux_bad]
    assert not unexplained, (tag, "warm-layer state differs where the outputs agree", unexplained[:10])


# ---------------------------------------------------------------------------------------------------------------------
# one runner per entry point
# ---------------------------------------------------------------------------------------------------------------------
RSW_STEP = (1.0, 0.7, 0.35)


def _model_gpu(ab, c, f, nt):
    """aerobulk_model_device over nt steps; returns per-step outputs and the warm-layer state after each step < nt."""
    n = f["sst"].size
    outs, states = [], []
    ab.reset()
    for jt in range(1, nt + 1):
        d = Dev(n)
        ins = [d.inp(f[k]) for k in pu.IN_KEYS]
        out = {k: d.out() for k in ("QL", "QH", "Tau_x", "Tau_y", "Evap") + (("T_s",) if c.skin else ())}
        kw = dict(Niter=NB_ITER)
        if c.skin:
            kw.update(l_use_skin=True, rad_sw=d.inp(RSW_STEP[jt - 1] * f["rad_sw"]), rad_lw=d.inp(f["rad_lw"]))
        d.run(ab, lambda: ab.aerobulk_model_device(jt, nt, c.algo, c.zt, c.zu, *ins, out=out, **kw))
        outs.append(_host(out))
        if c.skin and jt < nt:
            states.append([ab.get_state(w, n) for w in range(1 if c.algo == "ecmwf" else 4)])
    return outs, states


def _run_model(ab, c, size):
    from oracle.oracle import OracleSession
    f, n_syn = _ocean(size)
    n = f["sst"].size
    nt = 3 if c.skin else 1
    runs = {}
    try:
        for mode in (0, 1, 2):
            ab.set_sort(mode)
            runs[mode] = _model_gpu(ab, c, f, nt)
    finally:
        ab.set_sort(1)
    for mode in (0, 2):   # DESIGN.md 3.3: the stability sort changes the order of work, never a bit of the result
        for jt, (a, b) in enumerate(zip(runs[mode][0], runs[1][0]), start=1):
            for k in b:
                assert np.array_equal(a[k], b[k]), (str(c), "sort mode", mode, "step", jt, k)
        for a, b in zip(runs[mode][1], runs[1][1]):
            for x, y in zip(a, b):
                assert np.array_equal(x, y), (str(c), "sort mode", mode, "warm-layer state")
    osess = OracleSession(threads=8)
    worst = np.zeros(n)
    worst_state = np.zeros(n)
    rsw = []
    for jt in range(1, nt + 1):
        kw = dict(Niter=NB_ITER)
        if c.skin:
            rsw.append(RSW_STEP[jt - 1] * f["rad_sw"])
            kw.update(l_use_skin=True, rad_sw=rsw[-1], rad_lw=f["rad_lw"])
        ref = osess.model(jt, nt, c.algo, c.zt, c.zu, *[f[k] for k in pu.IN_KEYS], **kw)
        worst = np.maximum(worst, pu.worst_per_point(runs[1][0][jt - 1], ref))
        if c.skin and jt < nt:
            for w, sg in enumerate(runs[1][1][jt - 1]):
                so = osess.state(w, n)
                worst_state = np.maximum(worst_state, np.abs(sg - so) / (np.abs(so) + STATE_SCALE[w]))
    inputs = {k: f[k] for k in pu.IN_KEYS}
    inputs["rad_sw"] = rsw if c.skin else None
    inputs["rad_lw"] = f["rad_lw"] if c.skin else None
    tag = f"{c} n={n}"
    _gate(tag, "flux_kernel", worst, n_syn, inputs, pu.oracle_runner(OracleSession, c.algo, c.zt, c.zu, NB_ITER, c.skin, nt=nt),
          None)
    if c.skin:
        _state_gate(tag, worst_state, worst)


ISD_TURB = (5 * 3600, 6 * 3600, 7 * 3600)   # around dawn at the longitudes of the grid: the warm-layer reset fires
# S_f of the TURB_* outputs; the skin increments dT_cs and dT_wl are measured in K against S = 1 K, as T_s is here and as
# test_gpu_series.py measures the same increments.  dT_wl restarts from 0 at every dawn and grows from there: a purely
# relative error on it has no floor, so a 1e-14 K difference on a young warm layer would count as a branch flip.
TURB_SCALE = dict(pu.TURB_SCALE, pdT_cs=1.0, pdT_wl=1.0)


def _run_turb(ab, c, size):
    from oracle.oracle import OracleSession
    from aerobulk_b200.model import TURB_OPTIONAL
    f, n_syn = _ocean(size)
    n = f["sst"].size
    skin = c.cs or c.wl
    nt = 3 if c.wl else 1
    ssq = 0.98 * 0.622 * _magnus(f["sst"]) / (f["slp"] - 0.378 * _magnus(f["sst"]))
    theta = f["t_zt"] + 0.0098 * c.zt
    wnd = np.hypot(f["U_zu"], f["V_zu"])
    lon = np.linspace(-180.0, 180.0, n, endpoint=False)
    want = ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10") + (("pdT_cs",) if c.cs else ()) + \
        (("pdT_wl", "pHz_wl") if c.wl else ())
    keys = ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu", "T_s", "q_s") + want
    scale = {k: TURB_SCALE[k] for k in keys}
    L = ab.lib()
    ab.reset()
    ab.set_nb_iter(NB_ITER)
    ab.set_nitend(nt)
    o = OracleSession(threads=8)
    o.set_nb_iter(NB_ITER)
    o.set_nitend(nt)
    worst = np.zeros(n)
    worst_state = np.zeros(n)
    qsw = []
    for kt in range(1, nt + 1):
        qsw.append(RSW_STEP[kt - 1] * f["rad_sw"])
        d = Dev(n)
        Ts, qs = d.out(f["sst"]), d.out(ssq)
        ins = [d.inp(a) for a in (theta, f["hum_zt"], wnd)]
        rad = [d.inp(a) if skin else None for a in (qsw[-1], f["rad_lw"], f["slp"], lon)]
        out = {k: d.out() for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu") + want}
        opt = (C.c_void_p * 10)(*[_p(out.get(k)) for k in TURB_OPTIONAL])

        def call():
            rc = L.aerobulk_gpu_turb(c.algo.encode(), kt, c.zt, c.zu, n, 1, _p(Ts), _p(ins[0]), _p(qs), _p(ins[1]),
                                     _p(ins[2]), int(c.cs), int(c.wl), *[_p(out[k]) for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")],
                                     *[_p(a) for a in rad[:3]], ISD_TURB[kt - 1], _p(rad[3]), C.cast(opt, C.c_void_p), 1)
            ab.model._check(rc)

        d.run(ab, call)
        got = _host(out)
        got["T_s"], got["q_s"] = Ts.cpu().numpy(), qs.cpu().numpy()
        kw = dict(Qsw=qsw[-1], rad_lw=f["rad_lw"], slp=f["slp"], isecday_utc=ISD_TURB[kt - 1], plong=lon) if skin else {}
        ref = o.turb(c.algo, kt, c.zt, c.zu, f["sst"], theta, ssq, f["hum_zt"], wnd, l_use_cs=c.cs, l_use_wl=c.wl,
                     want=want, **kw)
        worst = np.maximum(worst, _worst(str(c), got, ref, scale))
        if c.wl and kt < nt:
            _state_check(str(c), ab, o, c.algo, n, worst_state)
    inputs = dict(T_s=f["sst"], t_zt=theta, q_s=ssq, q_zt=f["hum_zt"], U_zu=wnd)
    if skin:
        inputs.update(Qsw=qsw, rad_lw=f["rad_lw"], slp=f["slp"], plong=lon)
    run = pu.turb_runner(OracleSession, c.algo, c.zt, c.zu, NB_ITER, c.cs, c.wl, isecday=ISD_TURB[:nt])
    tag = f"{c} n={n}"
    _gate(tag, "turb_kernel", worst, n_syn, inputs, run, scale)
    if c.wl:
        _state_gate(tag, worst_state, worst)


def _run_series(ab, c, size):
    from oracle.oracle import OracleSession
    import test_gpu_series as ts
    Nt = 3
    S0 = N_SMALL if size == "small" else N_BIG
    d = synth.station_series(Nt, S0, start_s=4 * 3600)
    if size != "small":   # edge stations: the ocean edge points, constant in time
        e = _ocean_edge()
        m = e["sst"].size
        edge = dict(sst=e["sst"], t_zt=e["t_zt"], hum_zt=e["hum_zt"], wind=np.hypot(e["U_zu"], e["V_zu"]), slp=e["slp"],
                    rad_sw=e["rad_sw"], rad_lw=e["rad_lw"])
        for k, v in edge.items():
            d[k] = np.ascontiguousarray(np.concatenate([d[k], np.broadcast_to(v, (Nt, m))], axis=1))
        d["lon"] = np.r_[d["lon"], np.linspace(-180.0, 180.0, m, endpoint=False)]
    S = d["lon"].size
    n = Nt * S
    ab.reset()
    ab.set_nb_iter(NB_ITER)
    dv = Dev(n)
    ins = {k: dv.inp(d[k]) for k in ts.SERIES_IN}
    lon = dv.inp(d["lon"])
    out = {k: dv.out() for k in ab.SERIES_OUT}
    dv.run(ab, lambda: ab.series_device(c.algo, c.zt, c.zu, d["isecday_utc"], lon, *[ins[k] for k in ts.SERIES_IN],
                                        out=out, l_use_skin=c.skin))
    got = {k: v.reshape(Nt, S) for k, v in _host(out).items()}
    o = OracleSession(threads=8)
    o.set_nb_iter(NB_ITER)
    ref = o.series(c.algo, c.zt, c.zu, **d, l_use_skin=c.skin)

    def rerun(lon_, sub):
        oo = OracleSession(threads=8)
        oo.set_nb_iter(NB_ITER)
        return oo.series(c.algo, c.zt, c.zu, d["isecday_utc"], lon_, **sub, l_use_skin=c.skin)

    # the station gate of test_gpu_series.py: every station above TOL proven with the whole series of that station
    ts._compare(f"{c} S={S}", got, ref, S, d, rerun)
    r = REPORT.setdefault("series_kernel", [0.0, 0.0, 0])
    emax = ts._station_errors(got, ref, S)
    r[0] = max(r[0], float(emax[emax <= TOL].max(initial=0.0)))
    r[1] = max(r[1], float(emax[emax > TOL].max(initial=0.0)))
    r[2] += int((emax > TOL).sum())
    print(f"[parity] family series_kernel: worst unproven {r[0]:.3e}, worst proven {r[1]:.3e}, proven stations so far {r[2]}")


def _both(ab, gpu, ref, f):
    """test_gpu_ice._both: a point that trips AN05's rough_leng_tq fail-stop is replaced by its neighbour."""
    from oracle.oracle import OracleError
    import test_gpu_ice as ti
    return ti._both(gpu, ref, f, ab.AerobulkError, OracleError)


def _run_turb_ice(ab, c, size):
    from oracle.oracle import OracleSession, lib as olib
    from aerobulk_b200.model import ICE_OPTIONAL
    f, n_syn = _ice(size, "q")
    n = f["sit"].size
    Lo = olib()
    f = dict(Ts_i=f["sit"], t_zt=f["t_zt"] + 0.0098 * c.zt, qs_i=np.array([Lo.abo_q_sat_ice(t, p) for t, p in zip(f["sit"], f["slp"])]),
             q_zt=f["hum_zt"], U_zu=f["wind"], frice=f["frice"])
    cxn = CXN_EASY if c.algo == "easy" else None
    cx = None if cxn is None else np.array(cxn)
    L = ab.lib()
    ab.reset()
    ab.set_nb_iter(NB_ICE)
    o = OracleSession(threads=8)
    o.set_nb_iter(NB_ICE)

    def gpu(p):
        d = Dev(n)
        ins = [d.inp(p[k]) for k in ("Ts_i", "t_zt", "qs_i", "q_zt", "U_zu", "frice")]
        out = {k: d.out() for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu") + ICE_OPTIONAL}
        opt = (C.c_void_p * 8)(*[_p(out[k]) for k in ICE_OPTIONAL])
        d.run(ab, lambda: ab.model._check(L.aerobulk_gpu_turb_ice(
            c.algo.encode(), c.zt, c.zu, n, 1, *[_p(t) for t in ins], None if cx is None else cx.ctypes.data,
            *[_p(out[k]) for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")], C.cast(opt, C.c_void_p), 1)))
        return _host(out)

    got, ref, f = _both(ab, gpu, lambda p: o.turb_ice(c.algo, c.zt, c.zu, p["Ts_i"], p["t_zt"], p["qs_i"], p["q_zt"], p["U_zu"],
                                                      frice=p["frice"], cxn=cxn, want=ICE_OPTIONAL), f)
    masks = {"Ch": np.abs(ref["t_zu"] - f["Ts_i"]) > 0.05, "Ce": np.abs(ref["q_zu"] - f["qs_i"]) > 2e-5}
    scale = pu.ice_scale(("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu") + ICE_OPTIONAL)
    last = {k: v[-1] for k, v in f.items()} if c.algo.startswith("lg15") else None
    _gate(f"{c} n={n}", "ice_turb_kernel", _worst(str(c), got, ref, scale, masks), n_syn, f,
          pu.turb_ice_runner(OracleSession, c.algo, c.zt, c.zu, NB_ICE, cxn, last), scale, failstop=10)


def _run_oce_ice(ab, c, size):
    from oracle.oracle import OracleSession
    f, n_syn = _ice(size, c.hum)
    f = {k: f[k] for k in ("sit", "sst", "t_zt", "hum_zt", "wind", "slp", "frice")}
    n = f["sit"].size
    cxn = CXN_EASY if c.algo == "easy" else None
    cx = None if cxn is None else np.array(cxn)
    L = ab.lib()
    ab.reset()
    ab.set_nb_iter(NB_ICE)
    o = OracleSession(threads=8)
    o.set_nb_iter(NB_ICE)

    def gpu(p):
        d = Dev(n)
        ins = [d.inp(p[k]) for k in ("sit", "sst", "t_zt", "hum_zt", "wind", "slp", "frice")]
        out = {k: d.out() for k in ab.OCE_ICE_OUT}
        arr = (C.c_void_p * len(ab.OCE_ICE_OUT))(*[_p(out[k]) for k in ab.OCE_ICE_OUT])
        d.run(ab, lambda: ab.model._check(L.aerobulk_gpu_oce_ice(
            c.algo.encode(), c.oce.encode(), c.zt, c.zu, n, *[_p(t) for t in ins[:4]], HUM[c.hum], *[_p(t) for t in ins[4:]],
            None if cx is None else cx.ctypes.data, C.cast(arr, C.c_void_p), 1)))
        return _host(out)

    got, ref, f = _both(ab, gpu, lambda p: o.oce_ice(c.algo, c.oce, c.zt, c.zu, *[p[k] for k in f], hum_kind=HUM[c.hum], cxn=cxn), f)
    masks = {"Ch_i": np.abs(ref["QH_i"]) > 1.0, "Ce_i": np.abs(ref["QL_i"]) > 1.0,
             "Ch_w": np.abs(ref["QH_w"]) > 1.0, "Ce_w": np.abs(ref["QL_w"]) > 1.0}
    scale = pu.ice_scale(ab.OCE_ICE_OUT)
    last = {k: v[-1] for k, v in f.items()} if c.algo.startswith("lg15") else None
    _gate(f"{c} n={n}", "ice_flux_kernel+leads_kernel", _worst(str(c), got, ref, scale, masks), n_syn, f,
          pu.oce_ice_runner(OracleSession, c.algo, c.oce, c.zt, c.zu, NB_ICE, HUM[c.hum], cxn, last), scale, failstop=10)


def _run_series_ice(ab, c, size):
    from oracle.oracle import OracleSession
    f, n_syn = _ice(size, c.hum)
    keys_in = ("sic", "sit", "t_zt", "hum_zt", "wind", "slp", "rad_sw", "rad_lw")
    f = dict(sic=f["frice"], **{k: f[k] for k in keys_in[1:]})
    n = f["sit"].size
    L = ab.lib()
    ab.reset()
    ab.set_nb_iter(NB_ICE)
    o = OracleSession(threads=8)
    o.set_nb_iter(NB_ICE)

    def gpu(p):
        d = Dev(n)
        ins = [d.inp(p[k]) for k in keys_in]
        out = {k: d.out() for k in ab.SERIES_ICE_OUT}
        arr = (C.c_void_p * len(ab.SERIES_ICE_OUT))(*[_p(out[k]) for k in ab.SERIES_ICE_OUT])
        d.run(ab, lambda: ab.model._check(L.aerobulk_gpu_series_ice(
            c.algo.encode(), c.zt, c.zu, n, *[_p(t) for t in ins[:4]], HUM[c.hum], *[_p(t) for t in ins[4:]],
            C.cast(arr, C.c_void_p), 1)))
        return _host(out)

    got, ref, f = _both(ab, gpu, lambda p: o.series_ice(c.algo, c.zt, c.zu, *[p[k] for k in keys_in], hum_kind=HUM[c.hum]), f)
    ice = f["sic"] > 0.01
    for k in ab.SERIES_ICE_OUT:
        if k not in ("Qsw", "RiB_zt"):   # records without ice read 0 on both sides (test_gpu_ice.py)
            assert np.all(got[k][~ice] == 0.0) and np.all(ref[k][~ice] == 0.0), (str(c), k)
    got["L"], ref["L"] = np.where(ice, got["L"], 1.0), np.where(ice, ref["L"], 1.0)
    masks = {"Ch_i": np.abs(ref["QH"]) > 1.0, "Ce_i": np.abs(ref["QL"]) > 1.0}
    scale = pu.ice_scale(ab.SERIES_ICE_OUT)
    run = pu.series_ice_runner(OracleSession, c.algo, c.zt, c.zu, NB_ICE, HUM[c.hum])

    def run_view(pi):   # the same 1/L convention as the GPU side: L of a record without ice is 0 on both sides
        outs = run(pi)
        for o_ in outs:
            o_["L"] = np.where(np.isfinite(o_["L"]), o_["L"], 1.0)
        return outs

    _gate(f"{c} n={n}", "ice_series_kernel", _worst(str(c), got, ref, scale, masks), n_syn, f, run_view, scale, failstop=10)


RUN = {"model": _run_model, "turb": _run_turb, "series": _run_series, "turb_ice": _run_turb_ice, "oce_ice": _run_oce_ice,
       "series_ice": _run_series_ice}


@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    yield ab
    ab.set_sort(1)
    ab.reset()


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["big", "small"])
@pytest.mark.parametrize("case", CASES, ids=[str(c).replace(" ", "-") for c in CASES])
def test_instantiation_matches_oracle(ab, case, size):
    RUN[case.entry](ab, case, size)
    ab.reset()
