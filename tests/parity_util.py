"""Shared machinery of the GPU parity tests.

Metric (SURVEY.md 8d, BASELINE.json north_star): per output field f
    err_f = |gpu - oracle| / (|oracle| + S_f),   S = 10 W/m2 (QL, QH), 1e-2 N/m2 (tau), 1e-5 kg/m2/s (Evap), 1 K (T_s)
Gate: err <= TOL = 1e-10 at every point, EXCEPT points that are proven to sit on a discontinuity (or an
ill-conditioned spot) of the reference algorithm itself:

  branch-flip proof -- for every point above TOL the ORACLE is re-run on that point with its inputs nudged by
  +-1 ulp (then +-4, +-16, +-64 ulp: the GPU arithmetic differs from glibc by a few ulp per transcendental and
  contracts FMAs, so an intermediate quantity can be off by some tens of ulp after a few iterations).  The point
  is accepted only if the oracle's OWN answer moves by at least PROOF_RATIO x the GPU's deviation under one of
  those nudges, i.e. the reference algorithm is discontinuous / ill-conditioned there at the rounding level
  (SIGN-selected stable/unstable psi, RiB < 0.15 switch of ANDREAS, LKB table edges, warm-layer thresholds,
  MAX/MIN clips: SURVEY.md 7 "hard parts").  A point whose oracle answer stays put is a REAL mismatch and fails.

The same proof serves the other entry points (TURB_*, sea ice, station series): `scale` names their S_f, and
`failstop` accepts a nudge that makes the reference STOP (AN05's rough_leng_tq, code 10: a window of the roughness
Reynolds number where the reference has no answer at all) as proof of a discontinuity.

The number of proven points must stay below OUTLIER_FRACTION of the grid.  Their error is not capped: the reference
has genuine jumps (NCAR's ChN switches 18 -> 32.7 with the sign of zeta, src/mod_blk_ncar.f90:210: two ADJACENT doubles
of t_zt give QH = 4.73 and 9.13 W/m2, tests/test_parity_util_cpu.py::test_gate_proves_a_real_discontinuity).
"""
from __future__ import annotations

import re

import numpy as np

from aerobulk_b200 import synth

TOL = 1e-10
OUTLIER_FRACTION = 2e-5
UNPROVEN_MAX = 1e-9         # without the proof machinery (no oracle callback) nothing may exceed this
PROOF_RATIO = 0.1
NUDGES = (1, 4, 16, 64)

IN_KEYS = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
RAD_KEYS = ("rad_sw", "rad_lw")

# S_f of the TURB_* outputs (tests/test_gpu_turb.py): 0 = purely relative; the Obukhov length is compared as 1/L
TURB_SCALE = {"Cd": 0.0, "Ch": 0.0, "Ce": 0.0, "t_zu": 1.0, "q_zu": 0.0, "Ubzu": 1e-2, "T_s": 1.0, "q_s": 0.0,
              "CdN": 0.0, "ChN": 0.0, "CeN": 0.0, "xz0": 0.0, "xu_star": 0.0, "xL": 1e-3, "xUN10": 1e-2,
              "pdT_cs": 0.0, "pdT_wl": 0.0, "pHz_wl": 1e-2}
# S_f of the sea-ice outputs (tests/test_gpu_ice.py); _i / _w suffixed names use the scale of their base name
ICE_SCALE = {"Cd": 1e-3, "Ch": 1e-3, "Ce": 1e-3, "t_zu": 1.0, "q_zu": 1e-3, "Ubzu": 1e-2, "CdN": 1e-3, "ChN": 1e-3,
             "CeN": 1e-3, "xz0": 1e-5, "xu_star": 1e-2, "xL": 1e-2, "xUN10": 1e-2, "CdN_frm": 1e-3,
             "theta_zu": 1.0, "Ub": 1e-2, "RiB": 1e-2, "z0": 1e-5, "u_star": 1e-2, "L": 1e-2, "UN10": 1e-2, "rho_zu": 1.0,
             "Tau": 1e-2, "QH": 10.0, "QL": 10.0, "Evap": 1e-5}
# series_ice names -> the ICE_SCALE entry they are measured with
SERIES_ICE_BASE = {"Cd_i": "Cd", "Ch_i": "Ch", "Ce_i": "Ce", "TAU": "Tau", "SBLM": "Evap", "Ublk": "Ub", "RiB_zt": "RiB",
                   "RiB_zu": "RiB", "Qlw": "QH", "QNS": "QH", "Qsw": "QH"}
INVERTED = ("xL", "L", "L_i", "L_w")   # Obukhov lengths: L = 1/(1/L) blows up at neutrality, 1/L is compared


def ice_scale(names) -> dict:
    """{output name: S_f} for sea-ice outputs (turb_ice, oce_ice, series_ice names)."""
    out = {}
    for k in names:
        base = SERIES_ICE_BASE.get(k, k[:-2] if k.endswith(("_i", "_w")) else k)
        out[k] = ICE_SCALE[base]
    return out


def metric_view(d: dict) -> dict:
    """Outputs as the gate compares them: flat (Fortran order), Obukhov lengths as 1/L."""
    out = {}
    for k, v in d.items():
        v = np.ravel(np.asarray(v, dtype=np.float64), order="F")
        out[k] = 1.0 / v if k in INVERTED else v
    return out


def scaled_error(g: np.ndarray, r: np.ndarray, s: float) -> np.ndarray:
    return np.abs(g - r) / (np.abs(r) + s + 1e-300)


def worst_per_point(got: dict, ref: dict) -> np.ndarray:
    """max over the output fields of the scaled error, per point (flattened, Fortran order)."""
    errs = synth.parity_errors(got, ref)
    assert set(errs) == set(ref), (set(errs), set(ref))
    w = None
    for k, e in errs.items():
        assert not np.isnan(got[k]).any(), (k, "NaN in GPU output")
        e = np.ravel(e, order="F")
        w = e if w is None else np.maximum(w, e)
    return w


def _nudge(a: np.ndarray, ulps: int) -> np.ndarray:
    """a moved by `ulps` units in the last place (sign of ulps = direction); zeros stay zero (calm wind, night)."""
    out = a.copy()
    step = np.where(ulps > 0, np.inf, -np.inf)
    for _ in range(abs(ulps)):
        out = np.where(out != 0.0, np.nextafter(out, step), out)
    return out


def _variants(point_inputs: dict, ulps: int):
    """All single-field +-ulps nudges plus all-fields-together, for the selected points (1-D arrays of length m)."""
    keys = list(point_inputs)
    out = []
    for s in (+1, -1):
        for k in keys:
            if point_inputs[k] is None:
                continue
            v = dict(point_inputs)
            v[k] = _nudge(point_inputs[k], s * ulps)
            out.append(v)
        out.append({k: (None if a is None else _nudge(a, s * ulps)) for k, a in point_inputs.items()})
    return out


def _take(point_inputs: dict, keep: np.ndarray) -> dict:
    out = {}
    for k, a in point_inputs.items():
        if a is None:
            out[k] = None
        elif isinstance(a, list):
            out[k] = [np.ascontiguousarray(x[keep]) for x in a]
        else:
            out[k] = np.ascontiguousarray(a[keep])
    return out


def _run_stopping(run_oracle, point_inputs: dict, m: int, failstop):
    """run_oracle on the m selected points; with `failstop` (an error code), a point on which the oracle stops with that
    code is taken out and the rest run again.  Returns (outputs with NaN at the stopped points, stopped mask)."""
    live = np.arange(m)
    stopped = np.zeros(m, dtype=bool)
    while live.size:
        try:
            outs = run_oracle(point_inputs if live.size == m else _take(point_inputs, live))
        except Exception as e:   # OracleError (the oracle package is not imported here)
            if failstop is None or getattr(e, "code", None) != failstop:
                raise
            j = int(re.search(r"point (\d+)", str(e)).group(1)) - 1
            stopped[live[j]] = True
            live = np.delete(live, j)
            continue
        full = []
        for o in outs:
            f = {}
            for k, v in o.items():
                x = np.full(m, np.nan)
                x[live] = np.ravel(v)
                f[k] = x
            full.append(f)
        return full, stopped
    return None, stopped


def prove_flips(idx: np.ndarray, err_gpu: np.ndarray, inputs: dict, run_oracle, tag: str = "", scale: dict | None = None,
                failstop: int | None = None) -> np.ndarray:
    """idx: flat (Fortran-order) indices of the points above TOL; err_gpu: their scaled GPU-oracle error;
    inputs: {name: flat array of the WHOLE field or None, or a list of such per time step for rad_sw};
    run_oracle(point_inputs) -> list of output dicts (one per time step) for 1-D inputs of the selected points.
    scale: {output name: S_f} of the compared outputs (default synth.PARITY_SCALE, the aerobulk_model outputs);
    outputs not named in it are not looked at.  failstop: error code of a reference fail-stop (AN05's rough_leng_tq,
    10) that counts as proof when a nudge triggers it on a point.
    Returns a bool array: True where the oracle itself moves by >= PROOF_RATIO * err_gpu under some nudge."""
    scale = synth.PARITY_SCALE if scale is None else scale
    sel = {}
    for k, a in inputs.items():
        if a is None:
            sel[k] = None
        elif isinstance(a, (list, tuple)):
            sel[k] = [np.ascontiguousarray(np.ravel(x, order="F")[idx]) for x in a]
        else:
            sel[k] = np.ascontiguousarray(np.ravel(a, order="F")[idx])
    base, stop0 = _run_stopping(run_oracle, sel, idx.size, failstop)
    assert not stop0.any(), (tag, "the oracle stops on the unperturbed inputs", idx[stop0].tolist())
    proven = np.zeros(idx.size, dtype=bool)
    spread_best = np.zeros(idx.size)
    used = np.zeros(idx.size, dtype=int)
    for ulps in NUDGES:
        # the time-dependent rad_sw list is nudged as a whole (same direction at every step)
        flat = {k: v for k, v in sel.items() if not isinstance(v, list)}
        lists = {k: v for k, v in sel.items() if isinstance(v, list)}
        for var in _variants(flat, ulps):
            for s in ((+1, -1) if lists else (0,)):
                full = dict(var)
                for k, v in lists.items():
                    full[k] = [_nudge(x, s * ulps) if s else x for x in v]
                outs, stopped = _run_stopping(run_oracle, full, idx.size, failstop)
                spread = np.zeros(idx.size)
                for o, b in zip(outs or [], base):
                    for k in b:
                        if k in scale:
                            spread = np.fmax(spread, np.abs(o[k] - b[k]) / (np.abs(b[k]) + scale[k] + 1e-300))
                spread[stopped] = np.inf     # the reference has no answer an ulp away: a genuine discontinuity
                newly = (~proven) & (spread >= PROOF_RATIO * err_gpu)
                used[newly] = ulps
                proven |= newly
                spread_best = np.maximum(spread_best, spread)
        if proven.all():
            break
    for i in range(idx.size):
        print(f"[flip-proof] {tag} point {int(idx[i])}: gpu-oracle err {err_gpu[i]:.3e}, oracle moves by "
              f"{spread_best[i]:.3e} under <= {used[i] or NUDGES[-1]} ulp input nudges -> {'PROVEN' if proven[i] else 'NOT PROVEN'}")
    return proven


def assert_parity(tag: str, worst: np.ndarray, inputs: dict | None = None, run_oracle=None, scale: dict | None = None,
                  failstop: int | None = None, uncapped: np.ndarray | None = None) -> dict:
    """worst: per-point worst scaled error (over fields, and over steps for a session).  A NaN fails.
    uncapped: mask of points (an appended block of edge cases) that are not counted against OUTLIER_FRACTION; every
    one of them above TOL must still be proven.  scale / failstop: see prove_flips."""
    n = worst.size
    assert not np.isnan(worst).any(), (tag, "NaN in the scaled error", np.flatnonzero(np.isnan(worst))[:10].tolist())
    bad = np.flatnonzero(worst > TOL)
    s = np.sort(worst)
    rep = {"max": float(s[-1]), "second": float(s[-2]) if n > 1 else float(s[-1]), "above_tol": int(bad.size), "n": int(n),
           "proven": 0, "max_proven": 0.0, "max_unproven": float(worst[worst <= TOL].max(initial=0.0))}
    print(f"[parity] {tag}: n={n} max {rep['max']:.3e} 2nd {rep['second']:.3e} points>1e-10: {bad.size}")
    if bad.size == 0:
        return rep
    capped = bad if uncapped is None else bad[~uncapped[bad]]
    n_capped = n if uncapped is None else int(n - uncapped.sum())
    assert capped.size <= max(1, int(OUTLIER_FRACTION * n_capped)), (tag, "too many points above 1e-10", capped.size, n_capped)
    if run_oracle is None or inputs is None:
        assert float(worst[bad].max()) <= UNPROVEN_MAX, (tag, "point above 1e-9 and no branch-flip proof available")
        return rep
    proven = prove_flips(bad, worst[bad], inputs, run_oracle, tag, scale=scale, failstop=failstop)
    rep["proven"] = int(proven.sum())
    rep["max_proven"] = float(worst[bad][proven].max(initial=0.0))
    print(f"[parity] {tag}: proven {rep['proven']} of {bad.size}, worst proven {rep['max_proven']:.3e}, "
          f"worst unproven {rep['max_unproven']:.3e}")
    assert proven.all(), (tag, "points above 1e-10 where the oracle itself is NOT sensitive to ulp-level input nudges",
                          bad[~proven].tolist(), worst[bad][~proven].tolist())
    return rep


def oracle_runner(OracleSession, algo, zt, zu, nb_iter, skin, nt=1, threads=4, hum_first=None):
    """run_oracle callback for prove_flips: a fresh oracle session over `nt` steps on 1-D point arrays.
    AEROBULK_INIT detects the humidity type from field statistics: a handful of selected points could be classified
    differently from the full field, so the selected points are preceded by nothing -- the synthetic fields are 'sh'
    (< 0.08) / 'rh' / 'dp' at every single point, which the detection reads the same way for any subset."""

    def run(pi):
        s = OracleSession(threads=threads)
        outs = []
        for jt in range(1, nt + 1):
            kw = dict(Niter=nb_iter)
            if skin:
                rsw = pi["rad_sw"][jt - 1] if isinstance(pi["rad_sw"], list) else pi["rad_sw"]
                kw.update(l_use_skin=True, rad_sw=rsw, rad_lw=pi["rad_lw"])
            outs.append(s.model(jt, nt, algo, zt, zu, *[pi[k] for k in IN_KEYS], **kw))
        return outs

    return run


def turb_runner(OracleSession, algo, zt, zu, nb_iter, cs=False, wl=False, isecday=(0,), nitend=None, threads=4):
    """run_oracle callback for the TURB_* entry: kt = 1 .. len(isecday) on a fresh oracle session, one step per entry
    of `isecday` (isecday_utc of that step).  Point inputs: T_s, t_zt, q_s, q_zt, U_zu and, for the skin schemes, Qsw (an
    array, or a list with one per step), rad_lw, slp, plong.  Returns the outputs of every step, through metric_view."""

    def run(pi):
        s = OracleSession(threads=threads)
        s.set_nb_iter(nb_iter)
        s.set_nitend(nitend or len(isecday))
        outs = []
        for kt, isd in enumerate(isecday, start=1):
            kw = {}
            if cs or wl:
                q = pi["Qsw"]
                kw = dict(Qsw=q[kt - 1] if isinstance(q, list) else q, rad_lw=pi["rad_lw"], slp=pi["slp"],
                          isecday_utc=isd, plong=pi.get("plong"))
            o = s.turb(algo, kt, zt, zu, pi["T_s"], pi["t_zt"], pi["q_s"], pi["q_zt"], pi["U_zu"], l_use_cs=cs,
                       l_use_wl=wl, want=tuple(k for k in TURB_SCALE if k in s.TURB_OPT), **kw)
            outs.append(metric_view(o))
        return outs

    return run


def _with_last(pi: dict, last: dict | None) -> dict:
    """LG15 takes one form drag for all points from the LAST point of the call (mod_blk_ice_lg15.f90): a subset of
    points is run with the original last point appended, so its form drag is the one of the full call."""
    if last is None:
        return pi
    return {k: (None if v is None else np.append(v, last[k])) for k, v in pi.items()}


def _drop_last(o: dict, last: dict | None) -> dict:
    return o if last is None else {k: v[:-1] for k, v in o.items()}


def turb_ice_runner(OracleSession, algo, zt, zu, nb_iter, cxn=None, last=None, per_point_form_drag=False, threads=4):
    """run_oracle callback for TURB_ICE_*: point inputs Ts_i, t_zt, qs_i, q_zt, U_zu, frice.  `last`: the inputs of the
    call's last point, for LG15 (see _with_last)."""

    def run(pi):
        s = OracleSession(threads=threads)
        s.set_nb_iter(nb_iter)
        p = _with_last(pi, last)
        o = s.turb_ice(algo, zt, zu, p["Ts_i"], p["t_zt"], p["qs_i"], p["q_zt"], p["U_zu"], frice=p["frice"], cxn=cxn,
                       per_point_form_drag=per_point_form_drag, want=s.ICE_OPT)
        return [metric_view(_drop_last(o, last))]

    return run


def oce_ice_runner(OracleSession, ice, oce, zt, zu, nb_iter, hum_kind=0, cxn=None, last=None, threads=4):
    """run_oracle callback for the ice + leads computation: point inputs sit, sst, t_zt, hum_zt, wind, slp, frice."""

    def run(pi):
        s = OracleSession(threads=threads)
        s.set_nb_iter(nb_iter)
        p = _with_last(pi, last)
        o = s.oce_ice(ice, oce, zt, zu, p["sit"], p["sst"], p["t_zt"], p["hum_zt"], p["wind"], p["slp"], p["frice"],
                      hum_kind=hum_kind, cxn=cxn)
        return [metric_view(_drop_last(o, last))]

    return run


def series_ice_runner(OracleSession, algo, zt, zu, nb_iter, hum_kind=0, threads=4):
    """run_oracle callback for the sea-ice station series: point inputs sic, sit, t_zt, hum_zt, wind, slp, rad_sw,
    rad_lw (records are independent)."""

    def run(pi):
        s = OracleSession(threads=threads)
        s.set_nb_iter(nb_iter)
        o = s.series_ice(algo, zt, zu, *[pi[k] for k in ("sic", "sit", "t_zt", "hum_zt", "wind", "slp", "rad_sw", "rad_lw")],
                         hum_kind=hum_kind)
        return [metric_view(o)]

    return run
