"""Pageable (ordinary) host arrays of 65536 elements or more: the host-array entry points other than aerobulk_model move
them through the library's pinned slab on its copy threads (aerobulk_b200/csrc/ab_api.cu: Transport) instead of
driver-staged copies.  Every point (station) is independent, so the same input cut in two pieces that each stay below the
threshold (staged path) must give the same bits."""
import numpy as np
import pytest

from aerobulk_b200 import synth

pytestmark = pytest.mark.gpu
NI, NJ = 400, 200          # 80000 points; halves of 40000


@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    return ab


def _halves(a):
    return np.asfortranarray(a[:, :NJ // 2]), np.asfortranarray(a[:, NJ // 2:])


def _join(lo, hi):
    return {k: np.concatenate([lo[k], hi[k]], axis=1) for k in lo}


def _turb_inputs():
    f = synth.fields(NI, NJ, seed=4242)
    tc = f["sst"] - 273.15
    es = 611.2 * np.exp(17.67 * tc / (tc + 243.5))
    ssq = np.asfortranarray(0.98 * 0.622 * es / (f["slp"] - 0.378 * es))
    theta = np.asfortranarray(f["t_zt"] + 0.0098 * 2.0)
    wnd = np.asfortranarray(np.hypot(f["U_zu"], f["V_zu"]))
    lon = np.asfortranarray(np.broadcast_to(np.linspace(0.0, 360.0, NI, endpoint=False)[:, None], (NI, NJ)).copy())
    return f, ssq, theta, wnd, lon


@pytest.mark.parametrize("algo,skin", [("coare3p6", True), ("ecmwf", True), ("ncar", False)])
def test_turb_large_pageable_arrays(ab, algo, skin):
    f, ssq, theta, wnd, lon = _turb_inputs()
    want = ("CdN", "xu_star", "xL") + (("pdT_cs", "pdT_wl") if skin else ())

    def run(sl):
        ab.reset()
        ab.set_nb_iter(6)
        kw = dict(l_use_cs=True, l_use_wl=True, Qsw=sl(f["rad_sw"]), rad_lw=sl(f["rad_lw"]), slp=sl(f["slp"]),
                  isecday_utc=43200, plong=sl(lon)) if skin else {}
        return ab.turb(algo, 1, 2.0, 10.0, sl(f["sst"]), sl(theta), sl(ssq), sl(f["hum_zt"]), sl(wnd), want=want, **kw)

    whole = run(lambda a: a)
    parts = _join(run(lambda a: _halves(a)[0]), run(lambda a: _halves(a)[1]))
    for k in whole:
        assert np.array_equal(whole[k], parts[k]), k
    if not skin:   # INTENT(inout) arguments untouched without the skin schemes
        assert np.array_equal(whole["T_s"], f["sst"]) and np.array_equal(whole["q_s"], ssq)
    ab.reset()


def test_turb_ice_and_oce_ice_large_pageable_arrays(ab):
    n = NI * NJ
    f = synth.ice_fields(n, seed=99)
    shp = lambda a: np.asfortranarray(a.reshape((NI, NJ), order="F"))
    tc = f["sit"] - 273.15
    siq = 0.622 * 611.2 * np.exp(22.46 * tc / (tc + 272.62)) / f["slp"]
    ab.reset()
    ab.set_nb_iter(8)

    def ice(sl):
        return ab.turb_ice("lu12", 2.0, 10.0, sl(shp(f["sit"])), sl(shp(f["t_zt"])), sl(shp(siq)), sl(shp(f["hum_zt"])),
                           sl(shp(f["wind"])), frice=sl(shp(f["frice"])), want=("CdN", "xu_star"))

    whole = ice(lambda a: a)
    parts = _join(ice(lambda a: _halves(a)[0]), ice(lambda a: _halves(a)[1]))
    for k in whole:
        assert np.array_equal(whole[k], parts[k]), k

    h = n // 2
    for oce in ("ecmwf", None):
        whole = ab.oce_ice("nemo", oce, 2.0, 10.0, **f)
        lo = ab.oce_ice("nemo", oce, 2.0, 10.0, **{k: v[:h].copy() for k, v in f.items()})
        hi = ab.oce_ice("nemo", oce, 2.0, 10.0, **{k: v[h:].copy() for k, v in f.items()})
        for k in whole:
            assert np.array_equal(whole[k], np.concatenate([lo[k], hi[k]])), (oce, k)
        if oce is None:   # no leads: the over-water outputs are left as the caller passed them
            assert np.all(whole["QH_w"] == 0.0) and np.all(whole["Tau_w"] == 0.0)

    rng = np.random.default_rng(1)
    d = dict(sic=f["frice"], sit=f["sit"], t_zt=f["t_zt"], hum_zt=f["hum_zt"], wind=f["wind"], slp=f["slp"],
             rad_sw=300.0 * rng.random(n), rad_lw=180.0 + 100.0 * rng.random(n))
    whole = ab.series_ice("lg15", 2.0, 10.0, **d)
    lo = ab.series_ice("lg15", 2.0, 10.0, **{k: v[:h].copy() for k, v in d.items()})
    hi = ab.series_ice("lg15", 2.0, 10.0, **{k: v[h:].copy() for k, v in d.items()})
    for k in whole:
        assert np.array_equal(whole[k], np.concatenate([lo[k], hi[k]])), k
    ab.reset()


@pytest.mark.parametrize("algo", ["coare3p6", "ecmwf"])
def test_series_large_pageable_arrays(ab, algo):
    Nt, S = 24, 3000          # 72000 records; 36000 per half
    d = synth.station_series(Nt, S, seed=5)
    names = ("sst", "t_zt", "hum_zt", "wind", "slp", "rad_sw", "rad_lw")

    def run(sl):
        return ab.series(algo, 2.0, 10.0, d["isecday_utc"], d["lon"][sl], *[np.ascontiguousarray(d[k][:, sl]) for k in names])

    ab.reset()
    whole = run(slice(None))
    lo, hi = run(slice(0, S // 2)), run(slice(S // 2, S))
    for k in whole:
        assert np.array_equal(whole[k], np.concatenate([lo[k], hi[k]], axis=1), equal_nan=True), k


_KNOB_SCRIPT = r"""
import hashlib, sys
import numpy as np
import aerobulk_b200 as ab
from aerobulk_b200 import synth
ni, nj, nt = 640, 250, 3
f = synth.fields(ni, nj, seed=11)
names = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
outs = {k: np.zeros((ni, nj), order="F") for k in ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")}
ab.set_verbose(False)
h = hashlib.sha256()
for jt in range(1, nt + 1):
    ab.aerobulk_model(jt, nt, "coare3p6", 2., 10., *[f[k] for k in names], Niter=5, l_use_skin=True,
                      rad_sw=f["rad_sw"], rad_lw=f["rad_lw"], out=outs)
    for k in sorted(outs):
        h.update(outs[k].tobytes())
g = synth.ice_fields(ni * nj, seed=3)
r = ab.oce_ice("nemo", "ncar", 2.0, 10.0, **g, want=("Tau", "QH", "QL"))
for k in sorted(r):
    h.update(r[k].tobytes())
print("HASH", h.hexdigest())
"""


def test_pageable_path_knobs_do_not_change_results():
    """The environment knobs of the pageable-array path (read once per process, hence subprocesses): driver-staged copies,
    a pinned-slab budget too small for the grid (fallback), one copy thread, plain stores, small chunks -- same bits."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hashes = {}
    for tag, env in {"default": {}, "no bounce": {"AEROBULK_GPU_BOUNCE": "0"}, "slab budget 1 MB": {"AEROBULK_GPU_BOUNCE_MAX_MB": "1"},
                     "1 thread, plain stores": {"AEROBULK_GPU_HOST_THREADS": "1", "AEROBULK_GPU_COPY_STREAMING": "0"},
                     "small chunks, 3 threads": {"AEROBULK_GPU_BOUNCE_CHUNK_POINTS": "20000", "AEROBULK_GPU_HOST_THREADS": "3"}}.items():
        r = subprocess.run([sys.executable, "-c", _KNOB_SCRIPT], cwd=root, env={**os.environ, **env}, capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, (tag, r.stderr[-2000:])
        hashes[tag] = [l for l in r.stdout.splitlines() if l.startswith("HASH")][0]
    assert len(set(hashes.values())) == 1, hashes
