"""aerobulk_model on float32 fields: aerobulk_gpu_model_f32 / aerobulk_gpu_model_device_f32 (include/aerobulk_gpu.h).

The contract, at every output point of every step:

    f32_call(x) == float32_round_to_nearest(f64_call(float64(x)))     bit for bit,

and the warm-layer state after every step is bit-identical to the FP64 session's on the widened inputs.  The float
kernels are the FP64 kernels' twins with float loads and stores (flux_io_kernel<float, ALGO, SKIN, ZTEQ>,
classify_io_kernel<float>, stats_fast_io_kernel<float>, stats_fix_io_kernel<float>, ab_kernels.cu).  The census below
holds them to the rule test_gpu_kernel_matrix.py holds the FP64 kernels to: every float instantiation the library ships
has an entry in F32_MATRIX, and each entry runs on the GPU.

- each flux instantiation on the kernel-matrix fields (synthetic points plus the edge block, and 201 points), humidity
  as sh / rh / dp, under sort modes 0, 1 and 2, with sentinel tails past n;
- skin sessions of 3 steps, and one that alternates float32 and float64 calls;
- every host-array transport (test_gpu_model_transport.py), with the FP64 call's launch count on each;
- AEROBULK_INIT and tau > 10 errors: the FP64 call's codes and messages, and the same end of session;
- aerobulk_gpu_set_devices(2) against one GPU;
- one call per algorithm against the oracle: within half a float ulp of the FP64 gate.
"""
import ctypes as C
import hashlib
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

import parity_util as pu
import test_gpu_kernel_matrix as km
import test_gpu_model_transport as tr
from aerobulk_b200 import synth

gpu = pytest.mark.gpu
F32, F64 = np.float32, np.float64
IN = pu.IN_KEYS
OUT = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")
SENTINEL = F32(-1.2345e30)
TAIL = km.TAIL

# ---------------------------------------------------------------------------------------------------------------------
# case matrix and census (CPU)
# ---------------------------------------------------------------------------------------------------------------------
FLUX_CASES = [c for c in km.CASES if c.entry == "model"]


def _f32_matrix() -> dict:
    m = {}
    for c in FLUX_CASES:
        for name, args in c.keys():
            m[(name.replace("_kernel", "_io_kernel"), args)] = c
    # every jt == 1 device call takes the statistics, every sorting algorithm classifies (sort modes 1 and 2)
    m[("classify_io_kernel", ())] = FLUX_CASES[0]
    m[("stats_fast_io_kernel", ())] = FLUX_CASES[0]
    m[("stats_fix_io_kernel", ())] = FLUX_CASES[0]
    return m


F32_MATRIX = _f32_matrix()
_SYM_F32 = re.compile(r"_ZN3abk\d+(\w+?_io_kernel)If((?:Li\d+E|Lb[01]E)*)E")


def test_every_float_instantiation_has_a_case():
    from aerobulk_b200 import build
    lib = build.build()
    cuobjdump = os.path.join(os.path.dirname(os.path.realpath(build._nvcc())), "cuobjdump")
    if not os.path.exists(cuobjdump):
        cuobjdump = shutil.which("cuobjdump")
    assert cuobjdump, "cuobjdump not found next to nvcc"
    out = subprocess.run([cuobjdump, "-symbols", lib], capture_output=True, text=True, check=True).stdout
    found = {(name, tuple(int(v) for v in re.findall(r"L[ib](\d+)E", args))) for name, args in _SYM_F32.findall(out)}
    assert len([k for k in found if k[0] == "flux_io_kernel"]) == 16, sorted(found)
    assert not sorted(found - set(F32_MATRIX)), ("float instantiations without a case", sorted(found - set(F32_MATRIX)))
    assert not sorted(set(F32_MATRIX) - found), ("cases the library does not instantiate", sorted(set(F32_MATRIX) - found))


def test_argument_checks_come_before_the_device():
    """NULL arrays and jt < 1 are refused before any device work (no GPU needed); Python refuses other dtypes."""
    import aerobulk_b200 as ab
    L = ab.lib()
    a = np.zeros(4, dtype=F32)
    p = a.ctypes.data
    for entry in (L.aerobulk_gpu_model_f32, L.aerobulk_gpu_model_device_f32):
        rc = entry(1, 1, b"ncar", 2.0, 10.0, 4, 1, None, *[p] * 5, *[p] * 5, None, None, None, None, None)
        assert rc == 101, (entry, rc)
        rc = entry(1, 1, b"ncar", 2.0, 10.0, 4, 1, *[p] * 6, p, p, p, p, None, None, None, None, None, None)
        assert rc == 101, (entry, rc)
        rc = entry(0, 1, b"ncar", 2.0, 10.0, 4, 1, *[p] * 6, *[p] * 5, None, None, None, None, None)
        assert rc == 1 and "jt < 1" in ab.last_error(), (entry, rc)
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model_f32(1, 1, "ncar", 2.0, 10.0, *[np.zeros(4)] * 6)
    assert e.value.code == 101
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model_f32(1, 1, "ncar", 2.0, 10.0, *[a] * 6, out={"QL": np.zeros(4)})
    assert e.value.code == 101
    import torch
    t = torch.zeros(4, dtype=torch.float64)
    with pytest.raises(ab.AerobulkError) as e:
        ab.aerobulk_model_device_f32(1, 1, "ncar", 2.0, 10.0, *[t] * 6, out={k: t for k in OUT[:5]})
    assert e.value.code == 101


# ---------------------------------------------------------------------------------------------------------------------
# the contract on device pointers
# ---------------------------------------------------------------------------------------------------------------------
def _ocean(size: str, hum: str) -> dict:
    """The kernel-matrix fields (synthetic points plus the edge block, or 201 points) with humidity as `hum`, rounded to
    float32.  The edge block's specific humidity becomes the rh / dp of the same vapour pressure (Magnus)."""
    if size == "small":
        f = synth.fields(67, 3, seed=synth.SEED + 1, humidity=hum)
        f = {k: np.ravel(v, order="F") for k, v in f.items()}
    else:
        f = {k: np.ravel(v, order="F") for k, v in synth.fields(769, 9, humidity=hum).items()}
        e = km._ocean_edge()
        if hum != "sh":
            vp = e["hum_zt"] * e["slp"] / 0.622
            ln = np.log(vp / 611.2)
            e["hum_zt"] = 100.0 * vp / km._magnus(e["t_zt"]) if hum == "rh" else 273.15 + 243.5 * ln / (17.67 - ln)
        f = {k: np.r_[f[k], e[k]] for k in f}
    return {k: v.astype(F32) for k, v in f.items()}


def _device_session(ab, algo, skin, zt, zu, f, rsw, dtypes, sort=1):
    """One session of len(dtypes) steps on device pointers, step jt with element type dtypes[jt - 1] (F32 / F64) on the
    float32 fields `f` (widened for F64) and rad_sw rsw[jt - 1]; every output buffer has a sentinel tail past n.
    Returns per step the outputs (numpy) and, until the last step, the warm-layer state."""
    import torch
    n = f["sst"].size
    nt = len(dtypes)
    ab.reset()
    ab.set_sort(sort)
    steps = []
    for jt, dt in enumerate(dtypes, start=1):
        tdt = torch.float32 if dt is F32 else torch.float64
        inp = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
        bufs = {k: torch.full((n + TAIL,), float(SENTINEL), dtype=tdt, device="cuda") for k in (OUT if skin else OUT[:5])}
        out = {k: b[:n] for k, b in bufs.items()}
        kw = dict(Niter=km.NB_ITER)
        if skin:
            kw.update(l_use_skin=True, rad_sw=inp(rsw[jt - 1]), rad_lw=inp(f["rad_lw"]))
        fn = ab.aerobulk_model_device_f32 if dt is F32 else ab.aerobulk_model_device
        torch.cuda.synchronize()
        try:
            fn(jt, nt, algo, zt, zu, *[inp(f[k]) for k in IN], out=out, **kw)
        finally:
            ab.synchronize()
            torch.cuda.synchronize()
        for k, b in bufs.items():
            tail = b[n:].cpu().numpy()
            assert np.all(tail == tail.dtype.type(SENTINEL)), ("write past n", algo, jt, k)
        res = {k: v.cpu().numpy().copy() for k, v in out.items()}
        if skin and jt < nt:
            for w in range(1 if algo == "ecmwf" else 4):
                res[f"state{w}"] = ab.get_state(w, n)
        steps.append(res)
    ab.set_sort(1)
    ab.reset()
    return steps


def _assert_contract(got, ref, what):
    """float32 outputs == the FP64 outputs rounded to nearest; warm-layer state bit-identical."""
    assert len(got) == len(ref), what
    for jt, (g, r) in enumerate(zip(got, ref), start=1):
        assert set(g) == set(r), (what, jt)
        for k in g:
            want = r[k] if g[k].dtype == r[k].dtype else r[k].astype(F32)   # float64 -> float32 rounds to nearest
            if g[k].tobytes() != want.tobytes():
                u = np.uint32 if want.itemsize == 4 else np.uint64
                bad = np.flatnonzero(g[k].view(u) != want.view(u))
                raise AssertionError((what, "step", jt, k, "points", bad[:5].tolist(), g[k][bad[:5]], want[bad[:5]]))


def _rsw(f, nt):
    return [(km.RSW_STEP[j] * f["rad_sw"].astype(F64)).astype(F32) for j in range(nt)]


@pytest.fixture(scope="module")
def ab():
    import aerobulk_b200 as ab
    ab.lib()
    yield ab
    ab.set_sort(1)
    ab.reset()


@gpu
@pytest.mark.parametrize("hum", ["sh", "rh", "dp"])
@pytest.mark.parametrize("size", ["big", "small"])
@pytest.mark.parametrize("case", FLUX_CASES, ids=[str(c).replace(" ", "-") for c in FLUX_CASES])
def test_instantiation_keeps_the_contract(ab, case, size, hum):
    f = _ocean(size, hum)
    nt = 3 if case.skin else 1
    rsw = _rsw(f, nt)
    ref = _device_session(ab, case.algo, case.skin, case.zt, case.zu, f, rsw, [F64] * nt)
    for sort in (0, 1, 2):
        got = _device_session(ab, case.algo, case.skin, case.zt, case.zu, f, rsw, [F32] * nt, sort)
        _assert_contract(got, ref, (str(case), size, hum, "sort", sort))


@gpu
@pytest.mark.parametrize("algo", km.SKIN_ALGOS)
def test_skin_session_alternating_element_types(ab, algo):
    """The warm-layer state does not depend on the element type: float32 and float64 steps may alternate."""
    f = _ocean("big", "sh")
    rsw = _rsw(f, 3)
    ref = _device_session(ab, algo, True, 2.0, 10.0, f, rsw, [F64] * 3)
    _assert_contract(_device_session(ab, algo, True, 2.0, 10.0, f, rsw, [F32] * 3), ref, (algo, "f32"))
    _assert_contract(_device_session(ab, algo, True, 2.0, 10.0, f, rsw, [F32, F64, F32]), ref, (algo, "f32 f64 f32"))


# ---------------------------------------------------------------------------------------------------------------------
# host-array transports (as test_gpu_model_transport.py)
# ---------------------------------------------------------------------------------------------------------------------
NT = 3
HOST_SENTINEL = 7.25
BIG, SMALL = (1031, 450), (300, 200)
TCASES = {"coare3p6-skin": ("coare3p6", True), "ncar": ("ncar", False)}


def run(case, mode, dtype, shape=BIG):
    """The session of test_gpu_model_transport.run on float32-rounded fields, with arrays of `dtype`: per call the outputs
    (and, until jt == Nt, the warm-layer state) and the number of kernel launches."""
    import aerobulk_b200 as ab
    algo, skin = TCASES[case]
    ni, nj = shape
    n = ni * nj
    flat = lambda a: np.ravel(a, order="F").astype(F32).astype(dtype)
    if mode == "pageable":
        mk = lambda a: a.copy()
        full = lambda: np.full(n, HOST_SENTINEL, dtype=dtype)
        ptr = lambda x: None if x is None else x.ctypes.data
        back = lambda x: x.copy()
    else:
        import torch
        tdt = torch.float32 if dtype is F32 else torch.float64
        if mode == "pinned":
            mk = lambda a: torch.from_numpy(a.copy()).pin_memory()
            full = lambda: torch.full((n,), HOST_SENTINEL, dtype=tdt).pin_memory()
        else:
            mk = lambda a: torch.from_numpy(a).cuda()
            full = lambda: torch.full((n,), HOST_SENTINEL, dtype=tdt, device="cuda")
        ptr = lambda x: None if x is None else x.data_ptr()
        back = lambda x: x.cpu().numpy().copy()
    f = synth.fields(ni, nj, seed=606)
    ins = {k: mk(flat(f[k])) for k in IN + (("rad_lw",) if skin else ())}
    outs = OUT if skin else OUT[:5]
    L = ab.lib()
    entry = {(F64, False): L.aerobulk_gpu_model, (F64, True): L.aerobulk_gpu_model_device,
             (F32, False): L.aerobulk_gpu_model_f32, (F32, True): L.aerobulk_gpu_model_device_f32}[(dtype, mode == "device")]
    ab.reset()
    ab.set_sort(1)
    ab.set_verbose(False)
    steps = []
    for jt in range(1, NT + 1):
        rsw = mk(flat(synth.rad_sw_hour(ni, nj, 10 + 2 * jt))) if skin else None
        o = {k: full() for k in outs}
        if mode == "device":
            torch.cuda.synchronize()
        L.aerobulk_gpu_reset_launch_count()
        rc = entry(jt, NT, algo.encode(), 2.0, 10.0, ni, nj, *[ptr(ins[k]) for k in IN], *[ptr(o[k]) for k in OUT[:5]],
                   C.byref(C.c_int(5)), C.byref(C.c_int(1)) if skin else None, ptr(rsw), ptr(ins.get("rad_lw")),
                   ptr(o.get("T_s")))
        if mode == "device":
            torch.cuda.synchronize()
        assert rc == 0, (case, mode, jt, rc, ab.last_error())
        launches = L.aerobulk_gpu_launch_count()
        res = {k: back(v) for k, v in o.items()}
        for k, v in res.items():
            assert not np.any(v == HOST_SENTINEL), (case, mode, jt, k, "not written everywhere")
        if skin and jt < NT:
            for w in range(4):
                res[f"state{w}"] = ab.get_state(w, n)
        steps.append((res, launches))
    ab.reset()
    return steps


def digest(steps):
    h = hashlib.sha256()
    for res, _ in steps:
        for k in sorted(res):
            h.update(k.encode())
            h.update(np.ascontiguousarray(res[k]).tobytes())
    return h.hexdigest()


def _outs(steps):
    return [r for r, _ in steps]


def _launches(steps):
    return tuple(l for _, l in steps)


@pytest.fixture(scope="module")
def device_runs():
    return {(case, dt): run(case, "device", dt) for case in TCASES for dt in (F64, F32)}


@gpu
@pytest.mark.parametrize("mode", ["device", "pinned", "pageable"])
@pytest.mark.parametrize("case", list(TCASES))
def test_host_transports_keep_the_contract(device_runs, case, mode):
    ref = device_runs[(case, F64)]
    f64 = ref if mode == "device" else run(case, mode, F64)
    f32 = device_runs[(case, F32)] if mode == "device" else run(case, mode, F32)
    _assert_contract(_outs(f32), _outs(ref), (case, mode))
    assert digest(f32) == digest(device_runs[(case, F32)]), (case, mode)
    assert _launches(f32) == _launches(f64), (case, mode, _launches(f32), _launches(f64))
    # the launch table of test_gpu_model_transport.py: at jt == 1 on host arrays, 2 speculative chunks of statistics +
    # init_decide (+ classify) + flux
    assert _launches(f32) == tr.LAUNCHES[case][mode], (case, mode, _launches(f32))


def test_transport_grid_takes_two_speculative_chunks():
    import aerobulk_b200 as ab
    plan = lambda n, kind: ab.lib().aerobulk_gpu_chunk_plan(C.c_longlong(n), kind, (C.c_longlong * 17)())
    assert plan(BIG[0] * BIG[1], 3) >= 2


@gpu
def test_staged_transports_keep_the_contract(device_runs):
    """AEROBULK_GPU_BOUNCE=0 (pageable arrays) and AEROBULK_GPU_ZEROCOPY=0 (pinned arrays) are read once per process."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for name, (mode, env) in {"no-bounce": ("pageable", {"AEROBULK_GPU_BOUNCE": "0"}),
                              "no-zerocopy": ("pinned", {"AEROBULK_GPU_ZEROCOPY": "0"})}.items():
        script = ("import sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]\n"
                  "import numpy as np\n"
                  "import test_gpu_model_f32 as t\n"
                  "for case in t.TCASES:\n"
                  "    for dt in (np.float64, np.float32):\n"
                  f"        s = t.run(case, {mode!r}, dt)\n"
                  "        print('RUN', case, np.dtype(dt).name, t.digest(s), *t._launches(s))\n")
        r = subprocess.run([sys.executable, "-c", script, root, os.path.join(root, "tests")], cwd=root,
                           env={**os.environ, **env}, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (name, r.stderr[-2000:])
        got = {(l.split()[1], l.split()[2]): l.split()[3:] for l in r.stdout.splitlines() if l.startswith("RUN")}
        for case in TCASES:
            g64, g32 = got[(case, "float64")], got[(case, "float32")]
            assert g64[0] == digest(device_runs[(case, F64)]), (name, case, "float64")
            assert g32[0] == digest(device_runs[(case, F32)]), (name, case, "float32")
            assert g32[1:] == g64[1:], (name, case, g32[1:], g64[1:])


@gpu
@pytest.mark.parametrize("case", list(TCASES))
def test_small_grid_transports_keep_the_contract(case):
    ref = run(case, "device", F64, SMALL)
    for mode in ("device", "pageable"):
        f32 = run(case, mode, F32, SMALL)
        _assert_contract(_outs(f32), _outs(ref), (case, mode, "small"))
        assert _launches(f32) == _launches(run(case, mode, F64, SMALL) if mode != "device" else ref), (case, mode)


def _host_session(ab, dtype, ni, nj, nt=2):
    """An NCAR session of nt steps on pageable (ni, nj) arrays of `dtype` (float32-rounded values); the outputs per step."""
    f = synth.fields(ni, nj, seed=707)
    ins = [f[k].astype(F32).astype(dtype, order="F") for k in IN]
    call = ab.aerobulk_model_f32 if dtype is F32 else ab.aerobulk_model
    return [call(jt, nt, "ncar", 2.0, 10.0, *ins, Niter=5) for jt in range(1, nt + 1)]


@gpu
def test_odd_float32_rows_then_smaller_float64_calls(ab):
    """The staging arrays and the pinned slab are grow-only and shared by both element types.  A float32 call on an odd
    number of points sizes their rows; a smaller float64 call that reuses them must find 8-byte aligned rows and give
    the bits of a fresh process.  First pair: below the slab threshold, staged copies throughout.  Second pair: 2 * 65 536
    + 1 floats, then 65 536 doubles (the largest float64 call that fits the same rows): staged with the speculative init
    at jt == 1, the pinned slab at jt == 2."""
    for big, small in (((101, 1), (50, 1)), ((2 * 65536 + 1, 1), (256, 256))):
        ab.reset()
        _host_session(ab, F32, *big)
        got = _host_session(ab, F64, *small)
        again = _host_session(ab, F32, *big)
        ab.reset()
        ref = _host_session(ab, F64, *small)
        ab.reset()
        ref32 = _host_session(ab, F32, *big)
        ab.reset()
        for jt in range(2):
            for k in ref[jt]:
                assert got[jt][k].tobytes() == ref[jt][k].tobytes(), (big, small, jt + 1, k)
                assert again[jt][k].tobytes() == ref32[jt][k].tobytes(), (big, "float32 again", jt + 1, k)


# ---------------------------------------------------------------------------------------------------------------------
# errors
# ---------------------------------------------------------------------------------------------------------------------
def _error_scenario(ab, dtype, what):
    """(code, message, session flags after the error) of one failing call on pageable host arrays of `dtype`."""
    ni, nj = 40, 30
    f = {k: v.astype(F32) for k, v in synth.fields(ni, nj).items()}
    call = ab.aerobulk_model_f32 if dtype is F32 else ab.aerobulk_model
    ins = lambda g: [g[k].astype(dtype, order="F") for k in IN]
    rad = lambda g: dict(rad_sw=g["rad_sw"].astype(dtype, order="F"), rad_lw=g["rad_lw"].astype(dtype, order="F"))
    g = dict(f)
    ab.reset()
    if what == "humidity":
        g["hum_zt"] = (f["hum_zt"] * F32(1000.0) + F32(110.0)).astype(F32)
    elif what == "units":
        g["sst"] = (f["sst"] - F32(273.15)).astype(F32)
    elif what == "tau":
        call(1, 3, "coare3p6", 2.0, 10.0, *ins(f), Niter=7, l_use_skin=True, **rad(f))
        g["U_zu"] = f["U_zu"].copy()
        g["V_zu"] = f["V_zu"].copy()
        g["U_zu"][5, 7], g["V_zu"][5, 7] = 48.0, 0.0          # (ji, jj) = (6, 8)
    with pytest.raises(ab.AerobulkError) as e:
        if what == "tau":
            call(2, 3, "coare3p6", 2.0, 10.0, *ins(g), l_use_skin=True, **rad(g))
        else:
            call(1, 1, "ncar", 2.0, 10.0, *ins(g))
    after = (ab.use_skin(), ab.nb_iter(), ab.humidity_type(), ab.get_state(0, ni * nj) is None)
    ab.reset()
    return e.value.code, e.value.message, after


@gpu
@pytest.mark.parametrize("what", ["humidity", "units", "tau"])
def test_errors_are_the_fp64_errors(ab, what):
    c64, m64, a64 = _error_scenario(ab, F64, what)
    c32, m32, a32 = _error_scenario(ab, F32, what)
    assert (c32, a32) == (c64, a64), (what, c32, c64, a32, a64)
    assert c64 == {"humidity": 5, "units": 4, "tau": 8}[what], (what, c64, m64)
    if what == "tau":   # the magnitude is printed from the float outputs; the point is the same
        num = re.compile(r"=>\s+([0-9.]+) N/m\^2")
        assert abs(float(num.search(m32).group(1)) - float(num.search(m64).group(1))) <= 0.011, (m32, m64)
        m32, m64 = num.sub("", m32), num.sub("", m64)
        assert "At ji, jj = 0006, 0008" in m64, m64
    assert m32 == m64, (what, m32, m64)


# ---------------------------------------------------------------------------------------------------------------------
# multi-GPU split
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_split_over_two_gpus_is_bit_identical(ab):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ni, nj = 1031, 450
    f = {k: v.astype(F32) for k, v in synth.fields(ni, nj, seed=606).items()}
    res = {}
    try:
        for nd in (1, 2):
            ab.reset()
            ab.set_devices(nd)
            steps = []
            for jt in range(1, 4):
                rsw = synth.rad_sw_hour(ni, nj, 10 + 2 * jt).astype(F32, order="F")
                steps.append(ab.aerobulk_model_f32(jt, 3, "coare3p6", 2.0, 10.0, *[f[k] for k in IN], Niter=5,
                                                   l_use_skin=True, rad_sw=rsw, rad_lw=f["rad_lw"]))
            res[nd] = steps
    finally:
        ab.set_devices(1)
        ab.reset()
    for jt, (a, b) in enumerate(zip(res[1], res[2]), start=1):
        for k in a:
            assert a[k].dtype == F32 and a[k].tobytes() == b[k].tobytes(), (jt, k)


# ---------------------------------------------------------------------------------------------------------------------
# oracle sanity check
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("algo", ["coare3p0", "coare3p6", "ncar", "ecmwf", "andreas"])
def test_float_outputs_sit_on_the_oracle(ab, algo):
    """|f32 - oracle| <= half a float ulp + the 1e-10 scaled gate, wherever the FP64 path passes that gate unproven (the
    contract ties every other point to the FP64 path, which test_gpu_kernel_matrix.py gates)."""
    from oracle.oracle import OracleSession
    f = {k: np.ravel(v, order="F").astype(F32) for k, v in synth.fields(200, 60).items()}
    ab.reset()
    got = ab.aerobulk_model_f32(1, 1, algo, 2.0, 10.0, *[f[k] for k in IN], Niter=5)
    ab.reset()
    f64 = ab.aerobulk_model(1, 1, algo, 2.0, 10.0, *[f[k].astype(F64) for k in IN], Niter=5)
    ab.reset()
    ref = OracleSession(threads=8).model(1, 1, algo, 2.0, 10.0, *[f[k].astype(F64) for k in IN], Niter=5)
    gate = pu.worst_per_point(f64, ref) <= pu.TOL
    assert (~gate).sum() <= max(1, pu.OUTLIER_FRACTION * gate.size), (algo, int((~gate).sum()))
    for k in OUT[:5]:
        g, r = got[k], np.asarray(ref[k], dtype=F64)
        bound = 0.5 * np.spacing(np.abs(g)).astype(F64) + pu.TOL * (np.abs(r) + synth.PARITY_SCALE[k])
        err = np.abs(g.astype(F64) - r)
        bad = np.flatnonzero(gate & ~(err <= bound))
        assert bad.size == 0, (algo, k, bad[:5].tolist(), err[bad[:5]].tolist(), bound[bad[:5]].tolist())
