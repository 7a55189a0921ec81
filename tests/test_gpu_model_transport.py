"""How the caller's arrays reach the kernel must change neither what aerobulk_gpu_model computes nor how many kernels each
call launches.

model_impl (aerobulk_b200/csrc/ab_api.cu) takes one of the four paths of its Transport per call: the caller's device
pointers; the device aliases of pinned arrays (zero-copy, jt > 1); pageable arrays through the library's pinned slab
(jt > 1, from 65 536 points up); staged copies.  At jt == 1 the staged pipeline runs with the speculative AEROBULK_INIT,
fed from the slab when the arrays are pageable.  One session, jt = 1..3 of Nt = 3 with the warm-layer state carried on the device, runs through:
  - CUDA tensors (aerobulk_gpu_model_device);
  - pinned torch tensors: staged with the speculative AEROBULK_INIT at jt == 1, zero-copy after;
  - pageable numpy arrays: the slab-fed speculative pipeline at jt == 1, the slab after;
  - pageable numpy arrays in a process with AEROBULK_GPU_BOUNCE=0: staged kind-1 chunks after jt == 1;
  - pinned torch tensors in a process with AEROBULK_GPU_ZEROCOPY=0: staged throughout.
The knobs are read once per process, so the last two run in subprocesses and are compared by hash.  The grid, 1031 x 450 =
463 950 points, is no multiple of 2048 and gives 2 speculative chunks, 2 staged (kind-1) chunks and 3 slab chunks.  A
300 x 200 grid, below the slab threshold, runs through pageable and device arrays.  Every output array starts filled with a
sentinel, and every point of it must be written."""
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from aerobulk_b200 import synth

pytestmark = pytest.mark.gpu
NT = 3
SENTINEL = 7.25
BIG, SMALL = (1031, 450), (300, 200)
IN = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
OUT = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")
# coare3p6 with skin and radiation sorts its points where it may; ncar never sorts, and without radiation it has no T_s
CASES = {"coare3p6-skin": ("coare3p6", True), "ncar": ("ncar", False)}

# Kernel launches of the calls jt = 1, 2, 3.  Device pointers: statistics (3 kernels) + init_decide, then one chunk of
# classify (when sorting) + flux.  Host arrays at jt == 1: 2 speculative chunks of statistics + init_decide + classify +
# flux.  jt > 1: pinned arrays one zero-copy flux launch; pageable arrays one flux launch per slab chunk (3); staged
# copies 2 chunks of classify + flux.  Zero-copy launches never sort.
LAUNCHES = {
    "coare3p6-skin": {"device": (6, 2, 2), "pinned": (12, 1, 1), "pageable": (12, 3, 3), "no-bounce": (12, 4, 4),
                      "no-zerocopy": (12, 4, 4)},
    "ncar": {"device": (5, 1, 1), "pinned": (10, 1, 1), "pageable": (10, 3, 3), "no-bounce": (10, 2, 2),
             "no-zerocopy": (10, 2, 2)},
}
# 60 000 points: one chunk of every kind.  jt == 1 on host arrays takes the statistics of the whole field, judges them on
# the host and launches one chunk; jt > 1 is one staged chunk.
SMALL_LAUNCHES = {"coare3p6-skin": {"device": (6, 2, 2), "pageable": (5, 2, 2)},
                  "ncar": {"device": (5, 1, 1), "pageable": (4, 1, 1)}}
# the same calls in a process with the knob set
SUBPROCESS = {"no-bounce": ("pageable", {"AEROBULK_GPU_BOUNCE": "0"}), "no-zerocopy": ("pinned", {"AEROBULK_GPU_ZEROCOPY": "0"})}


def run(case, mode, shape=BIG):
    """The session of `case` with the caller's arrays in `mode` ("pageable" numpy, "pinned" torch tensors or "device" CUDA
    tensors): per call, the outputs (and, until jt == Nt releases it, the warm-layer state) as numpy arrays, and the
    number of kernel launches."""
    import aerobulk_b200 as ab
    algo, skin = CASES[case]
    ni, nj = shape
    n = ni * nj
    flat = lambda a: np.ravel(a, order="F").astype(np.float64)
    if mode == "pageable":
        mk = lambda a: a.copy()
        full = lambda: np.full(n, SENTINEL)
        ptr = lambda x: None if x is None else x.ctypes.data
        back = lambda x: x.copy()
    else:
        import torch
        if mode == "pinned":
            mk = lambda a: torch.from_numpy(a.copy()).pin_memory()
            full = lambda: torch.full((n,), SENTINEL, dtype=torch.float64).pin_memory()
        else:
            mk = lambda a: torch.from_numpy(a).cuda()
            full = lambda: torch.full((n,), SENTINEL, dtype=torch.float64, device="cuda")
        ptr = lambda x: None if x is None else x.data_ptr()
        back = lambda x: x.cpu().numpy().copy()
    f = synth.fields(ni, nj, seed=606)
    ins = {k: mk(flat(f[k])) for k in IN + (("rad_lw",) if skin else ())}
    outs = OUT if skin else OUT[:5]
    L = ab.lib()
    entry = L.aerobulk_gpu_model_device if mode == "device" else L.aerobulk_gpu_model
    ab.reset()
    ab.set_sort(1)          # the automatic sort policy, and banners off: the settings the launch tables assume
    ab.set_verbose(False)
    steps = []
    for jt in range(1, NT + 1):
        rsw = mk(flat(synth.rad_sw_hour(ni, nj, 10 + 2 * jt))) if skin else None
        o = {k: full() for k in outs}
        if mode == "device":
            torch.cuda.synchronize()   # the inputs and sentinels are written on torch's stream
        L.aerobulk_gpu_reset_launch_count()
        rc = entry(jt, NT, algo.encode(), 2.0, 10.0, ni, nj, *[ptr(ins[k]) for k in IN], *[ptr(o[k]) for k in OUT[:5]],
                   C.byref(C.c_int(5)), C.byref(C.c_int(1)) if skin else None, ptr(rsw), ptr(ins.get("rad_lw")),
                   ptr(o.get("T_s")))
        if mode == "device":
            torch.cuda.synchronize()   # jt < Nt on device pointers is asynchronous
        assert rc == 0, (case, mode, jt, rc, ab.last_error())
        launches = L.aerobulk_gpu_launch_count()
        res = {k: back(v) for k, v in o.items()}
        for k, v in res.items():
            assert not np.any(v == SENTINEL), (case, mode, jt, k, "not written everywhere")
        if skin and jt < NT:
            for w in range(4):
                res[f"state{w}"] = ab.get_state(w, n)
                assert res[f"state{w}"] is not None, (case, mode, jt, w)
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


def _same(got, ref, what):
    for jt, ((g, _), (r, _)) in enumerate(zip(got, ref), start=1):
        assert set(g) == set(r), (what, jt)
        for k in g:
            assert g[k].tobytes() == r[k].tobytes(), (what, jt, k)


@pytest.fixture(scope="module")
def device():
    return {case: run(case, "device") for case in CASES}


@pytest.mark.parametrize("case", list(CASES))
def test_device_pointers_launch_as_planned(device, case):
    assert tuple(l for _, l in device[case]) == LAUNCHES[case]["device"]


@pytest.mark.parametrize("mode", ["pinned", "pageable"])
@pytest.mark.parametrize("case", list(CASES))
def test_host_arrays_give_the_same_bits(device, case, mode):
    got = run(case, mode)
    _same(got, device[case], (case, mode))
    assert tuple(l for _, l in got) == LAUNCHES[case][mode]


def test_staged_copies_give_the_same_bits(device):
    """AEROBULK_GPU_BOUNCE=0 and AEROBULK_GPU_ZEROCOPY=0 are read once per process: these sessions run in subprocesses."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for name, (mode, env) in SUBPROCESS.items():
        script = ("import sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]\n"
                  "import test_gpu_model_transport as t\n"
                  "for case in t.CASES:\n"
                  f"    s = t.run(case, {mode!r})\n"
                  "    print('RUN', case, t.digest(s), *[l for _, l in s])\n")
        r = subprocess.run([sys.executable, "-c", script, root, os.path.join(root, "tests")], cwd=root,
                           env={**os.environ, **env}, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (name, r.stderr[-2000:])
        got = {l.split()[1]: l.split()[2:] for l in r.stdout.splitlines() if l.startswith("RUN")}
        assert set(got) == set(CASES), (name, r.stdout[-2000:])
        for case in CASES:
            assert got[case][0] == digest(device[case]), (name, case)
            assert tuple(int(x) for x in got[case][1:]) == LAUNCHES[case][name], (name, case, got[case])


@pytest.mark.parametrize("case", list(CASES))
def test_small_grid_gives_the_same_bits(case):
    dev, pag = run(case, "device", SMALL), run(case, "pageable", SMALL)
    _same(pag, dev, (case, "small"))
    assert tuple(l for _, l in dev) == SMALL_LAUNCHES[case]["device"]
    assert tuple(l for _, l in pag) == SMALL_LAUNCHES[case]["pageable"]


def test_chunk_plans_of_the_grids():
    """The grids above give the chunk counts the launch tables assume."""
    import aerobulk_b200 as ab
    L = ab.lib()
    plan = lambda n, kind: L.aerobulk_gpu_chunk_plan(C.c_longlong(n), kind, (C.c_longlong * 17)())
    n = BIG[0] * BIG[1]
    assert n % 2048 and (plan(n, 3), plan(n, 1), plan(n, 2)) == (2, 2, 3)
    assert all(plan(SMALL[0] * SMALL[1], kind) == 1 for kind in (1, 2, 3))
