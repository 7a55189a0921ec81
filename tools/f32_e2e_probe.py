"""aerobulk_model on float32 fields against float64, end to end and device-resident, in one process.

    python tools/f32_e2e_probe.py [--grid 4320x2160] [--reps 5] [--steps 8]

For COARE 3.6 + skin and for NCAR, on a grid far larger than L2: per call wall time of jt > 1 host-array calls, pinned
(zero-copy) and pageable (the copy threads' pinned slab), FP64 and FP32 alternating session by session; then the
flux-kernel time of device-resident calls (CUDA events around each flux launch, aerobulk_gpu_set_kernel_timing).  Every
shape is warmed up first.  Reports medians and the min..max of the per-session medians, in Gpt/s and ms per call, with
the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import aerobulk_b200 as ab  # noqa: E402
from aerobulk_b200 import synth  # noqa: E402

IN = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
OUT = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")
CASES = {"coare3p6+skin": ("coare3p6", True), "ncar": ("ncar", False)}


def card() -> str:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def arrays(f, dtype, mode, skin):
    """Inputs (rad_sw per step) and outputs as numpy (Ni, Nj) Fortran arrays; pinned ones are views of pinned tensors."""
    shape = f["sst"].shape
    n = f["sst"].size
    tdt = torch.float32 if dtype == np.float32 else torch.float64

    def mk(a=None):
        if mode == "pinned":
            t = torch.empty(n, dtype=tdt).pin_memory()
            x = t.numpy().reshape(shape, order="F")
            keep.append(t)
        else:
            x = np.empty(shape, dtype=dtype, order="F")
        if a is not None:
            x[...] = a
        return x

    keep = []
    ins = {k: mk(f[k]) for k in IN + (("rad_lw", "rad_sw") if skin else ())}
    outs = {k: mk() for k in (OUT if skin else OUT[:5])}
    return ins, outs, keep


def host_session(algo, skin, ins, outs, dtype, steps):
    """jt = 1 .. steps + 2 of one session; wall time [ms] of the jt > 1 calls but the last (which also frees the state)."""
    call = ab.aerobulk_model_f32 if dtype == np.float32 else ab.aerobulk_model
    kw = dict(Niter=5)
    if skin:
        kw.update(l_use_skin=True, rad_sw=ins["rad_sw"], rad_lw=ins["rad_lw"])
    nt = steps + 2
    ab.reset()
    ab.set_verbose(False)
    ts = []
    for jt in range(1, nt + 1):
        t0 = time.perf_counter()
        call(jt, nt, algo, 2.0, 10.0, *[ins[k] for k in IN], out=outs, **kw)
        if 1 < jt < nt:
            ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def device_session(algo, skin, f, dtype, steps):
    """Flux-kernel time [ms] (median over jt > 1) of device-resident calls."""
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    n = f["sst"].size
    d = {k: torch.from_numpy(np.ravel(f[k], order="F").astype(dtype)).cuda() for k in IN + ("rad_sw", "rad_lw")}
    out = {k: torch.empty(n, dtype=tdt, device="cuda") for k in (OUT if skin else OUT[:5])}
    call = ab.aerobulk_model_device_f32 if dtype == np.float32 else ab.aerobulk_model_device
    kw = dict(Niter=5)
    if skin:
        kw.update(l_use_skin=True, rad_sw=d["rad_sw"], rad_lw=d["rad_lw"])
    nt = steps + 2
    ab.reset()
    ab.set_verbose(False)
    times = []
    for jt in range(1, nt + 1):
        ab.set_kernel_timing(jt > 1)
        call(jt, nt, algo, 2.0, 10.0, *[d[k] for k in IN], out=out, **kw)
        ab.synchronize()
        if jt > 1:
            times.extend(ab.kernel_times().tolist())
    ab.set_kernel_timing(False)
    ab.reset()
    return float(np.median(times))


def report(label, n, per_rep):
    med = float(np.median(per_rep))
    lo, hi = min(per_rep), max(per_rep)
    print(f"  {label:34s} {med:8.3f} ms  [{lo:.3f} .. {hi:.3f}]  {n / med / 1e6:6.3f} Gpt/s", flush=True)
    return med


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", default="4320x2160")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=8)
    a = ap.parse_args()
    ni, nj = (int(v) for v in a.grid.split("x"))
    n = ni * nj
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: nothing is measured")
    print(f"card: {card()}")
    print(f"grid {ni}x{nj} = {n} points; {a.reps} sessions per entry, {a.steps} timed jt > 1 calls each, FP64 and FP32 "
          "alternating; median [min .. max of the session medians]", flush=True)
    f64 = synth.fields(ni, nj)
    f64 = {k: v.astype(np.float32).astype(np.float64, order="F") for k, v in f64.items()}   # the same values in both
    f32 = {k: v.astype(np.float32, order="F") for k, v in f64.items()}
    fields = {np.float64: f64, np.float32: f32}
    for name, (algo, skin) in CASES.items():
        print(f"{name}:", flush=True)
        res = {}
        for mode in ("pinned", "pageable"):
            bufs = {dt: arrays(fields[dt], dt, mode, skin) for dt in (np.float64, np.float32)}
            for dt in bufs:   # warm-up of every shape and path
                host_session(algo, skin, bufs[dt][0], bufs[dt][1], dt, 2)
            per = {np.float64: [], np.float32: []}
            for _ in range(a.reps):
                for dt in (np.float64, np.float32):
                    per[dt].append(host_session(algo, skin, bufs[dt][0], bufs[dt][1], dt, a.steps))
            for dt in (np.float64, np.float32):
                res[(mode, dt)] = report(f"end to end, {mode}, {np.dtype(dt).name}", n, per[dt])
            print(f"  {'':34s} FP32 / FP64 speed-up {res[(mode, np.float64)] / res[(mode, np.float32)]:.2f}x", flush=True)
            del bufs
        for dt in (np.float64, np.float32):
            device_session(algo, skin, fields[dt], dt, 2)
        per = {np.float64: [], np.float32: []}
        for _ in range(a.reps):
            for dt in (np.float64, np.float32):
                per[dt].append(device_session(algo, skin, fields[dt], dt, a.steps))
        for dt in (np.float64, np.float32):
            report(f"flux kernel, device, {np.dtype(dt).name}", n, per[dt])
    print(f"card: {card()}")


if __name__ == "__main__":
    main()
