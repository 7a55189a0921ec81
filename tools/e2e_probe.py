"""Per-call wall time of the host-array API (pinned buffers) for the bench workload."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import aerobulk_b200 as ab
from aerobulk_b200 import synth
NI, NJ, NT = 1440, 720, 24
n = NI * NJ
IN = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
OUT = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")
f = synth.fields(NI, NJ)
def pinned(a):
    t = torch.empty(n, dtype=torch.float64).pin_memory()
    t.numpy()[:] = np.ravel(a, order="F")
    return t
if os.environ.get("E2E_SLAB", "1") == "1":
    islab = torch.empty((7, n), dtype=torch.float64).pin_memory()
    host = {}
    for i, k in enumerate(IN + ("rad_lw",)):
        islab[i].numpy()[:] = np.ravel(f[k], order="F")
        host[k] = islab[i]
    host["rad_sw"] = pinned(f["rad_sw"])
    oslab = torch.empty((6, n), dtype=torch.float64).pin_memory()
    hout = {k: oslab[i] for i, k in enumerate(OUT)}
else:
    host = {k: pinned(f[k]) for k in IN + ("rad_lw", "rad_sw")}
    hout = {k: torch.empty(n, dtype=torch.float64).pin_memory() for k in OUT}
np_in = {k: v.numpy().reshape((NI, NJ), order="F") for k, v in host.items()}
np_out = {k: v.numpy().reshape((NI, NJ), order="F") for k, v in hout.items()}
ab.reset(); ab.set_verbose(False)
if os.environ.get("E2E_SORT"):
    ab.set_sort(int(os.environ["E2E_SORT"]))
best = []
for s in range(4):
    ts = []
    for jt in range(1, NT + 1):
        t0 = time.perf_counter()
        ab.aerobulk_model(jt, NT, "coare3p6", 2., 10., *[np_in[k] for k in IN], Niter=5, l_use_skin=True,
                          rad_sw=np_in["rad_sw"], rad_lw=np_in["rad_lw"], out=np_out)
        ts.append((time.perf_counter() - t0) * 1e3)
    best.append(np.median(ts[2:-1]))
    if os.environ.get("E2E_SORT"):
        ab.set_sort(int(os.environ["E2E_SORT"]))
print(f"slab={os.environ.get('E2E_SLAB','1')}: median per call {min(best):.3f} ms  ({n / min(best) / 1e3:.0f} Mpt/s)")
