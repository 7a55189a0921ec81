"""Wall time of a jt = Nt = 1 host-array call with PAGEABLE arrays (the plain relink case at the first step of a session):
the copy threads feed the staged pipeline chunk by chunk.  AEROBULK_GPU_HOST_THREADS applies.   usage: python tools/pageable_jt1_probe.py [Ni Nj] [algo] [skin 0/1]"""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import aerobulk_b200 as ab
from aerobulk_b200 import synth
Ni, Nj = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (4320, 2160)
algo = sys.argv[3] if len(sys.argv) > 3 else "ecmwf"
skin = (sys.argv[4] == "1") if len(sys.argv) > 4 else True
f = synth.fields(Ni, Nj)
IN = ("sst", "t_zt", "hum_zt", "U_zu", "V_zu", "slp")
ins = {k: np.array(f[k], order="F") for k in IN + ("rad_sw", "rad_lw")}
outs = {k: np.empty((Ni, Nj), order="F") for k in (("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s") if skin else ("QL", "QH", "Tau_x", "Tau_y", "Evap"))}
ab.set_verbose(False)
kw = dict(l_use_skin=True, rad_sw=ins["rad_sw"], rad_lw=ins["rad_lw"]) if skin else {}
ts = []
for rep in range(6):
    ab.new_session()
    t0 = time.perf_counter()
    ab.aerobulk_model(1, 1, algo, 2., 10., *[ins[k] for k in IN], Niter=5, out=outs, **kw)
    ts.append(time.perf_counter() - t0)
ms = 1e3 * float(np.median(ts[2:]))
nb = (8 + 6 if skin else 6 + 5) * 8 * Ni * Nj
print(f"{algo}{'+skin' if skin else ''} {Ni}x{Nj} pageable jt=1: {ms:8.2f} ms  {Ni * Nj / ms / 1e6:6.3f} Gpt/s  host arrays {nb / 1e9:.2f} GB -> {nb / ms / 1e6:6.1f} GB/s "
      f"(threads {os.environ.get('AEROBULK_GPU_HOST_THREADS', 'default')})")
