"""Where does the Stokes solve's scaled residual really stop, and what error does a given relres mean?

  python scripts/solver_floor_study.py <ncell> [nsteps] [rtol ...]

Steps the analytic C4-type fields (setups.convection_fields) through t = -nsteps..0 with the time-loop
solver settings of bench.py (warm start by extrapolation, eigenvalue estimates every 8 steps), then
  (a) for every rtol given: re-runs the sequence and reports iterations / relres / status of the last solve
      and, when the fixture tests/golden/large_conv<ncell+1>_*.npz exists, its error against the reference's direct solve;
  (b) one cold solve at rtol 1e-14 with PLB_DEBUG_FGMRES=1 to show the true-residual history (the fp64 floor).
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import large_fixtures  # noqa: E402
from pylamp_b200 import pylamp_stokes as S, setups  # noqa: E402

ncell = int(sys.argv[1])
nsteps = int(sys.argv[2]) if len(sys.argv) > 2 else 12
rtols = [float(v) for v in sys.argv[3:]] or [1e-9, 1e-10, 1e-11, 1e-12]
try:
    gold = large_fixtures.load("conv%d" % (ncell + 1))
except FileNotFoundError:
    gold = None
dev = torch.device("cuda")


def fields(t):
    nx, L, grid, gridmp, es, en, rho = setups.convection_fields(ncell, t)
    return nx, grid, [torch.as_tensor(a).to(dev) for a in (es, en, rho)]


def errors(x, nx):
    if gold is None:
        return None
    st = int(gold["stride"])
    out = []
    for k, nm in enumerate(("vz", "vx", "p")):
        a = x[k::3].reshape(nx)[::st, ::st].cpu().numpy()
        out.append(float(np.linalg.norm(a - gold[nm]) / np.linalg.norm(gold[nm])))
    return out


cache = {t: fields(t) for t in range(-nsteps, 1)}
for rtol in rtols:
    nx, grid, f = cache[-nsteps]
    work = [a.clone() for a in f]
    A = S.StokesOperator(nx, grid, *work, [1, 1, 1, 1])
    A.warn_unconverged = False
    for k, v in bench.stokes_params().items():
        A.set_param(k, v)
    log = []
    for t in range(-nsteps, 1):
        for w, a in zip(work, cache[t][2]):
            w.copy_(a)                       # in place, like the driver's grid fields
        A.set_coeffs(*work)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x = A.solve(None, rtol=rtol, maxit=600, raise_on_fail=False)
        torch.cuda.synchronize()
        st = A.stats
        log.append((st["iterations"], "%.1e" % st["relres"], st["status"][:4], "%.0fms" % (1e3 * (time.perf_counter() - t0))))
    print("ncell %d rtol %.0e: per-step (iters, relres, status, ms):" % (ncell, rtol), log[0], "...", log[-3:], flush=True)
    print("   last solve:", A.stats, "err(vz,vx,p) vs direct solve:", errors(x, nx), flush=True)
    A.close()

os.environ["PLB_DEBUG_FGMRES"] = "1"
nx, grid, f = cache[0]
A = S.StokesOperator(nx, grid, *f, [1, 1, 1, 1])
A.warn_unconverged = False
for k, v in bench.stokes_params().items():
    A.set_param(k, v)
A.set_param("warm_start", 0)
x = A.solve(None, rtol=1e-14, maxit=300, raise_on_fail=False)
print("cold solve to 1e-14:", A.stats, "err:", errors(x, nx), flush=True)
