"""Solver-parity fixtures at sizes where one direct solve costs minutes to half an hour (needs the original
PyLamp; run once, results committed as strided samples under tests/golden/large_*_0.npz, _1.npz).

    python oracle/make_golden_large.py conv513 solcx513 conv1025 solcx1025

For every case the UNMODIFIED reference assembles the system (pylamp_stokes.makeStokesMatrix,
imported through oracle/ref_shims.py from PYLAMP_REFERENCE_DIR) and SciPy's SuperLU solves it the way
pylamp2.py:360 does; one fp64 refinement step on top is the ground truth (SURVEY.md 8c).  The inputs
are analytic (pylamp_b200/setups.py: `convection_fields(ncell, t=0)`, `solcx_fields(n)`), so only
the solution has to be stored: every `stride`-th node in both directions (257 x 257 samples) of vz,
vx and P~, the same samples of the raw spsolve answer's distance (the oracle's own noise floor) and
the residual norms.  Test infrastructure only.
"""
import os
import sys
import time

import numpy as np
import scipy.sparse
import scipy.sparse.linalg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shims  # noqa: E402
from oracle.large_fixtures import save  # noqa: E402
from pylamp_b200 import setups  # noqa: E402

CASES = {"conv513": ("conv", 512), "conv1025": ("conv", 1024), "solcx513": ("solcx", 512),
         "solcx1025": ("solcx", 1024), "conv257": ("conv", 256), "solcx257": ("solcx", 256)}


def fields(kind, ncell):
    if kind == "conv":
        nx, L, grid, gridmp, etas, etan, rho = setups.convection_fields(ncell, t=0.0)
    else:
        nx, L, grid, gridmp, etas, etan, rho = setups.solcx_fields(ncell + 1)
    return nx, L, grid, etas, etan, rho


def make(name):
    kind, ncell = CASES[name]
    rt, rs, rd, rc = ref_shims.load()
    nx, L, grid, etas, etan, rho = fields(kind, ncell)
    t0 = time.perf_counter()
    A, rhs = rs.makeStokesMatrix(nx, grid, etas, etan, rho, [1, 1, 1, 1])
    t_asm = time.perf_counter() - t0
    A = scipy.sparse.csc_matrix(A)
    t0 = time.perf_counter()
    lu = scipy.sparse.linalg.splu(A)            # what spsolve does (SuperLU, COLAMD), factors kept
    x_raw = lu.solve(rhs)
    t_solve = time.perf_counter() - t0
    x = x_raw + lu.solve(rhs - A @ x_raw)
    del lu
    res_raw = np.linalg.norm(rhs - A @ x_raw) / np.linalg.norm(rhs)
    res_ref = np.linalg.norm(rhs - A @ x) / np.linalg.norm(rhs)
    stride = max(1, ncell // 256)
    comp = lambda v, k: v[k::3].reshape(nx)[::stride, ::stride].copy()
    out = {"ncell": ncell, "kind": kind, "stride": stride, "res_raw": res_raw, "res_refined": res_ref,
           "t_assemble_s": t_asm, "t_splu_solve_s": t_solve}
    for k, nm in enumerate(("vz", "vx", "p")):
        out[nm] = comp(x, k)
        full, raw = x[k::3], x_raw[k::3]
        out[nm + "_norm"] = np.linalg.norm(full)
        out[nm + "_floor"] = np.linalg.norm(raw - full) / np.linalg.norm(full)   # raw spsolve <-> refined, all nodes
    save(name, out)
    print(name, "nx", nx, "assemble %.1f s, splu+solve %.1f s" % (t_asm, t_solve), "residual raw %.2e refined %.2e" %
          (res_raw, res_ref), "floor", [float("%.2e" % out[n + "_floor"]) for n in ("vz", "vx", "p")], flush=True)


if __name__ == "__main__":
    for nm in sys.argv[1:]:
        make(nm)
