"""Solver parity AT SIZE with the time loop's solver settings (VERDICT r1, weak #1).

tests/golden/large_*.npz hold the solution of the UNMODIFIED reference's system (pylamp_stokes.
makeStokesMatrix + SciPy SuperLU as at pylamp2.py:360, plus one refinement step) for analytic C4-type
fields at 513^2 / 1025^2 nodes and for SolCx (viscosity jump 1e6) at 257^2 / 513^2 / 1025^2, sampled on
257 x 257 nodes (oracle/make_golden_large.py; one solve takes minutes to half an hour and 5-30 GB).
The GPU solver runs with EXACTLY bench.py's settings (bench.DEFAULTS: tolerance, extrapolated warm
start over 5 iterates, V(2,2), FGMRES(30), eigenvalue estimates every 8 coefficient updates) through a
sequence of slowly translating fields ending at the fixture's t = 0 -- what consecutive time steps hand
to the solver -- and must match vz, vx and P~ to 1e-8 relative L2 (north_star), or 3x the reference's own
raw-spsolve noise floor where that is larger (SolCx pressure: 1e-6..1e-5, SURVEY App. B).
"""
import numpy as np
import pytest

from oracle.large_fixtures import load as _load

pytestmark = [pytest.mark.gpu]
NSTEPS = 12      # > warm_start history (5) and > lmax_every (8): stale eigenvalue estimates are exercised


def _errors(x, nx, g):
    st = int(g["stride"])
    out = []
    for k, nm in enumerate(("vz", "vx", "p")):
        a = x[k::3].reshape(nx)[::st, ::st].cpu().numpy()
        out.append(float(np.linalg.norm(a - g[nm]) / np.linalg.norm(g[nm])))
    return out


def _check(label, err, g, A):
    floor = [float(g[n + "_floor"]) for n in ("vz", "vx", "p")]
    print(label, "iters", A.iterations, "stats", A.stats, "err(vz,vx,P)", ["%.1e" % e for e in err],
          "reference raw-vs-refined floor", ["%.1e" % f for f in floor])
    for e, f in zip(err, floor):
        assert e <= max(1e-8, 3 * f), (label, err, floor)


@pytest.mark.parametrize("name", ["conv513", "conv1025"])
def test_convection_fields_time_loop_settings(name):
    import torch
    import bench
    from pylamp_b200 import pylamp_stokes as S, setups
    g = _load(name)
    ncell = int(g["ncell"])
    dev = torch.device("cuda")
    work, A = None, None
    for t in range(-NSTEPS, 1):
        nx, L, grid, gridmp, es, en, rho = setups.convection_fields(ncell, t)
        f = [torch.as_tensor(a).to(dev) for a in (es, en, rho)]
        if A is None:
            work = f
            A = S.StokesOperator(nx, grid, *work, [1, 1, 1, 1])
            A.warn_unconverged = False
            for k, v in bench.stokes_params().items():
                A.set_param(k, v)
        else:
            for w, a in zip(work, f):
                w.copy_(a)                    # in place, like the driver's grid fields
            A.set_coeffs(*work)
        x = A.solve(None, rtol=bench.DEFAULTS["stokes_rtol"], maxit=600)
    assert A.stats["status"] == "converged", A.stats      # the bench's tolerance is actually reached
    _check(name, _errors(x, nx, g), g, A)


@pytest.mark.parametrize("name", ["solcx257", "solcx513", "solcx1025"])
def test_solcx_at_size(name):
    import torch
    from pylamp_b200 import pylamp_stokes as S, setups
    g = _load(name)
    n = int(g["ncell"]) + 1
    nx, L, grid, gridmp, es, en, rho = setups.solcx_fields(n)
    dev = torch.device("cuda")
    A = S.StokesOperator(nx, grid, *[torch.as_tensor(a).to(dev) for a in (es, en, rho)], [1, 1, 1, 1])
    A.warn_unconverged = False
    # a single cold solve of a static system: the drop-in's default solver (V(3,3), FGMRES(50), rtol 1e-12) with
    # the 2x2 viscosity coarsening that is exact for a jump on a grid line, as in tests/test_stokes_gpu.py
    A.set_param("coarsen_wide", 0)
    x = A.solve(None, maxit=600)
    _check(name, _errors(x, nx, g), g, A)


def test_solcx_converges_to_the_analytic_solution():
    """BASELINE.json configs[1]: "Stokes solve only vs analytic and vs spsolve" at 256^2-1024^2 cells.  The GPU
    solution of the reference's discrete system against the analytic SolCx-type solution (pylamp_b200/solcx.py;
    pinned on the CPU against the oracle's direct solve in tests/test_solcx_cpu.py): the reference's scheme puts
    the viscosity jump on a node line (the node takes the stiff value), so it converges at first order; the
    errors must halve with the spacing and equal what the reference's own direct solve gives (the fixtures)."""
    import torch
    from pylamp_b200 import pylamp_stokes as S, setups, solcx
    dev = torch.device("cuda")
    errs = {}
    for n in (257, 513, 1025):
        nx, L, grid, gridmp, es, en, rho = setups.solcx_fields(n)
        A = S.StokesOperator(nx, grid, *[torch.as_tensor(a).to(dev) for a in (es, en, rho)], [1, 1, 1, 1])
        A.warn_unconverged = False
        A.set_param("coarsen_wide", 0)
        x = A.solve(None, maxit=600)
        vel, p = S.x2vp(x, nx)
        errs[n] = solcx.errors(nx, grid, gridmp, vel[0].cpu().numpy(), vel[1].cpu().numpy(), p.cpu().numpy(), A.scaling[0])
        print("SolCx %d^2 nodes: iters %d, relative L2 error vs analytic (vz, vx, p) %s" %
              (n, A.iterations, ["%.3e" % e for e in errs[n]]))
        A.close()
    for a, b in ((257, 513), (513, 1025)):
        order = [float(np.log2(ea / eb)) for ea, eb in zip(errs[a], errs[b])]
        print("order %d -> %d:" % (a, b), ["%.2f" % o for o in order])
        assert all(0.9 < o < 1.2 for o in order), order
    assert max(errs[1025]) < 8e-3
