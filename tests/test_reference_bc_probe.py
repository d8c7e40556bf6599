"""Which wall types of the reference's Stokes assembly (pylamp_stokes.py:177-189, :257-276, :303-321, :525-551)
have a solution a drop-in can be held to (SURVEY.md §8f-4).  The probe runs the unmodified reference (only where
PYLAMP_REFERENCE_DIR names a checkout of the original PyLamp):
  * FLOWTHRU|FREESLIP (= 5) on the x = 0 wall: a REGULAR system (the anchor moves to cell (nz/2, 0)) -- supported by
    the drop-in since round 2 (tests/test_flowthru_gpu.py; round 1 had wrongly lumped it with the singular ones);
  * 5 on the x = L wall: the anchor lands on the ghost pressure column, the constant pressure stays undetermined
    (rank n-1, consistent); with 5 on both x-walls rank n-2 -- no unique reference pressure: refused;
  * pure FLOWTHRU (= 4), CYCLIC, NOSLIP x-walls: rows left empty, rank-deficient, `spsolve` returns NaN: refused
    (tests/test_stokes_gpu.py::test_unsupported_bcs_raise)."""
import warnings

import numpy as np
import pytest

from oracle import ref_shims

pytestmark = pytest.mark.skipif(not ref_shims.available(), reason="needs a checkout of the original PyLamp in PYLAMP_REFERENCE_DIR")

FREESLIP, NOSLIP, CYCLIC, FLOWTHRU = 1, 0, 2, 4


def _assemble(bc):
    import scipy.sparse as sp
    _, rs, _, _ = ref_shims.load()
    nx, L = [11, 9], [1.0, 0.8]
    grid = [np.linspace(0, L[i], nx[i]) for i in range(2)]
    rng = np.random.default_rng(0)
    etas, etan, rho = 10 ** rng.uniform(0, 2, nx), 10 ** rng.uniform(0, 2, nx), rng.uniform(1, 2, nx)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, _ = rs.makeStokesMatrix(nx, grid, etas, etan, rho, bc)
    A = sp.csr_matrix(A)
    empty = int((np.diff(A.indptr) == 0).sum())
    return A.shape[0], empty, int(np.linalg.matrix_rank(A.toarray()))


@pytest.mark.parametrize("bc", [[FREESLIP] * 4, [NOSLIP, FREESLIP, NOSLIP, FREESLIP],
                                [FREESLIP, FLOWTHRU | FREESLIP, FREESLIP, FREESLIP],
                                [NOSLIP, FLOWTHRU | FREESLIP, NOSLIP, FREESLIP]])
def test_supported_walls_give_regular_systems(bc):
    n, empty, rank = _assemble(bc)
    assert empty == 0 and rank == n


@pytest.mark.parametrize("bc", [[FREESLIP, CYCLIC, FREESLIP, CYCLIC],          # cyclic in x
                                [CYCLIC, FREESLIP, CYCLIC, FREESLIP],          # cyclic in z
                                [FREESLIP, FLOWTHRU, FREESLIP, FREESLIP],      # inflow wall at x=0
                                [FREESLIP, FREESLIP, FREESLIP, FLOWTHRU],
                                [FREESLIP, FLOWTHRU, FREESLIP, FLOWTHRU],
                                [FREESLIP, FLOWTHRU | FREESLIP, FREESLIP, FLOWTHRU | FREESLIP],
                                [FREESLIP, FREESLIP, FREESLIP, FLOWTHRU | FREESLIP],   # anchor on the ghost column
                                [FREESLIP, NOSLIP, FREESLIP, NOSLIP]])         # quirk 4: no-slip x-walls
def test_cyclic_flowthru_and_noslip_x_walls_are_singular_in_the_reference(bc):
    n, empty, rank = _assemble(bc)
    assert rank < n, (bc, empty, rank, n)
