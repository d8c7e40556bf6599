"""INTEGRATION.md 3: the UNMODIFIED reference driver pylamp2.py executed on top of the
drop-in modules (pylamp_b200.launcher: module registration + the spsolve/csc_matrix rebinding), and its
np.savez payload compared with the golden dump of the same script run on the reference's own modules
(tests/golden/c1_noinject.npz, oracle/make_golden.py).  The script is the original PyLamp's and not part of this
repository: the test runs where PYLAMP_REFERENCE_DIR names a checkout of it and is skipped elsewhere (nothing can
stand in for the reference's script)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle.ref_shims import REFERENCE_DIR as REF

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, "pylamp2.py"))),
                                 reason="needs a checkout of the original PyLamp in PYLAMP_REFERENCE_DIR")]


def test_unmodified_pylamp2_on_dropin_modules_matches_golden():
    from pylamp_b200 import launcher
    gold = np.load(os.path.join(GOLDEN, "c1_noinject.npz"))
    nsteps = 2
    # the configuration of the golden run (tracdens_min = 0: the marker injection draws np.random positions)
    out = launcher.run(os.path.join(REF, "pylamp2.py"), nsteps=nsteps, substitutions=[("tracdens_min = 25 ", "tracdens_min = 0 ")],
                       seed=int(gold["seed"]), quiet=True)
    assert len(out) == nsteps
    stride = int(gold["stride"])
    rel = lambda a, b: np.linalg.norm(a - b) / np.linalg.norm(b)
    for it, (grid, tracs) in enumerate(out):
        assert set(grid) == {"gridz", "gridx", "velz", "velx", "pres", "rho", "temp", "tstep", "time"}
        assert set(tracs) == {"tr_x", "tr_f", "tr_v"}
        e = {k: rel(grid[k], gold["s%d_%s" % (it, k)]) for k in ("velz", "velx", "pres", "rho")}
        print("step", it + 1, {k: "%.1e" % v for k, v in e.items()})
        # C1 (viscosity contrast 1e10): the reference's own direct solve is reproducible to ~5e-6 (DESIGN.md 2)
        assert e["rho"] < 1e-12 and e["velz"] < 3e-5 and e["velx"] < 3e-5, e
        assert tracs["tr_x"].shape[0] == int(gold["s%d_ntrac" % it])
        assert np.allclose(tracs["tr_x"][::stride], gold["s%d_tr_x" % it], rtol=1e-9, atol=0)
