"""Storage of the solver-parity fixtures tests/golden/large_<case>_0.npz / _1.npz (written by
oracle/make_golden_large.py, read by tests/test_stokes_large_gpu.py).  Each fixture is two files, the first
and second half of the rows of the sampled fields, so that no file exceeds 1 MB; the scalars go with the
first half.  NumPy only."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
FIELDS = ("vz", "vx", "p")


def _paths(name):
    return [os.path.join(GOLDEN, "large_%s_%d.npz" % (name, i)) for i in (0, 1)]


def save(name, out):
    h = (out["vz"].shape[0] + 1) // 2
    p0, p1 = _paths(name)
    np.savez_compressed(p0, **{k: (v[:h] if k in FIELDS else v) for k, v in out.items()})
    np.savez_compressed(p1, **{k: out[k][h:] for k in FIELDS})


def load(name):
    """The fixture `name` (e.g. "conv513") as a dict, halves joined; raises if it is missing."""
    p0, p1 = _paths(name)
    with np.load(p0) as a, np.load(p1) as b:
        g = {k: a[k] for k in a.files}
        for k in FIELDS:
            g[k] = np.concatenate([a[k], b[k]])
    return g
