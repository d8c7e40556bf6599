"""Import the UNMODIFIED reference -- test infrastructure only.

Only usable where the environment variable ``PYLAMP_REFERENCE_DIR`` names a checkout of the
original PyLamp (the repository does not contain it).  Used by ``oracle/make_golden.py`` and
``oracle/make_golden_large.py`` to generate ``tests/golden/*.npz``, and by
``tests/test_reference_bc_probe.py`` and ``tests/test_launcher_gpu.py``, which skip when the
reference is absent.

Three non-invasive shims (SURVEY.md Appendix A), none of which touches a reference file:
  1. ``pylamp_trac`` passes a *list* as a multi-axis index to ``np.add.at``
     (pylamp_trac.py:257-298), which NumPy >= 1.23 rejects; the module's ``np`` binding is
     replaced by a proxy that converts the list to a tuple.
  2. a fake single-rank ``mpi4py.MPI`` (pylamp2.py:3, 30-32, 122, 446, 454, 554-555).
  3. ``time.clock`` (removed in Python 3.8) aliased to ``time.process_time``
     (pylamp_tool.py:12, 16).
"""
import os
import sys
import time
import types

import numpy as _np

REFERENCE_DIR = os.environ.get("PYLAMP_REFERENCE_DIR", "")


def available():
    return bool(REFERENCE_DIR) and os.path.isfile(os.path.join(REFERENCE_DIR, "pylamp_trac.py"))


class _Add:
    def __call__(self, *a, **k):
        return _np.add(*a, **k)

    def at(self, a, idx, v):
        return _np.add.at(a, tuple(idx) if isinstance(idx, list) else idx, v)


class _NumpyProxy:
    add = _Add()

    def __getattr__(self, name):
        return getattr(_np, name)


def _install_fake_mpi():
    if "mpi4py" in sys.modules:
        return
    pkg = types.ModuleType("mpi4py")
    mpi = types.ModuleType("mpi4py.MPI")

    class _Comm:
        def Get_rank(self):
            return 0

        def Get_size(self):
            return 1

        def Bcast(self, buf, root=0):
            return None

        def Allreduce(self, send, recv, op=None):
            recv[0][...] = send[0]

    mpi.COMM_WORLD = _Comm()
    mpi.DOUBLE = "DOUBLE"
    mpi.SUM = "SUM"
    pkg.MPI = mpi
    sys.modules["mpi4py"] = pkg
    sys.modules["mpi4py.MPI"] = mpi


def load():
    """Returns (pylamp_trac, pylamp_stokes, pylamp_diff, pylamp_const) of the reference."""
    if not available():
        raise RuntimeError("reference not present at %s" % REFERENCE_DIR)
    _install_fake_mpi()
    if not hasattr(time, "clock"):
        time.clock = time.process_time
    if REFERENCE_DIR not in sys.path:
        sys.path.insert(0, REFERENCE_DIR)
    import pylamp_const
    import pylamp_diff
    import pylamp_stokes
    import pylamp_trac
    for m in (pylamp_trac, pylamp_stokes, pylamp_diff, pylamp_const):
        assert os.path.dirname(os.path.abspath(m.__file__)) == os.path.abspath(REFERENCE_DIR), m
    pylamp_trac.np = _NumpyProxy()
    return pylamp_trac, pylamp_stokes, pylamp_diff, pylamp_const


def run_driver(nsteps, seed, substitutions=(), workdir=None, quiet=True):
    """Execute the reference driver ``pylamp2.py`` for ``nsteps`` steps and return what it
    would have written with ``np.savez`` (a list of (griddata dict, tracs dict) per step).

    ``substitutions`` is a list of (old, new) source-text replacements applied to the
    in-memory copy of pylamp2.py (the reference has no config file: "edit the source",
    README:32-34); each ``old`` must occur exactly once.
    """
    import contextlib
    import io
    import tempfile
    load()
    src = open(os.path.join(REFERENCE_DIR, "pylamp2.py")).read()
    for old, new in substitutions:
        assert src.count(old) == 1, (old, src.count(old))
        src = src.replace(old, new)
    captured = []

    class _Stop(Exception):
        pass

    real_savez = _np.savez

    def fake_savez(fname, **kw):
        kw = {k: _np.array(v, copy=True) for k, v in kw.items()}
        if "griddata" in fname:
            captured.append([kw, None])
        else:
            captured[-1][1] = kw
            if len(captured) >= nsteps:
                raise _Stop()

    cwd = os.getcwd()
    tmp = workdir or tempfile.mkdtemp(prefix="pylamp_ref_")
    os.makedirs(os.path.join(tmp, "out"), exist_ok=True)
    _np.random.seed(seed)
    glb = {"__name__": "__main__", "__file__": os.path.join(REFERENCE_DIR, "pylamp2.py")}
    try:
        os.chdir(tmp)
        _np.savez = fake_savez
        sink = io.StringIO()
        with (contextlib.redirect_stdout(sink) if quiet else contextlib.nullcontext()):
            try:
                exec(compile(src, "pylamp2.py", "exec"), glb)
            except _Stop:
                pass
    finally:
        _np.savez = real_savez
        os.chdir(cwd)
    return captured
