"""The snapshot reader on the GPU (pylamp_b200/output.py: read_snapshot, driver.load_npz): the row selection kernel
plb_unpack_rows against torch, bit for bit; one-GPU round trips and continued runs against uninterrupted ones and
against the oracle continuing a file in the reference's own format; injection after a resume; and (>= 2 GPUs,
torchrun, scripts/resume_check.py) the multi-GPU reads."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import pylamp_oracle as O
from pylamp_b200 import setups
from pylamp_b200.pylamp_const import IX, IZ, TR__ID

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.contiguous().reshape(-1).view(torch.uint8)


def _unpack(ctx, x, f, v, nz, Lz, c0, c1, r0, r1, base=0, dst=None):
    """plb_unpack_rows on a chunk; dst = (tr_x, cols, trac_vel) to fill, None to count only."""
    from pylamp_b200 import _lib
    cnt = C.c_longlong(-1)
    if dst is None:
        ctx.call("plb_unpack_rows", x.shape[0], x.data_ptr(), None, 13, None, nz, float(Lz), c0, c1, r0, r1, 0, 0,
                 None, None, None, C.byref(cnt))
    else:
        dx, cols, dv = dst
        ctx.call("plb_unpack_rows", x.shape[0], x.data_ptr(), f.data_ptr(), 13,
                 v.data_ptr() if dv is not None else None, nz, float(Lz), c0, c1, r0, r1, base, dx.shape[0],
                 dx.data_ptr(), _lib.ptr_array(cols), dv.data_ptr() if dv is not None else None, C.byref(cnt))
    return cnt.value


def _chunk(n, nz, Lz, dist, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    z = (torch.rand(n, dtype=torch.float64, device="cuda", generator=g) * 1.1 - 0.05) * Lz   # z < 0 and z > Lz too
    if dist == "low":           # every marker in the lowest cell rows: the upper slabs are empty
        z = z.abs() * 0.2
    if dist == "edges" and n:   # exactly on cell-row (and so slab) boundaries
        z[::3] = torch.floor(z[::3] / Lz * (nz - 1)).clamp(0, nz - 1) * Lz / (nz - 1)
    x = torch.stack([z, torch.rand(n, dtype=torch.float64, device="cuda", generator=g)], 1).contiguous()
    f = torch.randn((n, 13), dtype=torch.float64, device="cuda", generator=g)
    f[:, TR__ID] = torch.arange(n, dtype=torch.float64, device="cuda")
    v = torch.randn((n, 2), dtype=torch.float64, device="cuda", generator=g)
    return x, f, v


@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 5000])
@pytest.mark.parametrize("dist", ["uniform", "low", "edges"])
def test_unpack_rows_equals_torch(n, dist):
    from pylamp_b200 import _lib, migrate
    ctx = _lib.default_context()
    nz, Lz = 33, 1e6
    x, f, v = _chunk(n, nz, Lz, dist, seed=n + len(dist))
    for W in (1, 2, 3, 5):
        b = migrate.slab_bounds(nz - 1, W)
        owner = migrate.owner_of(x[:, 0], nz, Lz, b)
        parts = []
        for r in range(W):
            idx = torch.nonzero(owner == r).flatten()
            k = idx.numel()
            assert _unpack(ctx, x, f, v, nz, Lz, b[r], b[r + 1], 0, n) == k
            base = 5                                      # rows already there, and 3 spare rows after the new ones
            dx = torch.full((base + k + 3, 2), 7.0, dtype=torch.float64, device="cuda")
            cols = [torch.full((base + k + 3,), 7.0, dtype=torch.float64, device="cuda") for _ in range(13)]
            dv = torch.full((base + k + 3, 2), 7.0, dtype=torch.float64, device="cuda")
            assert _unpack(ctx, x, f, v, nz, Lz, b[r], b[r + 1], 0, n, base, (dx, cols, dv)) == k
            torch.cuda.synchronize()
            assert torch.equal(_bits(dx[base:base + k]), _bits(x[idx])), (W, r)
            assert torch.equal(_bits(dv[base:base + k]), _bits(v[idx])), (W, r)
            for c in range(13):
                assert torch.equal(_bits(cols[c][base:base + k]), _bits(f[idx, c])), (W, r, c)
            for t in [dx, dv] + cols:
                assert bool((t[:base] == 7.0).all()) and bool((t[base + k:] == 7.0).all())
            parts.append(dx[base:base + k])
        # the ranks' rows, concatenated by rank: a stable sort of the chunk by owner
        order = torch.argsort(owner, stable=True)
        assert torch.equal(_bits(torch.cat(parts)), _bits(x[order])), W


def test_unpack_rows_window_and_no_velocities():
    """The file-row window of marker_ownership="index", without marker velocities."""
    from pylamp_b200 import _lib
    ctx = _lib.default_context()
    nz, Lz, n = 17, 2.0, 1000
    x, f, v = _chunk(n, nz, Lz, "uniform", seed=9)
    for r0, r1 in ((0, n), (0, 0), (300, 301), (255, 777), (600, n), (900, 2000), (-5, 10)):
        lo, hi = max(r0, 0), min(r1, n)
        k = max(hi - lo, 0)
        assert _unpack(ctx, x, f, v, nz, Lz, 0, nz - 1, r0, r1) == k
        dx = torch.zeros((k, 2), dtype=torch.float64, device="cuda")
        cols = [torch.zeros(k, dtype=torch.float64, device="cuda") for _ in range(13)]
        assert _unpack(ctx, x, f, v, nz, Lz, 0, nz - 1, r0, r1, 0, (dx, cols, None)) == k
        torch.cuda.synchronize()
        assert torch.equal(_bits(dx), _bits(x[lo:hi])) and torch.equal(_bits(torch.stack(cols, 1)), _bits(f[lo:hi]))


def test_unpack_rows_rejects_non_finite_z():
    from pylamp_b200 import _lib
    ctx = _lib.default_context()
    nz, Lz, n = 17, 2.0, 600
    for bad in (float("nan"), float("inf"), -float("inf")):
        x, f, v = _chunk(n, nz, Lz, "uniform", seed=4)
        x[413, 0] = bad
        dx = torch.full((n, 2), 7.0, dtype=torch.float64, device="cuda")
        cols = [torch.full((n,), 7.0, dtype=torch.float64, device="cuda") for _ in range(13)]
        for r0, r1 in ((0, n), (0, 10)):        # outside the window too: the row has no owner at all
            with pytest.raises(_lib.PlbError, match="non-finite"):
                _unpack(ctx, x, f, v, nz, Lz, 0, 3, r0, r1, 0, (dx, cols, None))
        torch.cuda.synchronize()
        assert bool((dx == 7.0).all()) and all(bool((c == 7.0).all()) for c in cols)


def _tensors(s):
    return {"tr_x": s.tr_x, "trac_vel": s.trac_vel, "velz": s.newvel[IZ], "velx": s.newvel[IX], "pres": s.newpres,
            "temp": s.newtemp, **{"col%d" % k: c for k, c in enumerate(s.cols)}}


def test_round_trip_one_gpu(tmp_path, monkeypatch):
    from pylamp_b200 import driver, output
    nx, L, tr_x, tr_f, opts = setups.convection(ncell=64)
    s, o = driver.State(nx, L, tr_x, tr_f), driver.Options(**opts)
    for _ in range(3):
        driver.timestep(s, o)
    monkeypatch.setattr(output, "CHUNK_BYTES", 8 * 13 * 777)        # 85 chunks
    a, b = str(tmp_path / "a") + "/", str(tmp_path / "b") + "/"
    os.makedirs(a), os.makedirs(b)
    driver.save_npz(s, a)
    stats = {}
    r = output.read_snapshot(a, 3, o, stats=stats)
    assert stats["chunks"] == 85 and stats["pinned_bytes"] == 2 * 8 * (17 * 777 + 1)
    assert r.nx == s.nx and r.L == s.L and r.it == 3 and r.totaltime == s.totaltime
    assert all(np.array_equal(p, q) for p, q in zip(r.grid + r.gridmp, s.grid + s.gridmp))
    assert len({c.data_ptr() for c in r.cols}) == 13
    want, got = _tensors(s), _tensors(r)
    for k, t in want.items():
        assert got[k].shape == t.shape and torch.equal(_bits(got[k]), _bits(t)), k
    # the resumed state writes the same files (rho apart: a fresh state rebuilds it in its first step)
    driver.save_npz(r, b)
    for name in ("griddata.3.npz", "tracs.3.npz"):
        with np.load(a + name) as p, np.load(b + name) as q:
            assert p.files == q.files
            for k in p.files:
                if k != "rho":
                    assert p[k].dtype == q[k].dtype and p[k].tobytes() == q[k].tobytes(), k
    r2 = driver.load_npz(b, 3, o)
    assert torch.equal(_bits(r2.tr_x), _bits(s.tr_x)) and torch.equal(_bits(r2.newtemp), _bits(s.newtemp))


def _rel(a, b):
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    return np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300)


def _agree(g, ref, label):
    """The criteria of test_driver_gpu._run_both: fields 1e-8 relative L2, marker positions 1e-10, the same limiter,
    the total count, kelem agreement above 0.9999.  `ref`: a driver.State or an oracle State."""
    e = {"vz": _rel(g.newvel[0], ref.newvel[0]), "vx": _rel(g.newvel[1], ref.newvel[1]),
         "P": _rel(g.newpres, ref.newpres), "T": _rel(g.newtemp, ref.newtemp), "x": _rel(g.tr_x, ref.tr_x)}
    print(label, "stats", g.stats, {k: "%.1e" % v for k, v in e.items()}, g.limiter, ref.limiter)
    assert all(e[k] <= 1e-8 for k in ("vz", "vx", "P", "T")), e
    assert e["x"] <= 1e-10, e
    assert g.limiter == ref.limiter
    rk = ref.kelem.cpu().numpy() if isinstance(ref.kelem, torch.Tensor) else ref.kelem
    rc = ref.count.cpu().numpy() if isinstance(ref.count, torch.Tensor) else ref.count
    assert int(g.count.sum()) == int(rc.sum()) == g.ntrac
    assert np.mean(g.kelem.cpu().numpy() == rk) > 0.9999


def test_resumed_run_continues_the_uninterrupted_one(tmp_path):
    from pylamp_b200 import driver
    nx, L, tr_x, tr_f, opts = setups.convection(ncell=64)
    o = driver.Options(**opts)
    full, part = driver.State(nx, L, tr_x, tr_f), driver.State(nx, L, tr_x, tr_f)
    for _ in range(3):
        driver.timestep(full, o)
        driver.timestep(part, o)
    prefix = str(tmp_path) + "/"
    driver.save_npz(part, prefix)
    r = driver.load_npz(prefix, 3, o)
    del part
    for step in range(3):
        driver.timestep(full, o)
        driver.timestep(r, o)
        if step == 0:
            print("first resumed step: stokes_iters", r.stats["stokes_iters"], "uninterrupted",
                  full.stats["stokes_iters"])
        assert r.it == full.it
        _agree(r, full, "step %d" % r.it)


def test_resume_from_the_reference_format(tmp_path):
    """A pair written as pylamp2.py:637-650 writes it (np.savez, its keys) by the oracle, continued on the GPU."""
    from pylamp_b200 import driver
    nx, L, tr_x, tr_f, opts = setups.convection(ncell=32)
    so, oo = O.State(nx, L, tr_x.copy(), tr_f.copy()), O.Options(solve=O.solve_refined, **opts)
    for _ in range(2):
        O.timestep(so, oo)
    prefix = str(tmp_path) + "/"
    np.savez(prefix + "griddata.2.npz", gridz=so.grid[IZ], gridx=so.grid[IX], velz=so.newvel[IZ],
             velx=so.newvel[IX], pres=so.newpres, rho=so.f_rho, temp=so.newtemp, tstep=so.it, time=so.totaltime)
    np.savez(prefix + "tracs.2.npz", tr_x=so.tr_x, tr_f=so.tr_f, tr_v=so.trac_vel)
    og = driver.Options(**opts)
    sg = driver.load_npz(prefix, 2, og)
    assert sg.it == 2 and sg.totaltime == so.totaltime and sg.trac_vel is not None
    for _ in range(3):
        O.timestep(so, oo)
        driver.timestep(sg, og)
        _agree(sg, so, "step %d" % sg.it)


def test_resume_with_injection(tmp_path):
    from pylamp_b200 import driver, output
    nx, L, tr_x, tr_f, opts = setups.convection(ncell=32)
    o = driver.Options(tracdens=20, tracdens_min=17, **opts)       # 16 markers per cell: every cell gets 4 more
    s = driver.State(nx, L, tr_x, tr_f)
    for _ in range(2):
        driver.timestep(s, o)
    assert s.trac_vel.shape[0] < s.ntrac                            # the new markers have no velocity yet
    prefix = str(tmp_path) + "/"
    driver.save_npz(s, prefix)
    r = driver.load_npz(prefix, 2, o)
    assert r.trac_vel is None and r.ntrac == s.ntrac
    assert torch.equal(_bits(r.tr_x), _bits(s.tr_x))
    with pytest.raises(TypeError):
        output.write_snapshot(r, prefix, 99)
    fmax = float(s.cols[TR__ID].max())
    M1 = r.ntrac
    driver.timestep(r, o)
    assert r.stats["injected"] > 0 and r.trac_vel is not None
    new = r.cols[TR__ID][M1:].cpu().numpy()
    old = r.cols[TR__ID][:M1].cpu().numpy()
    assert new.size == r.stats["injected"] and new.min() >= fmax and new.max() > fmax and old.max() == fmax
    driver.save_npz(r, prefix)                                     # a step later the writer works again


@pytest.mark.parametrize("mode,port", [("slab", 29571), ("one", 29573), ("index", 29575)])
def test_two_gpu_resume(mode, port):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "scripts", "resume_check.py"), mode]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:], r.stderr[-3000:])
    assert r.returncode == 0 and "RESUME_CHECK OK" in r.stdout
