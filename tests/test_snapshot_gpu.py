"""The snapshot writer on the GPU (pylamp_b200/output.py): the column pack kernel against torch.stack, one-GPU
snapshots against the state and against the former in-memory writer, and (>= 2 GPUs, torchrun) the multi-GPU
files against every rank's arrays gathered independently."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from pylamp_b200 import setups
from pylamp_b200.pylamp_const import IX, IZ, TR_IHT, TR_MRK, TR__ID

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.contiguous().reshape(-1).view(torch.uint8)


@pytest.mark.parametrize("r0,n", [(0, 0), (37, 0), (5, 1), (300, 1000), (0, 2049), (0, 5000), (1, 4999)])
@pytest.mark.parametrize("alias", [False, True])
def test_pack_columns_equals_torch_stack(r0, n, alias):
    from pylamp_b200 import _lib, output
    ctx = _lib.default_context()
    M = 5000
    g = torch.Generator(device="cuda").manual_seed(3)
    cols = [torch.randn(M, dtype=torch.float64, device="cuda", generator=g) for _ in range(13)]
    cols[4][::7] = float("nan")
    cols[9][::11] = -0.0
    if alias:       # the bench cloud's one zero column for TR_MRK, TR__ID and TR_IHT
        cols[TR_MRK] = cols[TR__ID] = cols[TR_IHT]
        cols[2] = cols[0]
    out = torch.full((n + 3, 13), 7.0, dtype=torch.float64, device="cuda")
    output.pack_columns(ctx, cols, r0, n, out)
    torch.cuda.synchronize()
    assert torch.equal(_bits(out[:n]), _bits(torch.stack(cols, 1)[r0:r0 + n]))
    assert bool((out[n:] == 7.0).all())                 # nothing written beyond n rows
    assert torch.equal(_bits(output.pack_columns(ctx, cols, r0, n)), _bits(torch.stack(cols, 1)[r0:r0 + n]))


def _old_save_npz(s, prefix, it):
    """driver.save_npz as it was before the streaming writer: every array in host memory, np.savez."""
    host = lambda t: t.detach().cpu().numpy() if t is not None else np.zeros(tuple(s.nx))
    np.savez("%sgriddata.%d.npz" % (prefix, it), gridz=s.grid[IZ], gridx=s.grid[IX], velz=host(s.newvel[IZ]),
             velx=host(s.newvel[IX]), pres=host(s.newpres), rho=host(s.f_rho), temp=host(s.newtemp),
             tstep=it, time=s.totaltime)
    np.savez("%stracs.%d.npz" % (prefix, it), tr_x=host(s.tr_x), tr_f=s.tr_f_host(), tr_v=host(s.trac_vel))


def _tensors(s):
    """Every tensor the state holds, by name."""
    out = {}
    for k, v in vars(s).items():
        if isinstance(v, torch.Tensor):
            out[k] = v
        elif isinstance(v, (list, tuple)):
            out.update({"%s[%d]" % (k, i): t for i, t in enumerate(v) if isinstance(t, torch.Tensor)})
    return out


def _same_npz(a, b):
    with np.load(a) as x, np.load(b) as y:
        assert x.files == y.files
        for k in x.files:
            assert x[k].dtype == y[k].dtype and x[k].shape == y[k].shape, k
            assert x[k].tobytes() == y[k].tobytes(), k


def test_one_gpu_snapshot_after_three_steps(tmp_path, monkeypatch):
    from pylamp_b200 import driver, output
    nx, L, tr_x, tr_f, opts = setups.convection(ncell=64)
    s, o = driver.State(nx, L, tr_x, tr_f), driver.Options(**opts)
    for _ in range(3):
        driver.timestep(s, o)
    monkeypatch.setattr(output, "CHUNK_BYTES", 8 * 13 * 777)        # tr_f: 85 chunks, tr_x / tr_v: 13 each
    before = {k: t.clone() for k, t in _tensors(s).items()}
    new, old = str(tmp_path / "new") + "/", str(tmp_path / "old") + "/"
    os.makedirs(new), os.makedirs(old)
    stats = output.write_snapshot(s, new)
    assert stats["chunks"] == 85 + 2 * 13 and stats["bytes"] > 0
    after = _tensors(s)
    assert set(after) == set(before)
    for k, t in before.items():
        assert after[k].dtype == t.dtype and after[k].shape == t.shape and torch.equal(_bits(after[k]), _bits(t)), k
    with np.load(new + "tracs.3.npz") as t, np.load(new + "griddata.3.npz") as g:
        assert t["tr_x"].tobytes() == s.tr_x.cpu().numpy().tobytes() and t["tr_x"].shape == tuple(s.tr_x.shape)
        assert t["tr_f"].tobytes() == s.tr_f_host().tobytes() and t["tr_f"].shape == (s.ntrac, 13)
        assert t["tr_v"].tobytes() == s.trac_vel.cpu().numpy().tobytes()
        planes = {"velz": s.newvel[IZ], "velx": s.newvel[IX], "pres": s.newpres, "rho": s.f_rho, "temp": s.newtemp}
        for k, f in planes.items():
            assert g[k].tobytes() == f.cpu().numpy().tobytes(), k
        assert int(g["tstep"]) == 3 and float(g["time"]) == s.totaltime
    # driver.save_npz writes the same arrays as the former in-memory writer
    driver.save_npz(s, new, it=5)
    _old_save_npz(s, old, 5)
    _same_npz(new + "griddata.5.npz", old + "griddata.5.npz")
    _same_npz(new + "tracs.5.npz", old + "tracs.5.npz")


def test_snapshot_before_the_first_step_writes_nothing(tmp_path):
    """As before the streaming writer: no velocities yet, so an error and no file."""
    from pylamp_b200 import driver
    nx, L, tr_x, tr_f, opts = setups.convection(ncell=16)
    s = driver.State(nx, L, tr_x, tr_f)
    with pytest.raises(TypeError):
        driver.save_npz(s, str(tmp_path) + "/")
    assert os.listdir(tmp_path) == []


@pytest.mark.parametrize("mode,port", [("slab local", 29551), ("index", 29553)])
def test_two_gpu_snapshot_equals_gathered_arrays(mode, port):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "scripts", "snapshot_check.py"), "64", "3"] + mode.split()
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and "SNAPSHOT_CHECK OK" in r.stdout
