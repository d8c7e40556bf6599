"""bench.py contract on the CPU side: the reference arm (`--impl reference`) prints ONE JSON line with
the keys the driver reads, on a small sample; under a multi-rank launch only rank 0 prints."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--ref-ncell", "24"], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.strip()]


def test_reference_arm_json_line():
    lines = _run({"RANK": "0", "WORLD_SIZE": "1"})
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "timesteps_per_s" and d["unit"] == "timesteps/s"
    assert d["higher_is_better"] is True and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["value"] > 0 and abs(d["value"] * d["ms_per_step"] * 1e-3 - 1.0) < 1e-9
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and d["vs_baseline"] is None
    # same config as the GPU arm's default workload; the value is the bounded sample's, scaled in proportion to the cells
    import bench
    assert d["config"]["workload"] == bench.workload_name(4096, 4) and d["config"]["grid_nodes"] == [4097, 4097]
    assert d["config"]["sample_grid_nodes"] == [25, 25]
    f = cb["scale_factor"]
    assert abs(f - (4096 / 24) ** 2) < 1e-6 and abs(cb["sample_timesteps_per_s"] / f - d["value"]) < 1e-12 * d["value"] + 1e-18


def test_reference_arm_other_ranks_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2"}) == []


def test_every_profiled_kernel_class_has_a_name():
    """bench.py names the kernel classes of csrc/common.cuh (PLB_K_*) in its breakdown; a class without a name
    once made rank 0 raise after the timed region while the other ranks waited (round 2)."""
    import re
    import bench
    src = open(os.path.join(ROOT, "pylamp_b200", "csrc", "common.cuh")).read()
    ids = [int(v) for v in re.findall(r"PLB_K_[A-Z0-9_]+ = (\d+),", src) if int(v) < 16]
    assert len(ids) >= 12
    for k in ids:
        assert k in bench.CLASS_NAMES, k
    assert bench.class_name(15).startswith("kernel class")


def test_dump_outputs_sample_is_fixed_and_order_independent(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every file holds its own field at the sampled nodes and the sampled markers' own rows,
    float64 and under the byte limit, and the marker sample does not depend on the order of the markers in memory
    (the device sort orders the markers inside a cell by the arrival of atomics)."""
    import types

    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_NODES", 5000)        # fewer nodes than the grid has: a true sample
    ncell, per_side = 160, 4            # more cells than the sample takes
    nx, L, M = [ncell + 1] * 2, [1e6, 2e6], ncell * ncell * per_side ** 2
    g = torch.Generator().manual_seed(0)
    r = lambda *shape: torch.rand(shape, generator=g, dtype=torch.float64)
    tr_x = r(M, 2) * torch.tensor(L, dtype=torch.float64)
    idx = torch.arange(M, dtype=torch.float64)            # every marker column and velocity names its marker
    grids = {"velz": r(*nx), "velx": r(*nx), "pres": r(*nx), "rho": r(*nx), "temp": r(*nx)}
    s = types.SimpleNamespace(nx=nx, L=L, tr_x=tr_x, cols=[idx + 1e7 * k for k in range(13)],
                              trac_vel=torch.stack([idx, -idx], 1), newvel=[grids["velz"], grids["velx"]],
                              newpres=grids["pres"], f_rho=grids["rho"], newtemp=grids["temp"])
    bench.dump_outputs(s, per_side, str(tmp_path / "a"))
    p = torch.randperm(M, generator=g)
    s.tr_x, s.trac_vel, s.cols = s.tr_x[p], s.trac_vel[p], [c[p] for c in s.cols]
    bench.dump_outputs(s, per_side, str(tmp_path / "b"))
    names = ["pres", "rho", "temp", "tr_f", "tr_v", "tr_x", "velx", "velz"]
    assert sorted(f.name for f in (tmp_path / "a").iterdir()) == [n + ".npy" for n in names]
    d, total = {}, 0
    for n in names:
        a, b = np.load(tmp_path / "a" / (n + ".npy")), np.load(tmp_path / "b" / (n + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, b), n
        d[n], total = a, total + a.nbytes
    assert total <= bench.DUMP_MAX_BYTES
    # the sample: bench.DUMP_SEED draws the nodes, then the cells
    rng = np.random.default_rng(bench.DUMP_SEED)
    nodes = np.sort(rng.choice(nx[0] * nx[1], 5000, replace=False))
    cells = rng.choice(ncell * ncell, bench.DUMP_MARKERS // per_side ** 2, replace=False)
    for n, f in grids.items():
        assert np.array_equal(d[n], f.reshape(-1).numpy()[nodes]), n
    x = tr_x.numpy()
    key = np.floor(ncell * x[:, 0] / L[0]).astype(np.int64) * ncell + np.floor(ncell * x[:, 1] / L[1]).astype(np.int64)
    want = np.flatnonzero(np.isin(key, cells))
    m = d["tr_f"][:, 0].astype(np.int64)                   # the marker of every dumped row
    assert 0 < len(m) < M and np.array_equal(np.sort(m), want)
    assert np.array_equal(d["tr_x"], x[m]) and np.array_equal(d["tr_v"], np.stack([m, -m], 1).astype(np.float64))
    assert np.array_equal(d["tr_f"], m[:, None] + 1e7 * np.arange(13)[None, :])
    assert np.all(np.diff(key[m]) >= 0)                    # ordered by cell
