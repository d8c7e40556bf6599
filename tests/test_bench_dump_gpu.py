"""bench.py --dump-outputs on the GPU: with the same arguments two runs time the requested number of steps and
write the same sampled outputs (same shapes; values up to the fp64 summation order of the marker->grid atomics)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--ncell", "64", "--steps", "3",
                        "--warmup", "1", "--spinup", "1", "--e2e-steps", "0", "--cpu-ncell", "0",
                        "--dump-outputs", str(out_dir)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_repeat(tmp_path):
    d = [_bench(tmp_path / "a"), _bench(tmp_path / "b")]
    for line in d:
        assert line["steps"] == 3 and len(line["ms_of_each_timed_step"]) == 3
    names = sorted(f.name for f in (tmp_path / "a").iterdir())
    assert names == sorted(f.name for f in (tmp_path / "b").iterdir()) and len(names) == 8
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float64 and a.shape == b.shape and a.size > 0, n
        assert np.linalg.norm(a - b) <= 1e-8 * np.linalg.norm(b), n
