"""bench.py --dump-outputs on the GPU path: the file holds what the timed V-cycles returned, and the inputs depend on the
arguments only, so runs that differ in --steps alone store the same vector."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _bench(steps, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--size", "16",
                        "--levels", "3", "--no-parity", "--no-cpu-baseline", "--no-weak-base", "--dump-outputs", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_holds_the_timed_vcycle_result(tmp_path):
    d2, d3 = _bench(2, tmp_path / "a"), _bench(3, tmp_path / "b")
    assert d2["steps"] == 2 and d3["steps"] == 3
    assert sorted(os.listdir(tmp_path / "a")) == ["z.npy"]
    za, zb = np.load(tmp_path / "a" / "z.npy"), np.load(tmp_path / "b" / "z.npy")
    assert za.dtype == np.float64 and za.shape == (d2["config"]["global_true_dofs"],)
    assert np.isfinite(za).all() and np.abs(za).max() > 0
    assert np.allclose(za, zb, rtol=0, atol=1e-12 * np.abs(za).max())
