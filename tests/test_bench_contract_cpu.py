"""bench.py contract, CPU side: the reference arm (--impl reference) runs without a GPU, prints ONE JSON line with
the keys the driver reads, and times only the oracle (the CPU restatement of the reference's path)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--ref-n", "16", "--dump-outputs", str(tmp_path)], cwd=ROOT,
                       env=dict(os.environ, OMP_NUM_THREADS="1"),      # what torchrun exports: the arm must override it
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "vcycle_dofs_per_s" and d["unit"] == "DOFs/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    threads = len(os.sched_getaffinity(0))
    assert d["cpu_baseline"]["cores"] == threads and d["cpu_baseline"]["omp_threads"] == threads
    assert d["cpu_baseline"]["setup"]["seconds"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "DOFs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["z.npy"]
    z = np.load(tmp_path / "z.npy")
    assert z.dtype == np.float64 and z.ndim == 1 and np.isfinite(z).all() and np.abs(z).max() > 0


def test_dump_outputs_samples_a_long_array_within_the_budget(tmp_path):
    import bench
    a = np.arange(10000, dtype=np.float64)
    bench.dump_outputs(str(tmp_path / "one"), {"short": a[:100], "long": a}, budget=8192)
    bench.dump_outputs(str(tmp_path / "two"), {"short": a[:100], "long": a}, budget=8192)
    assert os.path.getsize(tmp_path / "one" / "short.npy") + os.path.getsize(tmp_path / "one" / "long.npy") <= 8192
    assert np.array_equal(np.load(tmp_path / "one" / "short.npy"), a[:100])
    s = np.load(tmp_path / "one" / "long.npy")
    assert s.size == (4096 - 128) // 8 and np.all(np.diff(s) > 0) and np.array_equal(s, np.floor(s))
    assert np.array_equal(np.load(tmp_path / "two" / "long.npy"), s)         # the same entries from run to run


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_multi_rank_box_size_respects_the_host_memory():
    """N > 1: the per-rank box shrinks in steps of 16 when world x 56 GB would exceed 85 % of the node's memory; both arms
    derive it from the same constant of the box"""
    import unittest.mock as mock
    import bench
    for mem, want in ((2000.0, [144, 144, 144]), (512.0, [144, 144, 128]), (256.0, [144, 128, 112])):
        with mock.patch.object(bench, "host_memory_gb", lambda mem=mem: mem):
            assert [bench.fit_box_size(144, w) for w in (2, 4, 8)] == want
            assert bench.fit_box_size(144, 1) == 144
    assert bench.host_memory_gb() > 0.0
