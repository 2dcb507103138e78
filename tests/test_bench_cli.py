"""bench.py's command line on CPU: the argument checks that run before any device work, and the files --dump-outputs writes."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=120)


def test_steps_must_be_positive():
    r = _bench("--steps", "0")
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_dump_outputs_is_refused_for_the_cpu_sample(tmp_path):
    r = _bench("--impl", "reference", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not (tmp_path / "out").exists()


def test_dump_outputs_files(tmp_path):
    import bench

    ids = np.array([34302, 64490, 128255], dtype=np.int32)
    logits = np.linspace(-3, 3, 11, dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "one"), ids, logits)
    got_ids, got_logits = np.load(tmp_path / "one" / "ids.npy"), np.load(tmp_path / "one" / "logits.npy")
    assert got_ids.dtype == np.float64 and np.array_equal(got_ids, ids)
    assert got_logits.dtype == np.float32 and np.array_equal(got_logits.view(np.uint32), logits.view(np.uint32))
    bench.dump_outputs(str(tmp_path / "tp"), ids, None)  # tensor-parallel: ids only
    assert sorted(os.listdir(tmp_path / "tp")) == ["ids.npy"]
