"""bench.py on the GPU with the tiny debug models: --steps sets the timed steps and --dump-outputs writes what the last timed step returned,
the same arrays on every run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--no-cpu-baseline", "--steps", "2", "--warmup", "1",
                        "--denoise-steps", "3", "--dump-outputs", str(out_dir), *extra], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_bench_dumps_the_same_outputs_on_every_run(tmp_path):
    lines = [_bench(tmp_path / d) for d in ("a", "b")]
    assert all(ln["steps"] == 2 for ln in lines)
    a, b = np.load(tmp_path / "a" / "images.npy"), np.load(tmp_path / "b" / "images.npy")
    assert a.dtype == np.float32 and a.shape == (4, 1024, 1024, 3) and a.min() >= 0 and a.max() <= 255 and a.std() > 0
    d = np.abs(a - b)
    assert np.array_equal(a, b), (d.mean(), d.max(), (d > 0).mean())


def test_bench_dumps_the_text_answer_of_the_anyres_workload(tmp_path):
    line = _bench(tmp_path, "--workload", "anyres", "--batch", "1")
    assert line["steps"] == 2
    ids = np.load(tmp_path / "text_ids.npy")
    assert ids.shape == (1, 128) and np.array_equal(ids, np.round(ids))
    assert np.load(tmp_path / "images.npy").shape == (1, 1024, 1024, 3)
