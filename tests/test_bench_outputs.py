"""bench.py --dump-outputs: the flagship workload's last timed step (one CUDA-graph replay) written as .npy files, with
inputs that depend only on the arguments, so two runs of the same build agree."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, steps):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "bnn", "--steps", str(steps), "--warmup", "2",
                        "--no-cpu-baseline", "--no-api", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_bench_dump_outputs_repeat(tmp_path):
    d, a = run_bench(tmp_path / "a", 3)
    assert d["steps"] == 3
    shapes = {"weights1": (100, 784), "b1": (100, 1), "weights2": (10, 100), "b2": (10, 1)}
    want = {"loss": ()}
    for n, s in shapes.items():
        want["grad_%s_loc" % n] = want["grad_%s_scale" % n] = s
    assert {k: v.shape for k, v in a.items()} == want
    assert a["loss"].dtype == np.float64 and all(v.dtype == np.float32 for k, v in a.items() if k != "loss")
    assert all(np.isfinite(v).all() for v in a.values()) and np.abs(a["grad_weights1_loc"]).max() > 0
    _, b = run_bench(tmp_path / "b", 3)
    for k in a:
        np.testing.assert_allclose(b[k], a[k], rtol=1e-6, atol=1e-6 * np.abs(a[k]).max(), err_msg=k)
