"""bench.py --dump-outputs on a small batch: the files, their dtypes, shapes and total size, the timed step count
the JSON line reports; that the same arguments give the same outputs, and that the dump is the LAST timed step's."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCH = 16
SHAPES = {"loss": (), "outputs": (BATCH, 1), "encoding": (BATCH, 2048), "bn_running_stats": (2 * 26560,),
          "parameters_sample": (1 << 22,), "gradients_sample": (1 << 22,)}


def _bench_dump(steps, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                        "--batch", str(BATCH), "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    assert sorted(os.listdir(out_dir)) == sorted(n + ".npy" for n in SHAPES)
    assert sum(os.path.getsize(out_dir / f"{n}.npy") for n in SHAPES) <= 64 << 20
    return {n: np.load(out_dir / f"{n}.npy") for n in SHAPES}


def test_bench_dumps_the_last_timed_step(tmp_path):
    one_a = _bench_dump(1, tmp_path / "one_a")
    one_b = _bench_dump(1, tmp_path / "one_b")
    two = _bench_dump(2, tmp_path / "two")
    for name, shape in SHAPES.items():
        a = one_a[name]
        assert a.dtype == np.float32 and a.shape == shape, (name, a.dtype, a.shape)
        assert np.isfinite(a).all() and np.isfinite(two[name]).all(), name
        assert np.array_equal(a, one_b[name]), f"{name}: two runs with the same arguments differ"
    assert np.abs(two["gradients_sample"]).max() > 0
    # the second timed step trains on another batch after one more Adam update: a dump of the first step would match
    for name in ("loss", "outputs", "parameters_sample", "gradients_sample"):
        assert not np.array_equal(two[name], one_a[name]), f"{name}: --steps 2 dumped the first timed step"
