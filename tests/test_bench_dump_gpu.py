"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step of the headline path returned (refined poses,
scores, selected index) as float .npy files, and the same arguments give the same arrays."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--no-track",
                          "--no-standin", "--no-cpu-baseline", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_dump_outputs(tmp_path):
    line = _bench(tmp_path / "a", 2)
    assert line["steps"] == 2
    d = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("poses", "scores", "best")}
    assert sorted(os.listdir(tmp_path / "a")) == ["best.npy", "poses.npy", "scores.npy"]
    assert d["poses"].shape == (252, 4, 4) and d["poses"].dtype == np.float32 and np.isfinite(d["poses"]).all()
    assert d["scores"].shape == (252,) and d["scores"].dtype == np.float32 and np.isfinite(d["scores"]).all()
    assert d["best"].dtype == np.float64 and int(d["best"]) == line["best_index"] == int(np.argmax(d["scores"]))
    assert np.allclose(d["poses"][:, 3], [0, 0, 0, 1]) and np.allclose(np.linalg.det(d["poses"][:, :3, :3]), 1, atol=1e-3)
    line_b = _bench(tmp_path / "b", 3)
    assert line_b["steps"] == 3
    for n, a in d.items():
        np.testing.assert_allclose(np.load(tmp_path / "b" / f"{n}.npy"), a, rtol=0, atol=1e-5, err_msg=n)
