"""CPU: the reference arm of bench.py (`--impl reference`: the reference networks' CPU port on a bounded sample, the one
leg of the benchmark that needs no GPU) prints ONE JSON line with the keys the driver's contract names."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines                      # stdout carries the JSON line and nothing else
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "hyp/s" and d["n_gpus"] == 1
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and abs(d["ms_per_step"] * 1e-3 * d["value"] - d["config"]["hypotheses_per_step"]) < 1e-6
    assert "252 hyp" in d["metric"] and "5 refine iters" in d["metric"] and d["vs_baseline"] is None and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["unit"] == "hyp/s" and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "hyp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_rejects_zero_steps_and_dumps_of_other_arms(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, (extra, out.stderr[-2000:])
        assert out.stdout == ""
    assert not os.listdir(tmp_path)
