"""bench.py contract on the CPU: the reference arm (oracle port on the host cores) prints ONE JSON line
with the keys the driver reads.  No GPU, no CUDA library call."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra, env=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--images", "10", "--feats", "512", "--cpu-seconds", "1", *extra]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["metric"] == "image-pairs matched+verified/sec" and d["unit"] == "pairs/s"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["dtype"] == "u8" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_rejects_zero_steps_and_dumping_the_reference_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                             timeout=60, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr and out.stdout == "", extra


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    assert _run("--gpus", "2", env=env) == []
