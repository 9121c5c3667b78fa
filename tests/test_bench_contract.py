"""bench.py's stdout contract, checked without a GPU on the reference arm: exactly one line, valid JSON, the keys
the driver reads; anything a library or a child process prints lands on stderr."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_exactly_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path / "out")], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.splitlines()
    assert len(lines) == 1, r.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "verifies/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert "BASELINE.json configs[1]" in d["config"]["workload"]
    st = np.load(tmp_path / "out" / "secp256k1_verify_status.npy")      # the one step's 2^16 statuses
    assert st.dtype == np.float32 and st.shape == (1 << 16,)
    assert set(np.unique(st)) == {0.0, 1.0} and st.sum() == (1 << 16) - (1 << 10)   # 1/64 corrupted


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, "bench.py", "--steps", "0"], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout == ""


def test_stdout_is_claimed_before_anything_can_write_to_it():
    code = ("import bench, os; bench.claim_stdout(); print('library noise'); os.system('echo child noise');"
            " bench.emit({'ok': 1})")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert r.stdout == '{"ok": 1}\n'
    assert "library noise" in r.stderr and "child noise" in r.stderr
