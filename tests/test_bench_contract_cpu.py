"""CPU-side check of bench.py's reference arm (the one leg that needs no GPU): one JSON line with the contract's keys."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "gemm_gflops" and d["unit"] == "GFLOP/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["dtype"] == "f32" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "32768" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_rejects_zero_steps():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun only rank 0 runs the CPU arm; the other ranks exit 0 without output."""
    import os
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]
