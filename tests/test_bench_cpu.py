"""CPU: bench.py's reference arm (the oracle port on the host cores) runs here and prints the contract's keys."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_json_line(built):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-rows", "200000"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rows/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["steps"] == 2 and d["warmup"] == 1 and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly(built):
    import os
    env = dict(os.environ, RANK="3", WORLD_SIZE="8", LOCAL_RANK="3")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "8", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr
