"""bench.py's reference arm runs without a GPU (it times the reference's own receiver() on the
host cores); check the JSON contract of its line here.  The GPU arm's line is checked on the box."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    """Where oracle/_ref is not built the arm times the C restatement instead (cpu_baseline kind "port")."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "MSamples/s" and line["higher_is_better"] is True
    assert line["value"] > 10 and line["steps"] == 1 and line["data"] == "synthetic"
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert p.returncode == 0 and p.stdout.strip() == ""
