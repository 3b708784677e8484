"""The reference arm of bench.py (oracle port of the reference's shm path on the host) runs without a
GPU and prints the contract's JSON line."""

import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["state_dict_bytes"] == 16060522496
    gloo = d["cpu_baseline"]["gloo_transport"]  # the Gloo half of the reference's CPU transports, bounded sample
    assert gloo is not None and (gloo.get("value", 0) > 0 or "unavailable" in gloo)


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
