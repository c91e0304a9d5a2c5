"""bench.py contract, the parts that run without a GPU: the reference arm prints ONE JSON line with the keys a
reader of bench lines expects, measured through the unmodified reference extension on the host cores where it is
built (oracle/_ref), through the C restatement of oracle/ac_oracle.c otherwise."""
import json
import os
import subprocess
import sys

import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    res = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "haystack GB/s" and d["unit"] == "GB/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "u8" and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == ("reference" if oracle.ref_available("bytes") else "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and d["steps"] == 1 and d["warmup"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         cwd=ROOT, capture_output=True, text=True, timeout=120, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""
