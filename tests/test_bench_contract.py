"""CPU-only: the reference arm of bench.py runs here (it is the reference's CPU kernels) -- check the JSON line
against the contract: BASELINE.json's metric verbatim, the keys the driver reads, rank > 0 stays silent."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1",
                        "--width", "384", "--height", "256"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout.strip()


def test_reference_arm_line(refc):
    out = _run()
    d = json.loads(out.splitlines()[-1])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == base["metric"] and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["dtype"] == "u8" and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert "not a full encode" in d["metric_scope"]


def test_reference_arm_other_ranks_print_nothing():
    assert _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}) == ""
