"""CPU: the reference arm of bench.py (``--impl reference``: the verbatim reference on the host cores) prints one
JSON line with the keys the driver reads; under torchrun only rank 0 works and prints."""
import json
import os
import subprocess
import sys

import pytest

from oracle.ref_shim import reference_available

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(extra_env):
    env = dict(os.environ, OO_BENCH_CPU_SAMPLE_NAO="20", **extra_env)       # a tiny sample keeps the test in seconds
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stdout


@pytest.mark.skipif(not reference_available(), reason="needs the auto_oo reference sources, which are not part of "
                                                      "this repository (AUTO_OO_REFERENCE or baseline/_ref)")
def test_reference_arm_prints_one_json_line():
    out = run({})
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "oo_energy_gradient_hessian_evals_per_sec"
    assert d["unit"] == "evals/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["config"]["workload"] == "synthetic_n256_cas1212"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and "verbatim reference" in cb["sample"]
    assert cb["extrapolated"] is True and cb["sample_nao"] == 20 and cb["scale"] > 1 and cb["steps_measured"] == 1
    assert abs(cb["value"] - d["value"]) <= 1e-12 * d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    assert run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}).strip() == ""
