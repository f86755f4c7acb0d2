"""CPU: the bench.py JSON contract.  The reference arm really runs here (bounded CPU sample); the GPU arm's line is checked
on the committed output of the last GPU run (profiles/), since there is no GPU in this container."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["unit"] == "evals/s" and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_committed_gpu_line_has_every_contract_key():
    d = json.loads(open(os.path.join(ROOT, "profiles", "r01_bench_v6_default.json")).read().strip().splitlines()[-1])
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["metric"].startswith("masked forward evals/sec") and d["dtype"] == "bf16" and d["scaling"] == "weak"
    assert d["gpu_launches"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert abs(d["e2e"]["value"] - d["value"]) / d["value"] < 0.1            # same metric, host buffers inside the timed region
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    c = d["clocks"]
    assert c["sm_mhz"] > 0 and c["sm_max_mhz"] >= c["sm_mhz"] and not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"])
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_rejects_no_timed_steps_and_dumps_without_the_gpu_path():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                           timeout=120, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-800:])
