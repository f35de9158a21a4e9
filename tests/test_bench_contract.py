"""bench.py's JSON contract, as far as it can be checked without a GPU: the reference arm (the compiled reference on the host
cores) prints one well-formed line; the cuda arm refuses to produce a number when there is no device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def run_bench(*argv, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH, *argv], cwd=ROOT, env=e, capture_output=True, text=True, timeout=timeout)


def json_lines(text):
    return [json.loads(l) for l in text.splitlines() if l.startswith("{")]


def test_reference_arm_prints_one_contract_line(build_libs):
    r = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = json_lines(r.stdout)
    assert len(lines) == 1
    d = lines[0]
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["impl"] == "reference"
    assert d["metric"] == "sweeps/sec scan-to-map" and d["unit"] == "sweeps/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] >= 3  # W is raised to the contract's minimum
    assert d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1000.0) < 1.0
    from oracle import pydriver
    cb = d["cpu_baseline"]
    # the compiled reference when oracle/_ref was built from its sources, else the restatement ("port") stands in
    assert cb["kind"] == ("reference" if pydriver.available("reference", fast=True) else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_quietly(build_libs):
    # under torchrun only rank 0 times the reference; the other ranks print nothing and exit 0
    r = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
                  env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29533"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert json_lines(r.stdout) == []


@pytest.mark.skipif(os.path.exists("/dev/nvidiactl"), reason="needs a box WITHOUT a GPU")
def test_cuda_arm_fails_loudly_without_a_device(build_libs):
    r = run_bench("--steps", "1", "--warmup", "3", "--no-cpu-baseline")
    assert r.returncode != 0
    assert json_lines(r.stdout) == []  # no number of any kind


def test_usage_error_is_not_retried():
    r = run_bench("--no-such-flag")
    assert r.returncode == 2
    assert r.stderr.count("attempt") == 1
