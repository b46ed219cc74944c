"""bench.py contract checks that need no GPU: the reference arm's JSON line, and that the product arm refuses to run
(no CPU fallback) when there is no CUDA device."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, env=e, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = run_bench("--impl", "reference", "--n", "20000", "--steps", "2", "--warmup", "1", "--ref-procs", "2")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "gibbs_sweep_plus_vecchia_loglik_per_sec" and line["unit"] == "steps/s (1M-site blocks)"
    assert line["higher_is_better"] is True and line["dtype"] == "f64" and line["data"] == "synthetic" and line["vs_baseline"] is None
    assert line["value"] > 0 and line["steps"] == 2 and line["n_gpus"] == 1
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 2 and cb["value"] == line["value"] and "oracle restatement" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "steps/s (1M-site blocks)", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = run_bench("--impl", "reference", "--n", "20000", "--steps", "1", env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_arm_fails_loudly_without_a_gpu():
    r = run_bench("--steps", "1", "--warmup", "1", "--n", "2000")
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)


def test_dump_outputs_is_refused_where_it_is_not_implemented(tmp_path):
    r = run_bench("--impl", "reference", "--n", "2000", "--steps", "1", "--dump-outputs", str(tmp_path))
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
    assert list(tmp_path.iterdir()) == []
