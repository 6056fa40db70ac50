"""CPU: the contract of `bench.py --impl reference` (the arm the driver runs beside the GPU arm): one JSON line with the
GPU arm's metric / unit / config keys, `impl: reference`, a `cpu_baseline` describing the run and an `e2e` object with
zero copied bytes; other ranks of a torchrun launch print nothing and exit 0.  A reduced clip / text length keeps it
short (the weights are still the 1.3B model's: the timing itself is not asserted)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, PYTHONWARNINGS="ignore", **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                           "--frames", "2", "--text-len", "16", "--queries", "16"], cwd=ROOT, env=env, capture_output=True,
                          text=True, timeout=900)


def test_reference_arm_prints_one_contract_line():
    r = _run({})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == dict(value=d["value"], unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_reference_arm_is_silent_on_other_ranks():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == "", (r.stdout, r.stderr[-500:])


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], cwd=ROOT, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode != 0 and "--steps" in r.stderr and not r.stdout.strip()


def test_product_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback, no silent substitute number: without a CUDA device the product arm exits non-zero and prints no
    JSON line (the oracle is never on its path)."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--no-cpu-baseline"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode != 0
    assert not any(l.lstrip().startswith("{") for l in r.stdout.splitlines())
