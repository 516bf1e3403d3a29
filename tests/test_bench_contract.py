"""bench.py's reference arm on the GPU-less host: the JSON line the driver parses (keys, units, the cpu_baseline / e2e objects of
the reference arm, exactly one line on stdout) and the rank rule under a launcher (ranks other than 0 exit 0 without work)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                           "--no-cpu-full-step", *args], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "dit_steps_per_s" and d["unit"] == "steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and abs(d["value"] - 1e3 / d["ms_per_step"]) <= 1e-6 * d["value"]
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["gpu_launches"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["unit"] == "steps/s" and cb["sample"]
    assert d["e2e"] == dict(value=d["value"], unit="steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert d["extrapolated"] is True      # one block timed, x 48: said so in the line


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(dict(RANK="1", LOCAL_RANK="1", WORLD_SIZE="2"), ("--gpus", "2"))
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_bad_arguments_are_refused_before_any_work():
    """--steps is the number of timed steps, so it must be at least 1; --dump-outputs writes the product arm's outputs only."""
    for args in (("--steps", "0"), ("--steps", "-3"), ("--dump-outputs", "unused")):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--warmup", "0", *args],
                           capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 2 and r.stdout.strip() == "", (args, r.returncode, r.stdout[-500:])
        assert "--steps" in r.stderr or "--dump-outputs" in r.stderr, r.stderr[-500:]


def test_product_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: on a host without a CUDA device the product arm exits non-zero and prints no result line."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                       env=env, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and r.stdout.strip() == "" and "no CPU fallback" in r.stderr
