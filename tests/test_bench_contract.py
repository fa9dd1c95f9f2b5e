"""CPU: the parts of bench.py's contract that run without a GPU — the reference arm (the unmodified
reference, or the oracle port where /root/reference is absent, timed on host cores) prints exactly
one JSON line with the keys the driver reads, alone on rank 0 under a multi-rank launch; and the
GPU arm refuses to run without a device instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "cpu_baseline", "impl"}


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=600, env=e)


def test_reference_arm_prints_one_line():
    res = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-sample-bases", "1200000")
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    line = json.loads(lines[0])
    assert BASE_KEYS <= set(line), BASE_KEYS - set(line)
    assert line["impl"] == "reference" and line["unit"] == "Gbp/s" and line["steps"] == 2 and line["warmup"] == 1
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["workload"].startswith("config 3") and line["config"]["bases"] == 3_100_000_000


def test_reference_arm_other_ranks_stay_silent():
    res = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-sample-bases", "1200000",
                    env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert res.returncode == 0 and res.stdout.strip() == "", (res.stdout, res.stderr[-1000:])


def test_rejects_invalid_arguments():
    for args in (("--steps", "0"), ("--warmup", "-1"), ("--impl", "reference", "--dump-outputs", "out")):
        res = run_bench(*args)
        assert res.returncode == 2 and res.stdout == "", (args, res.stderr[-500:])


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        return  # covered by the GPU tests
    res = run_bench("--steps", "1", "--warmup", "0", "--bases", "1200000", "--no-cpu-baseline")
    assert res.returncode != 0
    assert "{" not in res.stdout  # no result line from a CPU fallback
