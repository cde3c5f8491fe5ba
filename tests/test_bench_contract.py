"""bench.py contract checks: the reference arm (CPU oracle on host cores) prints one JSON line with the agreed keys, the
product arm refuses to run (no CPU fallback) when no CUDA device exists, and on a GPU --dump-outputs repeats exactly."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


def _run(*args, timeout=300):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=str(ROOT))


def test_reference_arm_prints_the_contract_line():
    p = _run("--impl", "reference", "--steps", "2", "--warmup", "1")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_s" and d["unit"] == "env-steps/s" and d["steps"] == 2
    assert d["vs_baseline"] is None and d["dtype"] == "u8" and "workload" in d["config"] and "model" not in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a machine without a GPU")
def test_product_arm_has_no_cpu_fallback():
    p = _run("--steps", "1", "--warmup", "1", timeout=120)
    assert p.returncode != 0
    assert not [l for l in p.stdout.splitlines() if l.startswith("{")], "the product arm must not print a bench line without a GPU"


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")
def test_dump_outputs_repeat_exactly(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same arrays (float32 / float64) of the last timed step."""
    args = ("--envs-per-gpu", "256", "--steps", "5", "--warmup", "3", "--preroll", "10", "--legs", "none", "--also-envs", "0",
            "--e2e-steps", "3", "--cpu-baseline-seconds", "0.1")
    outs = []
    for k in range(2):
        p = _run(*args, "--dump-outputs", str(tmp_path / str(k)))
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][0])
        assert line["steps"] == 5
        outs.append({f.name: np.load(f) for f in sorted((tmp_path / str(k)).iterdir())})
    assert sorted(outs[0]) == ["done.npy", "info_sum.npy", "obs.npy", "reward.npy"]
    assert outs[0]["obs.npy"].shape == (256, 72, 80, 4) and outs[0]["reward.npy"].shape == outs[0]["done.npy"].shape == (256,)
    assert outs[0]["info_sum.npy"][0] == 256  # slot 0 carries the env count
    for name, a in outs[0].items():
        assert a.dtype in (np.float32, np.float64), name
        assert np.array_equal(a, outs[1][name]), name
