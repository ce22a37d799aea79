"""bench.py's contract, as far as it can be checked without a GPU: the reference arm runs the reference's own sources on the host
cores and prints ONE JSON line with the keys the driver reads; the product arm refuses to run without a CUDA device (there is no CPU
fallback behind it)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from helpers import assert_parity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def check_dump(d):
    """--dump-outputs wrote fp64 g and jac of the dump_rows() instances, at most 64 MB, equal to the oracle on the same inputs."""
    assert sorted(os.listdir(d)) == ["g.npy", "jac.npy"]
    assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64_000_000
    got = {k: np.load(os.path.join(d, f"{k}.npy")) for k in ("g", "jac")}
    assert all(a.dtype == np.float64 for a in got.values())
    o = bench.oracle_problem()
    want = o.eval_batch(bench.make_inputs(0)[bench.dump_rows()], want=("g", "jac"))
    assert_parity(got, {"g": want["g"], "jac": want["jac"]}, o, "bench --dump-outputs")


def test_reference_arm_prints_the_contract_line():
    r = run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "instances/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("configs[1]") and "65,536" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_dumps_its_last_step(tmp_path):
    """Without oracle/_ref the reference arm runs the C oracle itself, so this checks the dump's rows, dtype, names and size;
    the parity of the GPU path's dump is test_product_arm_dumps_its_last_step."""
    r = run("--impl", "reference", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 0, r.stderr[-2000:]
    check_dump(tmp_path / "out")


@pytest.mark.gpu
def test_product_arm_dumps_its_last_step(cuda_device, tmp_path):
    r = run("--steps", "5", "--warmup", "3", "--regions", "1", "--no-cpu", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["gpu_launches"] == 5 and d["timing"]["timed_regions"]["n"] == 1  # launches one timed region issued
    check_dump(tmp_path / "out")


def test_product_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present: the product arm would run")
    r = run("--steps", "1", "--warmup", "3", timeout=120)
    assert r.returncode != 0 and "no CPU fallback" in (r.stdout + r.stderr)
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]      # no number without the CUDA path
