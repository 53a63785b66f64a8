"""bench.py output contract: the reference arm (the reference's own processor on the CPU) on the tiny contract-test
workload must print ONE JSON line with every key the driver reads; the GPU arm is checked the same way on a B200.
The reference is not part of this repository: without its files the reference arm must say so and the GPU arm must
report `cpu_baseline` as unavailable.  --dump-outputs must write the same arrays from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _run(extra):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", *extra],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, res.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    if not ref_loader.available():
        pytest.skip("the reference's own files are absent (VORTA_REFERENCE_ROOT, or a staged oracle/_ref)")
    d = _run(["--impl", "reference", "--steps", "2", "--warmup", "1"])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "dit_denoise_step_ms" and d["unit"] == "ms" and d["higher_is_better"] is False
    assert d["vs_baseline"] is None and "workload" in d["config"] and "model" not in d["config"]
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"] == d["ms_per_step"]          # measured, never extrapolated
    assert d["e2e"] == {"value": d["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_without_the_reference_says_so(tmp_path):
    """Nothing else is timed under the reference's name: with no reference files the arm exits with the reason."""
    code = ("import runpy, sys; from oracle import ref_loader; ref_loader.REFERENCE_ROOT = sys.argv[1]; "
            "sys.argv = ['bench.py', '--workload', 'tiny', '--impl', 'reference']; "
            "runpy.run_path('bench.py', run_name='__main__')")
    res = subprocess.run([sys.executable, "-c", code, str(tmp_path)], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert res.returncode != 0 and res.stdout.strip() == ""
    assert "reference not available" in res.stderr


def test_dump_outputs_within_budget_and_same_sample_every_run(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 4096 + 2 * 4 * 1000)          # 1000 elements per array
    small = torch.arange(600, dtype=torch.bfloat16).reshape(2, 3, 100)
    big = torch.randn(10_007, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), dict(small=small, big=big))
    a_small, a_big = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert a_small.dtype == np.float32 and np.array_equal(a_small, small.float().numpy())        # written whole
    assert a_big.dtype == np.float32 and a_big.shape == (1000,)                                   # a sample
    assert np.array_equal(a_big, np.load(tmp_path / "b" / "big.npy"))
    assert np.isin(a_big, big.float().numpy()).all() and len(np.unique(a_big)) == 1000            # distinct elements
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES


def test_reference_arm_other_ranks_exit_silently():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--impl", "reference"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, RANK="1"))
    assert res.returncode == 0 and res.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_prints_the_contract_line(tmp_path):
    d = _run(["--steps", "2", "--warmup", "3", "--dump-outputs", str(tmp_path / "a")])
    sample = np.load(tmp_path / "a" / "sample.npy")
    assert sample.dtype == np.float32 and sample.ndim == 5 and np.isfinite(sample).all()
    # seeded inputs and weights: another run, with another step count, computes the same step.  Bitwise equality is a
    # deliberate contract (the dumps exist to compare builds output for output): the kernels use no floating-point
    # atomics; the attention kernel's dynamic work queue only decides which CTA computes an item, and each output
    # element comes from one item's fixed-order reduction.  A split reduction must keep that property.
    _run(["--steps", "1", "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "b")])
    assert np.array_equal(sample, np.load(tmp_path / "b" / "sample.npy"))
    assert BASE_KEYS | {"roofline", "cpu_baseline", "clocks"} <= set(d)
    assert d["metric"] == "dit_denoise_step_ms" and d["dtype"] == "bf16" and d["n_gpus"] == 1
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and r["peak"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    rr = d["roofline"]
    assert rr["cross_attention"]["launches_per_step"] > 0 and rr["launches_per_step"] > 0
    fl = d["attn_flops_per_step"]
    assert abs(fl["library_counter"] - fl["closed_form"]) <= 1e-6 * fl["closed_form"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    lfl = d["like_for_like"]
    assert lfl["gpu_ms"] > 0 and lfl["gpu_e2e_ms"] > 0 and d["cpu_baseline"]["kind"] == "reference"
    if not ref_loader.available():
        # nothing timed under the reference's name; the same layer is checked against the reference's stored output
        # by test_gpu_parity.py::test_wan_processors_vs_reference
        assert d["cpu_baseline"]["available"] is False and d["cpu_baseline"]["value"] is None
        assert "reference not available" in d["cpu_baseline"]["reason"] and "parity" not in lfl
        return
    assert d["cpu_baseline"]["value"] > 0 and lfl["reference_cpu_ms"] == d["cpu_baseline"]["value"]
    assert lfl["parity"]["cosine"] >= 0.99
    # both arms print the SAME config (the reference arm runs "on your arm's config")
    ref = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert ref["config"] == d["config"] and ref["metric"] == d["metric"] and ref["unit"] == d["unit"]
