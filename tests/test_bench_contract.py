"""bench.py's output contract, as far as it can be exercised without a GPU: the reference arm prints exactly
ONE JSON line on stdout with the keys the driver reads."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(args, extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    proc = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True, env=env,
                          timeout=300, cwd=REPO)
    assert proc.returncode == 0, proc.stderr[-2000:]
    return proc.stdout


def run_reference(extra_env=None, extra_args=()):
    return run_bench(["--impl", "reference", "--nx", "32", "--ny", "32", "--steps", "2", "--warmup", "1", *extra_args], extra_env)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = [ln for ln in run_reference().splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["vs_baseline"] is None
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config"):
        assert key in line, key
    assert line["unit"] == "elements/s" and line["dtype"] == "f64" and "workload" in line["config"]
    assert line["value"] > 0 and line["steps"] == 2 and line["warmup"] == 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    baseline = line["cpu_baseline"]
    assert baseline["kind"] in ("port", "reference") and baseline["cores"] >= 1 and baseline["value"] == line["value"]
    assert "sample" in baseline


def test_reference_arm_runs_on_rank_zero_only():
    # under torchrun the other ranks exit 0 without work and without output
    assert run_reference({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}).strip() == ""


def test_steps_below_one_are_refused():
    proc = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "0"],
                          capture_output=True, text=True, timeout=300, cwd=REPO)
    assert proc.returncode != 0 and "--steps" in proc.stderr and proc.stdout == ""


def test_reference_arm_dumps_its_outputs(tmp_path):
    """--dump-outputs: the CSR values and load vector of the CPU port, identical from run to run.  The expected arrays
    come from the same CPU port, so this checks the plumbing; the GPU test below checks the GPU arms against this dump."""
    from oracle.torch_cpu_port import reference_assembly_cpu
    from pytorch_fem_solver_b200 import meshgen

    first, second = tmp_path / "a", tmp_path / "b"
    for out in (first, second):
        assert len(run_reference(extra_args=("--dump-outputs", str(out))).strip().splitlines()) == 1
    mesh = meshgen.structured_rectangle(32, 32, jitter=0.25, seed=1234, topology=False)
    matrix, load = reference_assembly_cpu(torch.from_numpy(mesh["vertices"]), torch.from_numpy(mesh["triangles"]), 3)
    expected = {"csr_values": matrix.values().numpy(), "load": load.numpy().reshape(-1)}
    assert sorted(os.listdir(first)) == ["csr_values.npy", "load.npy"]
    for name, ref in expected.items():
        a, b = np.load(first / f"{name}.npy"), np.load(second / f"{name}.npy")
        assert a.dtype == np.float64 and a.shape == ref.shape
        assert np.array_equal(a, b)
        np.testing.assert_allclose(a, ref, rtol=1e-12, atol=1e-14 * np.abs(ref).max())


def test_dump_keeps_a_fixed_sample_of_large_outputs(tmp_path, monkeypatch):
    import bench

    monkeypatch.setattr(bench, "DUMP_MAX_ELEMENTS", 10)
    values, load = torch.arange(100, dtype=torch.float64), torch.arange(7, dtype=torch.float32).reshape(7, 1)
    for out in ("a", "b"):
        bench.dump_outputs(str(tmp_path / out), values, load)
    sample = np.load(tmp_path / "a" / "csr_values.npy")
    assert sample.dtype == np.float64 and sample.shape == (10,)
    assert np.all(np.diff(sample) > 0) and set(sample) <= set(range(100))  # distinct entries, in index order
    assert np.array_equal(sample, np.load(tmp_path / "b" / "csr_values.npy"))
    small = np.load(tmp_path / "a" / "load.npy")
    assert small.dtype == np.float64 and np.array_equal(small, np.arange(7.0))  # short arrays are written whole


def test_dump_of_two_large_outputs_stays_within_the_byte_budget(tmp_path):
    """Both arrays longer than the per-array cap (a mesh of more than DUMP_MAX_ELEMENTS vertices): the directory,
    .npy headers included, stays within DUMP_MAX_BYTES = 64 MB."""
    import bench

    assert bench.DUMP_MAX_BYTES <= 64_000_000
    values = torch.arange(bench.DUMP_MAX_ELEMENTS + 1_000_000, dtype=torch.float64)
    load = torch.arange(bench.DUMP_MAX_ELEMENTS + 300_000, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path), values, load)
    for name in ("csr_values", "load"):
        assert np.load(tmp_path / f"{name}.npy").shape == (bench.DUMP_MAX_ELEMENTS,)
    assert sum(os.path.getsize(tmp_path / name) for name in os.listdir(tmp_path)) <= bench.DUMP_MAX_BYTES


@pytest.mark.gpu
@pytest.mark.parametrize("path,kernels_per_step", [("tiled", 1), ("two_pass", 3)])
def test_gpu_arm_dumps_what_the_reference_computes(tmp_path, path, kernels_per_step):
    """The GPU arm runs exactly --steps timed steps and dumps the same CSR values and load as the CPU port."""
    size = ["--nx", "48", "--ny", "32"]
    run_reference(extra_args=(*size, "--dump-outputs", str(tmp_path / "ref")))
    out = run_bench([*size, "--path", path, "--steps", "4", "--warmup", "1", "--no-cpu-baseline", "--no-e2e",
                     "--dump-outputs", str(tmp_path / "ours")])
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    line = json.loads(lines[0])
    assert line["steps"] == 4 and line["gpu_launches"] == 4 * kernels_per_step
    for name in ("csr_values", "load"):
        ours, ref = np.load(tmp_path / "ours" / f"{name}.npy"), np.load(tmp_path / "ref" / f"{name}.npy")
        assert ours.dtype == np.float64 and ours.shape == ref.shape
        np.testing.assert_allclose(ours, ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())
