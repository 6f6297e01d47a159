"""bench.py's JSON contract, checked on the CPU tier through the reference arm (the GPU arm needs a device): one JSON line
with the base keys, the same `metric` / `config` as the GPU arm, the `cpu_baseline` and `e2e` objects the tier asks for."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-sample-n", "512"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["vs_baseline"] is None
    assert d["dtype"] == "f64" and d["unit"] == "evals/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["sample_n"] == 512 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the reference arm runs on the GPU arm's workload description
    sys.path.insert(0, ROOT)
    import bench
    assert d["metric"] == bench.METRIC and d["config"] == bench.workload_config(32768, 1)
    assert "N=32768" in d["config"]["workload"] and "inputs_exceed_l2" in d["config"]["l2"]
    assert d["ms_per_step"] < d["ms_per_step_full_size_extrapolated"]


@pytest.mark.parametrize("args", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(args, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=300, cwd=tmp_path)
    assert out.returncode == 2 and "error:" in out.stderr, out.stderr[-2000:]
    assert not out.stdout.strip() and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: the loss and the three hyper-parameter gradients of the last timed step, float64, equal to the
    oracle's on the same seeded inputs (and to the reference's loss pin at this size); --steps is the timed step count."""
    sys.path.insert(0, ROOT)
    from oracle import gp_oracle as O
    n, dump = 2048, tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--num-points", str(n), "--steps", "2",
                          "--warmup", "1", "--no-cpu-baseline", "--no-vendor-baseline", "--no-sharded",
                          "--no-int8-sliced", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2
    got = {f[:-len(".npy")]: np.load(dump / f) for f in os.listdir(dump)}
    assert set(got) == {"loss", "kernel.variance.grad", "kernel.length_scales.grad", "likelihood.variance.grad"}
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["loss"].shape == (1,) and got["loss"][0] == line["loss"]
    assert abs(got["loss"][0] - -1420.2752146205817) <= 1e-9 * 1420.3          # BASELINE.md section 3 pin
    X, Y, _ = O.synth_regression(n, 8)
    ref_loss, ref = O.gpr_loss_and_grads("Rbf", X, Y, np.ones(8), 1.0, 0.01)
    rel = lambda a, b: float(np.abs(a - b).max() / np.abs(b).max())  # noqa: E731
    assert rel(got["loss"], ref_loss.numpy()) <= 1e-9
    assert rel(got["kernel.variance.grad"], ref["variance"].numpy()) <= 1e-7
    assert rel(got["kernel.length_scales.grad"], ref["length_scales"].numpy()) <= 1e-7
    assert rel(got["likelihood.variance.grad"], ref["noise"].numpy()) <= 1e-7


def test_sharded_bench_module_is_importable_without_a_gpu():
    sys.path.insert(0, ROOT)
    import bench_sharded
    assert bench_sharded.VFE_N == 10_000_000 and bench_sharded.VFE_M == 1024 and bench_sharded.SVGP_M == 2048
    assert bench_sharded.VFE_SHARDS % 8 == 0 and bench_sharded.C5_N == 131072
