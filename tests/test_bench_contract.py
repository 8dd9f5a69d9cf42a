"""bench.py's output contract, checked without a GPU: (1) the `--impl reference` arm (CPU oracle port, the one arm that runs here)
prints ONE JSON line with the keys the driver parses; (2) the device arm refuses to run without CUDA (there is no CPU fallback to time
by accident); (3) the committed line of the final single-GPU run carries every key of the contract; (4) --dump-outputs, on the host
and (marked gpu) end to end through the device arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
             "data", "config", "e2e", "cpu_baseline")


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"], env={"THB_BENCH_CPU_ITEMS": "2"})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and all(k in d for k in BASE_KEYS)
    assert d["value"] > 0 and d["higher_is_better"] is True and d["scaling"] == "strong" and d["dtype"] == "f64"
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 2 and "2 of 4096" in d["cpu_baseline"]["sample"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_device_arm_does_not_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-c2"], timeout=300)
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]      # no number is printed
    assert "NVIDIA" in r.stderr or "CUDA" in r.stderr or "cuda" in r.stderr


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_writes_seeded_float64_sample(tmp_path):
    """--dump-outputs on the optimizer's own info type: float64 .npy files, the same item sample on every run, the poses of exactly those
    items, every per-item field of the info, and at the headline size (4096 items x 2 500 poses) no more than 64 MB in all."""
    import numpy as np
    import torch
    from theseus_b200.optimizer import NonlinearOptimizerInfo, NonlinearOptimizerStatus as S
    bench = _bench_module()
    B, names = 300, [f"P{i}" for i in range(5)]
    gen = torch.Generator().manual_seed(0)
    values = {n: torch.randn(B, 3, 4, generator=gen, dtype=torch.float64) for n in names}
    status = np.array([S.CONVERGED, S.MAX_ITERATIONS, S.FAIL] * (B // 3))
    info = NonlinearOptimizerInfo(best_solution=None, status=status, converged_iter=torch.arange(B) % 11, best_iter=torch.arange(B) % 7,
                                  err_history=None, last_err=torch.rand(B, generator=gen, dtype=torch.float64), best_err=None, state_history=None)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), values, info, names)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["best_iter.npy", "converged_iter.npy", "last_err.npy", "poses_sample.npy", "poses_sample_items.npy", "status.npy"]
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b), f
    items = np.load(tmp_path / "a" / "poses_sample_items.npy").astype(np.int64)
    assert len(items) == bench.DUMP_ITEMS and len(np.unique(items)) == len(items) and items.max() < B
    poses = np.load(tmp_path / "a" / "poses_sample.npy")
    np.testing.assert_array_equal(poses, np.stack([values[n].numpy()[items] for n in names], 1))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "last_err.npy"), info.last_err.numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "converged_iter.npy"), np.arange(B) % 11)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "best_iter.npy"), np.arange(B) % 7)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "status.npy"), np.array([1.0, 2.0, -1.0] * (B // 3)))
    full = 8 * (bench.DUMP_ITEMS * bench.C5_RINGS * bench.C5_PER_RING * 12 + 5 * 4096)
    assert full <= 64 * 2 ** 20


@pytest.mark.gpu
def test_device_arm_dumps_what_its_last_timed_step_returned(tmp_path):
    """bench.py --dump-outputs end to end on a small batch of the headline workload: the files of the last timed step, consistent with
    the JSON line the same run prints (final error); LM with tolerances 0 ends every item at the iteration limit (status 2, converged_iter
    -1 as in the reference)."""
    import numpy as np
    bench = _bench_module()
    B = 12
    r = _run(["--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-c2", "--dump-outputs", str(tmp_path)],
             env={"THB_BENCH_C5_BATCH": str(B)}, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert d["steps"] == 2 and d["e2e"]["steps"] == 2
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(got) == ["best_iter", "converged_iter", "last_err", "poses_sample", "poses_sample_items", "status"]
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["last_err"].shape == (B,) and np.isclose(got["last_err"].mean(), d["final_err_mean"], rtol=1e-12)
    assert np.all(got["status"] == 2.0) and np.all(got["converged_iter"] == -1.0)
    np.testing.assert_array_equal(got["poses_sample_items"], np.arange(B))
    P = got["poses_sample"]
    assert P.shape == (B, bench.C5_RINGS * bench.C5_PER_RING, 3, 4) and np.all(np.isfinite(P))
    R = P[..., :3]
    np.testing.assert_allclose(R @ np.swapaxes(R, -1, -2), np.broadcast_to(np.eye(3), R.shape), atol=1e-9)   # solutions are SE3 poses


def test_committed_final_line_has_every_contract_key():
    d = json.loads(open(os.path.join(ROOT, "profiles", "r02n_bench_n1_line_final.json")).read())
    for k in BASE_KEYS + ("clocks", "gpu_launches", "roofline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["gpu_launches"] > 0 and d["vs_baseline"] is None
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["e2e"]["value"] < d["value"]                                         # copies inside the timed region cost something
    rf = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(rf) and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"]) and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert d["parity"]["ok"] is True
