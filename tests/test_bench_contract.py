"""bench.py's output contract on the CPU side: the reference arm prints exactly one JSON line on stdout
with the keys the driver reads, whatever libraries write to file descriptor 1 meanwhile."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent

REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"}


def run_reference(*extra):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample", "4", *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_prints_one_json_line(native):
    line = run_reference()
    assert REQUIRED <= set(line)
    assert line["impl"] == "reference" and line["unit"] == "solves/s" and line["higher_is_better"] is True
    assert line["metric"] == "batched OCP SQP solves/sec (H=20)" and "workload" in line["config"]
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1


def test_reference_arm_other_ranks_stay_silent(native, monkeypatch):
    monkeypatch.setenv("RANK", "1")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--cpu-sample", "4"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_workload_switch_changes_metric_and_config():
    import importlib
    sys.path.insert(0, str(ROOT))
    bench = importlib.import_module("bench")

    class Args:
        workload, batch = "cartpole", 0
    try:
        bench.select_workload(Args)
        assert bench.METRIC == "batched OCP SQP solves/sec (H=200)" and Args.batch == 592
        assert "cart-pole" in bench.workload_config(Args.batch, 1)["workload"]
    finally:
        Args.workload, Args.batch = "quadrotor", 0
        bench.select_workload(Args)
    assert bench.METRIC == "batched OCP SQP solves/sec (H=20)" and Args.batch == 4096


def test_dump_outputs_keeps_one_seeded_sample_under_the_limit(tmp_path, monkeypatch):
    import importlib
    sys.path.insert(0, str(ROOT))
    bench = importlib.import_module("bench")
    B, N = 1000, 20
    arrays = {"x": np.arange(B * N, dtype=np.float64).reshape(B, N), "f": np.arange(B, dtype=np.float64),
              "stats": np.ones((B, 12))}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    for k, a in arrays.items():
        assert np.array_equal(np.load(tmp_path / "all" / f"{k}.npy"), a)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted((tmp_path / "a").iterdir())
    assert [f.name for f in files] == ["f.npy", "stats.npy", "x.npy"]
    assert sum(f.stat().st_size for f in files) <= 100_000
    x, f = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "a" / "f.npy")
    assert x.dtype == np.float64 and 0 < f.size < B
    assert np.array_equal(x[:, 0], N * f)                  # the same instances in every array
    for k in arrays:                                       # and the same sample in every run
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy"))


def test_bench_builds_stage_libraries_outside_the_tree(native, tmp_path):
    """The tree bench.py runs from may be read-only: generated stage libraries go to a temporary directory, in which
    the ones build() left in the package are reused."""
    code_gen = ROOT / "optimal_control_problem_b200" / "share" / "code_gen"
    before = sorted(code_gen.iterdir()) if code_gen.exists() else []
    code = ("import sys; sys.path.insert(0, sys.argv[1]); import bench; bench.private_share_dir(); "
            "import optimal_control_problem_b200 as ocp; print(ocp.Problem('cartpole', horizon=2).model_library)")
    env = {k: v for k, v in os.environ.items() if k != "OCP_B200_SHARE_DIR"}
    r = subprocess.run([sys.executable, "-c", code, str(ROOT)], env=env, capture_output=True, text=True, timeout=600,
                       cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    lib = Path(r.stdout.split()[-1])
    assert ROOT not in lib.parents and not lib.exists()    # in the temporary directory, removed at exit
    assert (sorted(code_gen.iterdir()) if code_gen.exists() else []) == before
    assert list(tmp_path.iterdir()) == []
