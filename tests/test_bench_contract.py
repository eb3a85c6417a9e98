"""bench.py contract checks that run without a GPU: the reference arm prints one JSON line with the required keys, and
under torchrun-style env (RANK != 0) it exits 0 without work."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line(built):
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup",
                          "0", "--horizon", "5"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "robot-steps/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1 and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_dump_outputs_writes_every_scenario_or_a_seeded_sample_within_the_budget(tmp_path):
    import numpy as np
    import torch

    import bench
    B = 1000
    arrays = {"result": torch.arange(4 * B, dtype=torch.float32).reshape(4, B),
              "x_ee": torch.arange(9 * B, dtype=torch.float64).reshape(3, 3, B)}
    keep = np.setdiff1d(np.arange(B), [3, 500, 999])
    bench.dump_outputs(str(tmp_path / "all"), arrays, keep)
    assert np.array_equal(np.load(tmp_path / "all" / "scenario_index.npy"), keep)
    for name, t in arrays.items():
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, t[..., keep].float().numpy())
    budget = 3 * 128 + 100 * (8 + 4 * 4 + 4 * 9) + 50                       # room for 100 scenarios
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, keep, budget=budget)
    files = sorted((tmp_path / "a").iterdir())
    assert [f.name for f in files] == ["result.npy", "scenario_index.npy", "x_ee.npy"]
    assert sum(f.stat().st_size for f in files) <= budget
    idx = np.load(tmp_path / "a" / "scenario_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 100 and np.all(np.diff(idx) > 0) and np.isin(idx, keep).all()
    for name, t in arrays.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert np.array_equal(got, t[..., idx.astype(np.int64)].float().numpy())
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy"))


def test_calm_drops_the_scenarios_whose_horizon_blows_up(built):
    """Scenarios 772, 5278 and 8579 of the benchmark's batch (seed 0) blow up within the horizon (oracle O2 returns
    NaN); the first three stay calm."""
    import numpy as np

    import bench
    import multi_robot_fabrics_b200 as m
    rec = np.ascontiguousarray(m.scenarios.generate(65536, 3, seed=0), dtype=np.float32)
    assert bench.calm(rec[[0, 1, 2, 772, 5278, 8579]], 20).tolist() == [True, True, True, False, False, False]


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                          str(tmp_path)], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--impl ours only" in out.stderr


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""
