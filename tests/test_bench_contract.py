"""bench.py's contract: the reference arm prints exactly one JSON line on stdout with the result keys (CPU), and --dump-outputs writes
what the timed episode computed (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-envs", "256"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["higher_is_better"] is True and line["scaling"] == "weak"
    assert "CliffordGym 8q" in line["metric"] and line["value"] > 0 and line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 0
    assert line["vs_baseline"] is None and line["data"] == "synthetic" and "workload" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "256 envs" in cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["unit"] == line["unit"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_oracle_episode(tmp_path):
    """--steps sets the timed launches, and --dump-outputs writes the last timed episode: at 256 environments the sample is the whole
    batch, and every array equals the CPU oracle's on the same seeded targets, actions and add_inverts coins."""
    import bench
    from oracle import oracle as orc
    from qiskit_gym_b200 import workloads as W
    argv = ["--steps", "3", "--warmup", "0", "--envs", "256", "--episode-steps", "24", "--add-inverts", "1", "--no-cpu-baseline", "--no-e2e",
            "--no-per-step", "--no-synth", "--no-packed", "--no-collector", "--dump-outputs", str(tmp_path)]
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout)
    assert line["steps"] == 3 and line["gpu_launches"] == 3 and line["engine_error_flags"] == 0

    args = bench.parse_args(argv)
    kind, n, gateset, kw = bench.workload(args)
    targets, actions, coins = bench.episode_inputs(args, args.envs)
    assert coins is not None
    cfg = orc.make_config(kind, n, gateset, max_depth=args.episode_steps, add_perms=False, **dict(kw, add_inverts=True))
    ref = orc.run_batch(cfg, targets, W.payload_lengths(kind, n, targets), actions, coins=coins)
    got = {name: np.load(tmp_path / f"{name}.npy") for name in ("obs", "mask", "reward", "done", "success")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got["obs"], ref["obs"].astype(np.float32))
    assert np.array_equal(got["reward"].view(np.uint32), ref["reward"].view(np.uint32))
    assert np.array_equal(got["done"], ref["done"].astype(np.float32)) and np.array_equal(got["success"], ref["success"].astype(np.float32))
    assert np.array_equal(got["mask"], np.repeat(1 - ref["success"][..., None], len(gateset), axis=2).astype(np.float32))
