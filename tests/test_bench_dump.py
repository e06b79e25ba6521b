"""bench.py --dump-outputs: what the last timed step computed, written as .npy files that two builds can be compared by."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_last_step_outputs_sample_and_types():
    """Fixed seeded sample of envs for every per-env array, float32 / float64 only, within the size limit at full width."""
    import bench
    N = bench.DUMP_ENVS + 808
    g = torch.Generator().manual_seed(1)
    task = types.SimpleNamespace(
        num_envs=N, obs_buf=torch.rand(N, 1750, generator=g), rew_buf=torch.rand(N, generator=g),
        reset_buf=torch.randint(0, 2, (N,), generator=g), joint_position_targets=torch.rand(N, 4, generator=g),
        joint_velocity_targets=torch.rand(N, 6, generator=g),
        extras={"pos_reward": torch.rand(N, generator=g), "collision_penalty": torch.randint(0, 2, (N,), generator=g)})
    stats = torch.rand(16, dtype=torch.float64, generator=g)
    out = bench.last_step_outputs(task, stats)
    again = bench.last_step_outputs(task, stats)
    ids = out["env_ids"].astype(np.int64)
    assert ids.shape == (bench.DUMP_ENVS,) and (np.diff(ids) > 0).all() and ids[-1] < N
    assert np.array_equal(out["obs"], task.obs_buf.numpy()[ids]) and np.array_equal(out["rew"], task.rew_buf.numpy()[ids])
    assert np.array_equal(out["reset"], task.reset_buf.numpy()[ids]) and out["reset"].dtype == np.float64
    assert np.array_equal(out["extras_collision_penalty"], task.extras["collision_penalty"].numpy()[ids])
    assert out["joint_velocity_targets"].shape == (bench.DUMP_ENVS, 6) and np.array_equal(out["stats"], stats.numpy())
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert all(np.array_equal(out[k], again[k]) for k in out)
    assert sum(a.nbytes for a in out.values()) <= bench.DUMP_MAX_BYTES


def _bench(out_dir, steps, warmup):
    cmd = [sys.executable, BENCH, "--envs", "9000", "--length", "20", "--nv", "72", "--K", "64", "--stones", "100", "--no-cpu",
           "--steps", str(steps), "--warmup", str(warmup), "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_dump_is_reproducible_and_steps_are_timed(tmp_path):
    """4 warm-up + 2 timed steps and 3 + 3 reach the same state: every dumped array is identical, while the timed region of
    the second run holds one step more (--steps sets the timed steps, not only a label)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    a_line, a = _bench(tmp_path / "a", steps=2, warmup=4)
    b_line, b = _bench(tmp_path / "b", steps=3, warmup=3)
    assert a_line["steps"] == 2 and b_line["steps"] == 3
    assert b_line["gpu_launches"] * 2 == a_line["gpu_launches"] * 3
    assert sorted(a) == sorted(b) and {"obs", "rew", "reset", "env_ids", "stats"} <= set(a)
    assert a["obs"].shape == (8192, 1750) and a["rew"].shape == (8192,)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert (a["obs"][:, 4:] != 5.5).mean() > 0.5           # the rays do hit the terrain (11.0 / 2 is a miss)
