"""bench.py --dump-outputs: what the timed path computed, written as float arrays that two runs (or two builds) can be
compared on.  Same arguments -> the same arrays; --steps moves the step that is dumped."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--envs", "4096",
                        "--ppo-envs", "2048", "--ppo-iters", "1", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900, cwd=str(out_dir.parent))
    assert r.returncode == 0, r.stderr[-3000:]
    assert len([l for l in r.stdout.splitlines() if l.strip()]) == 1, r.stdout
    return {p[:-4]: np.load(os.path.join(out_dir, p)) for p in sorted(os.listdir(out_dir))}


def test_dump_outputs_reproducible_and_follow_steps(tmp_path):
    a, b, c = _bench_dump(tmp_path / "a", 5), _bench_dump(tmp_path / "b", 5), _bench_dump(tmp_path / "c", 6)
    assert a.keys() == b.keys() == c.keys()
    assert {"env_step_obs_car", "env_step_rewards", "env_step_done", "ppo_act", "ppo_actor_choice_params"} <= set(a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["env_step_obs_car"].shape[0] == 4096 and a["ppo_act"].shape == (80, 4, 1024)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert any(not np.array_equal(a[k], c[k]) for k in a if k.startswith("env_step_"))
