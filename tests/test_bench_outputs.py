"""bench.py --dump-outputs: the files hold what the timed path (rbg_connector_rollout_random) computed in its last
timed step, and the oracle reproduces them from the same seeded inputs after burn-in + warm-up + exactly --steps steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_are_the_last_timed_step(rbg, orc, tmp_path):
    G, N, B, time_limit = 10, 5, 1024, 50
    burnin, warmup, steps = 7, 3, 27  # 27 timed steps = one 20-step rollout call + one of 7 steps
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup), "--burnin", str(burnin), "--envs", str(B),
                        "--skip-e2e", "--skip-secondary", "--skip-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["gpu_launches"] == 2, line

    rst, _ = orc.connector_reset_batch("parallel_random_walk", orc.split(orc.PRNGKey(0), B), G, N)
    for _ in range(burnin + warmup + steps):
        act = orc.random_actions_batch(rst)
        rst, rts = orc.connector_step_batch(rst, act, time_limit=time_limit, autoreset_kind="parallel_random_walk")
    want = {
        "env_index": np.arange(B), "observation_grid": rts["obs"], "observation_action_mask": rts["action_mask"], "observation_step_count": rts["obs_step_count"],
        "reward": rts["reward"], "discount": rts["discount"], "step_type": rts["step_type"], "num_connections": rts["num_connections"],
        "ratio_connections": rts["ratio_connections"], "total_path_length": rts["total_path_length"], "action": act,
        "state_grid": rst["grid"], "state_step_count": rst["step_count"], "state_key": rst["key"],
        "agent_id": rst["agent_id"], "agent_start": rst["start"], "agent_target": rst["target"], "agent_position": rst["position"],
    }
    assert sorted(f[:-4] for f in os.listdir(tmp_path)) == sorted(want)
    for name, ref in want.items():
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == (np.float64 if name in ("env_index", "state_key") else np.float32), name
        assert got.shape == ref.shape and np.array_equal(got, ref.astype(got.dtype)), name
