"""bench.py --dump-outputs: the arrays it writes are what the last timed step computed (the same reset + rollout through the public API
reproduces them bit for bit), they are float32 / float64 and within 64 MB, and two runs with the same arguments write the same arrays."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
N, T, SLOTS, STEPS = 8192, 300, 16, 2      # one step writes N*T transitions, more than the ring holds: the ring is the last step's
ARGS = ["--steps", str(STEPS), "--warmup", "1", "--envs-per-gpu", str(N), "--horizon", str(T), "--ring-slots", str(SLOTS),
        "--skip-ddpg", "--skip-cpu-baseline"]


def run_bench(d):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + ["--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert len(out.stdout.strip().splitlines()) == 1
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_are_the_last_timed_step(sb, tmp_path):
    a, b = run_bench(tmp_path / "a"), run_bench(tmp_path / "b")
    assert sorted(a) == sorted(b) and sum(x.nbytes for x in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert a[k].tobytes() == b[k].tobytes(), k
    env = sb.Shems(T, sb.series.synth_charger98(T + 1, seed=98), n_envs=N)
    mem = sb.Replay(N * SLOTS)
    seed = 1000 + STEPS - 1                 # the seed of bench.py's last timed step
    env.reset(rng=seed)
    out = env.rollout(sb.POLICY_RANDOM, T, seed=seed, replay=mem, want_return=True)
    envs = a["env_ids"].astype(np.int64)
    assert len(envs) == N
    np.testing.assert_array_equal(out["ep_return"].cpu().numpy()[envs], a["ep_return"])
    np.testing.assert_array_equal(env.state[:, envs], a["state"])
    np.testing.assert_array_equal(env.idx[envs], a["state_idx"])
    rows = a["replay_rows"].astype(np.int64)
    assert len(rows) == N * SLOTS
    for name, x in zip(("replay_s", "replay_a", "replay_r", "replay_s2", "replay_done"), mem.get()):
        np.testing.assert_array_equal(x[..., rows], a[name], err_msg=name)
