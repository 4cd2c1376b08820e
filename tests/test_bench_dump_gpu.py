"""bench.py --dump-outputs: the files hold what the last of the --steps timed steps returned, at a fixed seeded sample of envs,
identically from run to run, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0x7AC0            # bench.py's SEED (bench.py is not imported: it redirects file descriptor 1 when loaded)
ONLY_MAIN = ["--no-e2e", "--no-small", "--no-extra-configs", "--no-actor", "--no-cpu-baseline"]
NAMES = ("env_index", "obs", "states", "rew", "reset", "time_outs", "rollout_stats")


def _bench(out_dir, n, steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup), "--envs-per-gpu", str(n),
           "--dump-outputs", str(out_dir)] + ONLY_MAIN
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_is_the_last_timed_step_and_repeats_exactly(tmp_path):
    import taco_b200
    n, steps, warmup = 100_000, 7, 5                 # more envs than bench.py dumps: the sampled path
    lines = [_bench(tmp_path / d, n, steps, warmup) for d in ("a", "b")]
    dumps = [{k: np.load(tmp_path / d / f"{k}.npy") for k in NAMES} for d in ("a", "b")]
    a, b = dumps
    assert all(line["steps"] == steps and line["dump_outputs"]["envs"] == len(a["env_index"]) for line in lines)
    assert sum(os.path.getsize(tmp_path / "a" / f"{k}.npy") for k in NAMES) <= 64 * 1024 * 1024
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    idx = a["env_index"].astype(np.int64)
    assert 0 < len(idx) < n and np.array_equal(idx, np.unique(idx)) and idx[-1] < n
    for k in NAMES:
        if k == "rollout_stats":                     # float64 sums over envs
            assert np.allclose(a[k], b[k], rtol=1e-12, atol=0), k
        else:
            assert np.array_equal(a[k], b[k]), k
    assert a["rollout_stats"][7] == n * steps        # env-steps of the timed window: --steps sets it
    # the same sequence in this process: warm-up, stats reset, then the timed steps; compare the last step's return values
    env = taco_b200.FpvVecTask(taco_b200.make_cfg("flip", n), "cuda:0", "cuda:0", -1, True, env_offset=0, num_envs_global=n, seed=SEED,
                               strict_fp=True)
    acts = [env.random_actions(t) for t in range(4)]
    for t in range(max(warmup, 3)):
        env.step(acts[t % 4])
    env.stats()
    for t in range(steps):
        obs, rew, reset, extras = env.step(acts[t % 4])
    sel = torch.from_numpy(idx).cuda()
    want = {"obs": obs["obs"][sel], "states": obs["states"][sel], "rew": rew[sel], "reset": reset[sel], "time_outs": extras["time_outs"][sel]}
    for k, v in want.items():
        assert np.array_equal(a[k], v.float().cpu().numpy()), k
    env.close()
