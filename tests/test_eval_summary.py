"""Host side of the evaluation path (taco_b200.evaluate): per-task summaries of synthetic episode records and the trajectory files.
CPU only."""
import math
import os

import numpy as np
import pytest

from taco_b200 import evaluate as ev
from taco_b200 import _capi


def _records(task, ret, length, timed_out, **fields):
    r = np.zeros(len(ret), dtype=ev.EPISODE_DTYPE)
    r["task"], r["ret"], r["length"], r["timed_out"] = task, ret, length, timed_out
    for k, v in fields.items():
        r[k] = v
    return r


def test_record_dtype_matches_the_c_struct():
    assert ev.EPISODE_DTYPE.itemsize == 48 and ev.EPISODE_DTYPE.itemsize % 16 == 0
    offs = {n: ev.EPISODE_DTYPE.fields[n][1] for n in ev.EPISODE_DTYPE.names}
    assert offs == dict(env_id=0, end_step=8, length=12, task=16, timed_out=18, ret=20, pos_err_mean=24, pos_err_final=28,
                        tilt_max=32, speed_mean=36, angvel_max=40, roll_travel=44)


def test_summary_groups_by_task():
    rng = np.random.default_rng(0)
    pos = _records(0, rng.normal(30, 5, 200).astype(np.float32), rng.integers(10, 1000, 200), rng.random(200) < 0.7,
                   pos_err_mean=rng.random(200).astype(np.float32), tilt_max=rng.random(200).astype(np.float32),
                   speed_mean=rng.random(200).astype(np.float32), angvel_max=rng.random(200).astype(np.float32))
    flip = _records(2, rng.normal(10, 2, 50).astype(np.float32), np.full(50, 999), np.ones(50, bool),
                    roll_travel=np.full(50, 4 * math.pi, np.float32))
    recs = np.concatenate([flip[:20], pos, flip[20:]])
    s = ev.summarise_episodes(recs)
    assert set(s) == {"pos", "flip"}
    p = s["pos"]
    ret = pos["ret"].astype(np.float64)
    assert p["episodes"] == 200
    assert p["survival"] == pytest.approx(np.mean(pos["timed_out"] != 0))
    assert p["ret_mean"] == pytest.approx(ret.mean())
    for q in (5, 50, 95):
        assert p[f"ret_p{q}"] == pytest.approx(np.percentile(ret, q))
    assert p["length_mean"] == pytest.approx(pos["length"].mean())
    assert p["pos_err_mean"] == pytest.approx(pos["pos_err_mean"].astype(np.float64).mean())
    assert p["tilt_max_p95"] == pytest.approx(np.percentile(pos["tilt_max"].astype(np.float64), 95))
    assert p["speed_mean"] == pytest.approx(pos["speed_mean"].astype(np.float64).mean())
    assert p["angvel_max_mean"] == pytest.approx(pos["angvel_max"].astype(np.float64).mean())
    assert "flips_per_episode" not in p
    assert s["flip"]["episodes"] == 50 and s["flip"]["survival"] == 1.0
    assert s["flip"]["flips_per_episode"] == pytest.approx(2.0)
    assert ev.summarise_episodes(np.zeros(0, dtype=ev.EPISODE_DTYPE)) == {}


def test_save_trajectories_splits_at_resets(tmp_path):
    T, k = 12, 2
    data = np.zeros((T, k, 68), np.float32)
    data[:, :, ev.TRAJ_COLUMNS.index("pos_z")] = np.arange(T, dtype=np.float32)[:, None]
    data[:, :, 64:] = 0.25
    # env column 0: episodes of 4 and 5 steps, then 3 steps of one still running; column 1: starts mid-episode, ends at row 6
    prog0 = [1, 2, 3, 4, 1, 2, 3, 4, 5, 1, 2, 3]
    reset0 = [0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0]
    prog1 = [7, 8, 9, 10, 11, 12, 13, 1, 2, 3, 4, 5]
    reset1 = [0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1]
    data[:, 0, ev.TRAJ_COLUMNS.index("progress")] = prog0
    data[:, 0, ev.TRAJ_COLUMNS.index("reset")] = reset0
    data[:, 1, ev.TRAJ_COLUMNS.index("progress")] = prog1
    data[:, 1, ev.TRAJ_COLUMNS.index("reset")] = reset1
    traj = {"env_ids": np.array([3, 4100]), "local_ids": np.array([3, 4]), "step": np.arange(100, 100 + T, dtype=np.uint32), "data": data}
    out = ev.save_trajectories(traj, str(tmp_path / "traj"))
    names = sorted(os.path.basename(p) for p in out)
    assert names == sorted(f"{b}.{x}" for b in ("env3_ep0000", "env3_ep0001", "env3_ep0002_partial", "env4100_ep0000_partial",
                                                  "env4100_ep0001") for x in ("npy", "csv"))
    a = np.load(tmp_path / "traj" / "env3_ep0001.npy")
    assert a.dtype.names == tuple(["step"] + ev.TRAJ_COLUMNS) and len(ev.TRAJ_COLUMNS) == 68
    assert list(a["step"]) == [104, 105, 106, 107, 108] and list(a["progress"]) == [1, 2, 3, 4, 5]
    assert list(a["pos_z"]) == [4, 5, 6, 7, 8] and np.all(a["action_3"] == 0.25)
    b = np.load(tmp_path / "traj" / "env4100_ep0001.npy")
    assert list(b["step"]) == list(range(107, 112))
    lines = open(tmp_path / "traj" / "env3_ep0000.csv").read().splitlines()
    assert lines[0].split(",") == ["step"] + ev.TRAJ_COLUMNS
    assert len(lines) == 5 and lines[1].split(",")[0] == "100"
    assert float(lines[4].split(",")[1 + ev.TRAJ_COLUMNS.index("reset")]) == 1.0


def test_state_columns_follow_the_export_layout():
    assert len(ev.STATE_COLUMNS) == _capi.STATE_WORDS
    assert ev.STATE_COLUMNS[21] == "roll_continuous" and ev.STATE_COLUMNS[34] == "progress" and ev.STATE_COLUMNS[38] == "reset"
