"""FpvVecTask as the observation storage of the reference's consumer: ``PPO.run`` of IsaacGymEnvs/algorithms/ppo_asymmetry.py
keeps the tensors ``reset()`` returns and reads them after ``env.step`` (rollout loop :286-393).  GPU only."""
import pytest

pytestmark = pytest.mark.gpu


def test_reset_returns_storage_the_env_never_overwrites():
    """PPO.run keeps reset()'s tensors as its own observation storage and reads them AFTER env.step
    (ppo_asymmetry.py:297-299,326-329); the reference returns fresh clamp() results (vec_task_asymmetry.py:358-359)."""
    import taco_b200
    env = taco_b200.FpvFlip(taco_b200.make_cfg("flip", 256), "cuda:0", "cuda:0", -1, True, False, False)
    d = env.reset()
    obs, states = d["obs"], d["states"]
    for t in range(3):
        env.step(env.random_actions(t))
    assert float(obs.abs().max()) == 0.0 and float(states.abs().max()) == 0.0
    env.close()

