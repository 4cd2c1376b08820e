"""Checkpoint / export paths around the native rollout (SURVEY.md section 5 "checkpoint / resume"; ppo_asymmetry.py:369-393,
452-468): agent state dicts interchangeable with the reference's parameter names, TorchScript actor export, and the env-state
checkpoint (which the reference does not have) continuing bit-identically."""
import os

import numpy as np
import pytest
import torch


def _agent():
    from taco_b200.ppo import TorchActorCritic
    torch.manual_seed(3)
    return TorchActorCritic(26, 4, [64, 64], 26, 32, [64], lstm_layers=1)


def test_state_dict_round_trip_and_reference_parameter_names(tmp_path):
    from taco_b200.ppo import load_checkpoint, make_optimizer, save_checkpoint, PPOConfig
    a = _agent()
    names = set(a.state_dict())
    # the names nets_asymmetry.PPO_ActorCritic produces for this configuration (MLP.layers Sequential, nn.LSTM under .layers)
    assert {"log_std", "actor_mlp.layers.0.weight", "actor_mlp.layers.4.bias", "critic_encoder.layers.weight_ih_l0",
            "critic_encoder.layers.bias_hh_l0", "critic_mlp.layers.2.weight"} <= names
    p = str(tmp_path / "model_5_0.1.pt")
    save_checkpoint(p, a, para_only=True)                       # PPO.save(para_only=True): a bare state dict
    b = _agent()
    with torch.no_grad():
        for prm in b.parameters():
            prm.add_(1.0)
    assert load_checkpoint(p, b) is None
    for (k, v), (_, w) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(v, w), k
    # resumable form: optimiser moments and epoch come back too
    opt = make_optimizer(a, PPOConfig())
    a.evaluate(torch.randn(8, 1, 26), torch.randn(8, 5, 26), torch.randn(8, 4))[0].sum().backward()
    opt.step()
    p2 = str(tmp_path / "resume.pt")
    save_checkpoint(p2, a, optimizer=opt, epoch=17, para_only=False)
    c = _agent()
    opt_c = make_optimizer(c, PPOConfig())
    assert load_checkpoint(p2, c, optimizer=opt_c) == 17
    sa, sc = opt.state_dict()["state"], opt_c.state_dict()["state"]
    assert sa.keys() == sc.keys() and all(torch.equal(sa[k]["exp_avg_sq"], sc[k]["exp_avg_sq"]) for k in sa)


def test_reference_state_dict_loads_and_gives_the_reference_outputs(golden_dir, tmp_path):
    """State dicts in the reference's format load into TorchActorCritic and give the reference's own action mean and value.
    tests/golden/ppo_update.npz holds PPO_ActorCritic.state_dict() of the reference (plain_init__<key>): it must load with exactly
    its keys and shapes.  tests/golden/actor.npz and critic.npz hold weights, inputs and outputs of the reference's actor MLP /
    act() and LSTM critic (case a); under the reference's parameter names they must reproduce those outputs."""
    from taco_b200.ppo import TorchActorCritic, load_checkpoint
    z = np.load(os.path.join(golden_dir, "ppo_update.npz"))
    ref_sd = {k[len("plain_init__"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("plain_init__")}
    p = str(tmp_path / "ref_model.pt")
    torch.save(ref_sd, p)
    ours = TorchActorCritic(26, 4, [32, 24], 26, 16, [20])
    assert load_checkpoint(p, ours) is None                    # strict load_state_dict: no missing or unexpected key
    got = ours.state_dict()
    assert got.keys() == ref_sd.keys() and all(torch.equal(got[k], ref_sd[k]) for k in ref_sd)
    a, c = np.load(os.path.join(golden_dir, "actor.npz")), np.load(os.path.join(golden_dir, "critic.npz"))
    sd = {"log_std": a["log_std"]}
    for i in range(3):
        sd[f"actor_mlp.layers.{2 * i}.weight"], sd[f"actor_mlp.layers.{2 * i}.bias"] = a[f"w{i}"], a[f"b{i}"]
        sd[f"critic_mlp.layers.{2 * i}.weight"], sd[f"critic_mlp.layers.{2 * i}.bias"] = c[f"a_w{i}"], c[f"a_b{i}"]
    for nm in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
        sd[f"critic_encoder.layers.{nm}_l0"] = c[f"a_{nm}_l0"]
    p2 = str(tmp_path / "ref_model_2.pt")
    torch.save({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, p2)
    ours = TorchActorCritic(26, 4, [64, 128], 26, 48, [64, 32])
    load_checkpoint(p2, ours)
    with torch.no_grad():
        m = ours(torch.from_numpy(a["obs"]))
        v = ours.critic_mlp(ours.critic_encoder(torch.from_numpy(c["a_states"])))
    for want in (a["mean"], a["act_mean"]):
        assert torch.allclose(m, torch.from_numpy(want), atol=1e-6)
    for want in (c["a_value"], c["a_act_value"]):
        assert torch.allclose(v, torch.from_numpy(want), atol=1e-6)


def test_export_actor_torchscript(tmp_path):
    from taco_b200.ppo import export_actor
    a = _agent()
    p = str(tmp_path / "actor_0.pt")
    eager, traced = export_actor(a, p, 1, 26, device="cpu")
    assert torch.equal(eager, traced)
    mod = torch.jit.load(p)
    x = torch.randn(5, 1, 26)
    with torch.no_grad():
        assert torch.allclose(mod(x), a(x), atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("task,dr", [("flip", False), ("mix", True)])
def test_env_state_checkpoint_continues_bit_identically(task, dr, tmp_path):
    import taco_b200
    cfg = taco_b200.make_cfg(task, 1000, domain_randomization=dr, observation_noise=dr, **{"env.maxEpisodeLength": 12})
    a = taco_b200.FpvVecTask(cfg, seed=11)
    a.reset()
    for t in range(9):
        a.step(a.random_actions(t))
    a.difficulty = 0.6
    path = str(tmp_path / "env.npy")
    a.save_state(path)
    want = []
    for t in range(9, 16):
        o, r, x, e = a.step(a.random_actions(t))
        want.append((o["obs"].clone(), o["states"].clone(), r.clone(), x.clone(), e["time_outs"].clone()))
    stats_a = a.stats().cpu()
    b = taco_b200.FpvVecTask(cfg, seed=999)                     # other seed / difficulty: both come from the checkpoint
    b.load_state(path)
    assert b.step_count == 9 and b.difficulty == pytest.approx(0.6)
    for t, w in zip(range(9, 16), want):
        o, r, x, e = b.step(b.random_actions(t))
        got = (o["obs"], o["states"], r, x, e["time_outs"])
        for g_, w_ in zip(got, w):
            assert torch.equal(g_, w_), t
    assert torch.equal(b.stats().cpu(), stats_a)
    assert np.array_equal(a.export_state(), b.export_state())
    with pytest.raises(RuntimeError):                           # a checkpoint of another configuration is refused
        c = taco_b200.FpvVecTask(taco_b200.make_cfg(task, 1001), seed=1)
        c.load_state_checkpoint(np.load(path))
    a.close(); b.close()
