"""The native PPO update (taco_ppo_*, taco_b200/ppo_native.py): tcgen05 GEMM forward / backward, device-side KL early stop,
gradient clipping, Adam and the spectral projection.  GPU only.

Bars:
  * the GEMM kernel itself (TMA tensor maps, split-K, ragged M / N / K): <= 2e-6 of the largest output against fp32 matmul of
    the same bf16 operands;
  * forward (action mean, value), losses and approx KL of a minibatch: <= 2e-3 absolute / 1e-3 relative against the fp32
    PyTorch twin (``TorchActorCritic.evaluate``, itself pinned to the reference);
  * gradients: <= 1e-2 of every tensor's norm against the bf16-operand emulation of the same arithmetic (oracle/ppo_bf16.py),
    whose back-propagation formulas equal autograd to 1e-6 when the rounding is switched off (checked here on the CPU).  Against
    fp32 autograd the same gradients differ by 4-9 % of a tensor's norm: ReLU masks flip wherever a pre-activation is within bf16
    rounding of zero (~0.4 % of the units); the emulation shows the same figure, so it is a property of bf16 operands, not of
    the kernels;
  * a whole update against the reference's own ``PPO.update`` (tests/golden/ppo_update_native.npz, generated from the imported
    reference class): logged losses / KL <= 2e-3 relative, optimiser step count equal, and the parameter update (final - init)
    points the same way: cosine >= 0.9 per network, >= 0.97 over all parameters (Adam turns a gradient into lr * sign-like
    steps, so an element whose gradient is near zero can move the other way; the fp32 twin in taco_b200.ppo reproduces the same
    golden to 2e-5 and stays the parity path);
  * the KL early stop leaves the parameters untouched and reports the stop, like ppo_asymmetry.py:223-226.
"""
import ctypes as C
import os
import types

import numpy as np
import pytest
import torch


def test_emulation_backprop_equals_autograd_without_rounding():
    """CPU: oracle/ppo_bf16.py with the bf16 rounding replaced by the identity == autograd of taco_b200.ppo's loss."""
    import oracle.ppo_bf16 as pb
    from taco_b200.ppo import TorchActorCritic
    torch.manual_seed(0)
    agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32])
    with torch.no_grad():
        agent.log_std.fill_(-0.3)
    B = 256
    obs, states, act = torch.randn(B, 1, 26) * 0.7, torch.randn(B, 5, 26) * 0.7, torch.randn(B, 4).clamp(-1.5, 1.5)
    adv, ret = torch.randn(B), torch.randn(B) * 0.5
    with torch.no_grad():
        old = agent.evaluate(obs, states, act)[0] + 0.1 * torch.randn(B)
    logp, ent, value, mean, _ = agent.evaluate(obs, states, act)
    ratio = torch.exp(logp - old)
    loss = -torch.min(adv * ratio, adv * torch.clamp(ratio, 0.8, 1.2)).mean() + 0.5 * torch.nn.functional.mse_loss(ret.view(-1, 1), value) \
        + 0.01 * (-ent.mean())
    loss.backward()
    keep, pb.r = pb.r, (lambda x: x)
    try:
        g, _ = pb.minibatch_grads(agent, obs, states, act, old, adv, ret, 0.2, 1.0, 0.5, 0.01)
    finally:
        pb.r = keep
    for n, prm in agent.named_parameters():
        assert float((g[n] - prm.grad).norm() / (prm.grad.norm() + 1e-12)) <= 5e-6, n


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,k,splits", [(4096, 256, 256, 1), (300, 48, 96, 1), (256, 32, 8192, 16), (4, 256, 4096, 37), (1000, 16, 16, 1),
                                          (256, 96, 5120, 20), (128, 256, 64, 1), (70000, 64, 256, 1)])
def test_gemm_kernel_against_matmul(m, n, k, splits):
    from taco_b200.ppo_native import gemm_selftest
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    a = (torch.randn(m, k, device="cuda", generator=g) * 0.5).bfloat16()
    b = (torch.randn(n, k, device="cuda", generator=g) * 0.5).bfloat16()
    d = gemm_selftest(a, b, splits)
    ref = a.float() @ b.float().T
    assert float((d - ref).abs().max() / ref.abs().max()) <= 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,k,splits", [(256, 256, 4096, 8), (256, 32, 8192, 16), (64, 96, 5120, 20), (256, 64, 65536, 74), (48, 256, 640, 3),
                                          (128, 16, 64, 1), (16, 8, 136, 1), (296, 72, 1000, 5)])
def test_gemm_kernel_transposed_operands(m, n, k, splits):
    """The MN-major operand mode (weight gradients dW = dZ^T X straight from the batch-major tensors)."""
    from taco_b200.ppo_native import gemm_selftest
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    at = (torch.randn(k, m, device="cuda", generator=g) * 0.5).bfloat16()
    bt = (torch.randn(k, n, device="cuda", generator=g) * 0.5).bfloat16()
    d = gemm_selftest(at, bt, splits, transposed=True)
    ref = at.float().T @ bt.float()
    assert float((d - ref).abs().max() / ref.abs().max()) <= 2e-6


def _hyper(cfg, lr, lip):
    from taco_b200 import _capi
    return _capi.TacoPPOHyper(lr=lr, clip=cfg.clip, target_kl=cfg.target_kl, max_grad=cfg.max_grad, pi_coef=cfg.pi_coef, vf_coef=cfg.vf_coef,
                              ent_coef=cfg.ent_coef, lipschitz=lip, use_lipschitz=1 if cfg.use_lipschitz else 0, world=1)


@pytest.mark.gpu
@pytest.mark.parametrize("actor_hidden,critic_hidden,n_total,batch", [([64, 48], [32], 1024, 256), ([256, 256, 256], [256, 256, 256], 8192, 4096)])
def test_forward_losses_and_gradients_of_one_minibatch(actor_hidden, critic_hidden, n_total, batch):
    import oracle.ppo_bf16 as pb
    from taco_b200 import _capi
    from taco_b200.ppo import PPOConfig, TorchActorCritic
    from taco_b200.ppo_native import NativePPO
    torch.manual_seed(1)
    agent = TorchActorCritic(26, 4, actor_hidden, 26, 64, critic_hidden).cuda()
    with torch.no_grad():
        agent.log_std.fill_(-0.3)
    gen = torch.Generator(device="cuda").manual_seed(1)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    obs, states, act = rnd(n_total, 1, 26) * 0.7, rnd(n_total, 5, 26) * 0.7, rnd(n_total, 4).clamp(-1.5, 1.5)
    adv, ret = rnd(n_total), rnd(n_total) * 0.5
    with torch.no_grad():
        old_logp = agent.evaluate(obs, states, act)[0] + 0.1 * rnd(n_total)
    idx = torch.randperm(n_total, device="cuda", generator=gen)[:batch]
    cfg = PPOConfig(target_kl=1e9, ent_coef=0.01)
    nat = NativePPO(agent, batch)
    nat._create(5)
    hy = _hyper(cfg, 1e-3, 4.0)
    L, s, p = nat._lib, nat._stream(), (lambda t: C.c_void_p(t.data_ptr()))
    _capi.check(L.taco_ppo_begin_update(nat._h, s), "begin")
    _capi.check(L.taco_ppo_forward_loss(nat._h, C.byref(hy), p(obs.reshape(n_total, -1)), p(states), p(act), p(old_logp), p(adv), p(ret), p(idx), s), "fwd")
    torch.cuda.synchronize()
    sums = nat.loss_sums.clone()
    _capi.check(L.taco_ppo_decide(nat._h, C.byref(hy), s), "decide")
    _capi.check(L.taco_ppo_backward(nat._h, s), "bwd")
    torch.cuda.synchronize()
    mean_n, value_n = nat.debug_outputs()
    # ---- forward and losses against the fp32 twin
    with torch.no_grad():
        logp, ent, value, mean, _ = agent.evaluate(obs[idx], states[idx], act[idx])
        ratio = torch.exp(logp - old_logp[idx])
        sur = -torch.min(adv[idx] * ratio, adv[idx] * torch.clamp(ratio, 1 - cfg.clip, 1 + cfg.clip)).mean()
        vl = torch.nn.functional.mse_loss(ret[idx].view(-1, 1), value)
        kl = ((ratio - 1) - (logp - old_logp[idx])).mean()
    assert float((mean_n - mean).abs().max()) <= 2e-3 and float((value_n - value.view(-1)).abs().max()) <= 2e-3
    assert float(sums[0] / batch) == pytest.approx(float(sur), rel=5e-3, abs=2e-5)
    assert float(sums[1] / batch) == pytest.approx(float(vl), rel=1e-3)
    assert float(sums[2] / batch) == pytest.approx(float(kl), rel=5e-3, abs=1e-6)
    # ---- gradients against the bf16-operand emulation
    g, st = pb.minibatch_grads(agent, obs[idx], states[idx], act[idx], old_logp[idx], adv[idx], ret[idx], cfg.clip, cfg.pi_coef, cfg.vf_coef, cfg.ent_coef)
    assert float((mean_n - st["mean"]).abs().max()) <= 2e-4 and float((value_n - st["value"]).abs().max()) <= 2e-4
    views = nat._views(nat.grad)
    worst = {n: float((views[n] - g[n]).norm() / (g[n].norm() + 1e-12)) for n in g}
    assert max(worst.values()) <= 1e-2, worst
    nat.close()


def _golden(tag):
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ppo_update_native.npz"))
    # what the "lip" case shares with the "plain" case (initial weights, buffer, minibatches, epoch) is stored once, under plain_
    gg = {k[len("plain_"):]: torch.from_numpy(np.asarray(z[k])) for k in z.files if k.startswith("plain_")}
    gg.update({k[len(tag) + 1:]: torch.from_numpy(np.asarray(z[k])) for k in z.files if k.startswith(tag + "_")})
    init = {k[6:]: v for k, v in gg.items() if k.startswith("init__")}
    final = {k[7:]: v for k, v in gg.items() if k.startswith("final__")}
    buf = types.SimpleNamespace(**{k[5:]: v.cuda() for k, v in gg.items() if k.startswith("buf__")})
    log = {k[5:]: float(v) for k, v in gg.items() if k.startswith("log__")}
    return gg, init, final, buf, log


def _golden_cfg(use_lip, target_kl=0.5):
    from taco_b200.ppo import PPOConfig
    return PPOConfig(clip=0.2, target_kl=target_kl, max_grad=0.5, epochs=40, train_iters=2, lr=1e-3, pi_coef=1.0, vf_coef=0.5, ent_coef=0.01,
                     lr_ratio=0.3, lr_lp_index=0.7, lr_epoch_index=30, use_lipschitz=use_lip, lipschitz_para=2.0,
                     lip_ratio=[1.0, 0.3], lip_lp_index=[0.3, 0.7], lip_epoch_index=[5, 30], diff_value=[0.1, 1.0],
                     diff_lp_index=[0.3, 0.7], diff_epoch_index=[5, 30])


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["plain", "lip"])
def test_update_against_the_reference_update(tag):
    from taco_b200.ppo import TorchActorCritic
    from taco_b200.ppo_native import NativePPO
    gg, init, final, buf, log = _golden(tag)
    agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32])
    agent.load_state_dict(init)
    agent.cuda()
    idx = [row.tolist() for row in gg["idx"]]
    env = types.SimpleNamespace(difficulty=0.0)
    nat = NativePPO(agent, len(idx[0]))
    out = nat.update(buf, _golden_cfg(tag == "lip"), int(gg["epoch"]), env=env, batch_idx=idx)
    nat.store_to(agent)
    assert out["optim_steps"] == int(gg["optim_step"]) and not out["early_stop"]
    assert abs(env.difficulty - float(gg["difficulty"])) < 1e-6
    for name in ("policy_gradient_loss", "value_loss", "entropy_loss", "sum_loss", "approx_kl", "learning_rate", "lipschitz_para", "mean_value", "explained_variance"):
        assert out[name] == pytest.approx(log[name], rel=2e-3, abs=2e-5), name
    sd = {k: v.cpu() for k, v in agent.state_dict().items()}
    cos = lambda keys: float(torch.nn.functional.cosine_similarity(torch.cat([(sd[k] - init[k]).flatten() for k in keys]),
                                                                   torch.cat([(final[k] - init[k]).flatten() for k in keys]), dim=0))
    groups = {"actor": [k for k in sd if k.startswith("actor_mlp")], "lstm": [k for k in sd if k.startswith("critic_encoder")],
              "critic": [k for k in sd if k.startswith("critic_mlp")], "all": list(sd)}
    cs = {g: cos(ks) for g, ks in groups.items()}
    assert min(cs["actor"], cs["lstm"], cs["critic"]) >= 0.9 and cs["all"] >= 0.97, cs
    if tag == "lip":                                                        # the projection bit: no actor matrix above the bound
        c = out["lipschitz_para"]
        for k in groups["actor"]:
            if sd[k].dim() == 2:
                assert float(torch.linalg.matrix_norm(sd[k], ord=2)) <= c * (1 + 2e-3), k
        sig_ref = [float(torch.linalg.matrix_norm(final[k], ord=2)) for k in groups["actor"] if final[k].dim() == 2]
        sig = [float(torch.linalg.matrix_norm(sd[k], ord=2)) for k in groups["actor"] if sd[k].dim() == 2]
        assert np.allclose(sig, sig_ref, rtol=5e-3)
    nat.close()


@pytest.mark.gpu
def test_kl_early_stop_is_decided_on_the_device():
    from taco_b200.ppo import TorchActorCritic
    from taco_b200.ppo_native import NativePPO
    gg, init, final, buf, log = _golden("plain")
    agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32])
    agent.load_state_dict(init)
    agent.cuda()
    idx = [row.tolist() for row in gg["idx"]]
    nat = NativePPO(agent, len(idx[0]))
    out = nat.update(buf, _golden_cfg(False, target_kl=1e-5), int(gg["epoch"]), batch_idx=idx)      # 1.5 * 1e-5 < the first minibatch's KL
    assert out["early_stop"] and out["optim_steps"] == 0 and len(out["log"]) == 1 and out["log"][0, 6] == 1.0
    nat.store_to(agent)
    for k, v in agent.state_dict().items():
        assert torch.equal(v.cpu(), init[k]), k
    # optimiser state round trip: Adam moments and step survive store_to / load_from
    out = nat.update(buf, _golden_cfg(False), int(gg["epoch"]), batch_idx=idx)
    assert out["optim_steps"] == 4
    from taco_b200.ppo import make_optimizer
    opt = make_optimizer(agent, _golden_cfg(False))
    nat.store_to(agent, opt)
    nat2 = NativePPO(agent, len(idx[0]))
    nat2._create(5)
    nat2.load_from(agent, opt)
    assert torch.equal(nat2.params, nat.params) and torch.equal(nat2.adam_m, nat.adam_m) and torch.equal(nat2.adam_v, nat.adam_v)
    assert int(nat2.step.item()) == 4
    nat.close(); nat2.close()
