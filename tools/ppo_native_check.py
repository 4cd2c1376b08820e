"""Diagnostics of the native PPO update on a GPU box: GEMM self-test, forward / gradient parity against PyTorch autograd,
the reference-generated golden update, and the update time at the reference's scale (4096 envs x 64 steps, 16 optimiser steps).
usage: python tools/ppo_native_check.py [--no-time]"""
import ctypes as C
import json
import os
import sys
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from taco_b200 import _capi  # noqa: E402
from taco_b200.ppo import PPOConfig, TorchActorCritic, make_optimizer, ppo_update  # noqa: E402
from taco_b200.ppo_native import NativePPO, gemm_selftest  # noqa: E402

out = {}
torch.manual_seed(0)
# ---------------------------------------------------------------- 1. GEMM
g = {}
for (m, n, k, sp) in ((4096, 256, 256, 1), (300, 48, 96, 1), (256, 32, 8192, 16), (4, 256, 4096, 37), (1000, 16, 16, 1), (256, 96, 5 * 1024, 20),
                      (65536, 256, 256, 1), (128, 256, 64, 1), (70000, 64, 256, 1)):
    a = (torch.randn(m, k, device="cuda") * 0.5).bfloat16()
    b = (torch.randn(n, k, device="cuda") * 0.5).bfloat16()
    d = gemm_selftest(a, b, sp)
    ref = a.float() @ b.float().T
    g[f"{m}x{n}x{k}/{sp}"] = float((d - ref).abs().max() / ref.abs().max())
out["gemm_rel_err"] = g
print(json.dumps(out), flush=True)


# ---------------------------------------------------------------- 2. forward / gradient parity on a random minibatch
def hyper(cfg, lr, lip, world=1):
    return _capi.TacoPPOHyper(lr=lr, clip=cfg.clip, target_kl=cfg.target_kl, max_grad=cfg.max_grad, pi_coef=cfg.pi_coef, vf_coef=cfg.vf_coef,
                              ent_coef=cfg.ent_coef, lipschitz=lip, use_lipschitz=1 if cfg.use_lipschitz else 0, world=world)


def parity(actor_hidden, critic_hidden, n_total, batch):
    agent = TorchActorCritic(26, 4, actor_hidden, 26, 64, critic_hidden).cuda()
    with torch.no_grad():
        agent.log_std.fill_(-0.3)
    gen = torch.Generator(device="cuda").manual_seed(1)
    obs = torch.randn(n_total, 1, 26, device="cuda", generator=gen) * 0.7
    states = torch.randn(n_total, 5, 26, device="cuda", generator=gen) * 0.7
    act = torch.randn(n_total, 4, device="cuda", generator=gen).clamp(-1.5, 1.5)
    adv = torch.randn(n_total, device="cuda", generator=gen)
    ret = torch.randn(n_total, device="cuda", generator=gen) * 0.5
    with torch.no_grad():
        lp = agent.evaluate(obs, states, act)[0]
    old_logp = lp + 0.1 * torch.randn(n_total, device="cuda", generator=gen)
    idx = torch.randperm(n_total, device="cuda", generator=gen)[:batch]
    cfg = PPOConfig(target_kl=1e9, ent_coef=0.01)
    nat = NativePPO(agent, batch)
    nat._create(5)
    hy = hyper(cfg, 1e-3, 4.0)
    L, s, p = nat._lib, nat._stream(), (lambda t: C.c_void_p(t.data_ptr()))
    _capi.check(L.taco_ppo_begin_update(nat._h, s), "begin")
    _capi.check(L.taco_ppo_forward_loss(nat._h, C.byref(hy), p(obs.reshape(n_total, -1)), p(states), p(act), p(old_logp), p(adv), p(ret), p(idx), s), "fwd")
    torch.cuda.synchronize()
    sums = nat.loss_sums.clone()
    _capi.check(L.taco_ppo_decide(nat._h, C.byref(hy), s), "decide")
    _capi.check(L.taco_ppo_backward(nat._h, s), "bwd")
    torch.cuda.synchronize()
    mean_n, value_n = nat.debug_outputs()
    # fp32 autograd twin of the same minibatch (ppo_update's loss lines)
    agent.zero_grad()
    logp, ent, value, mean, _ = agent.evaluate(obs[idx], states[idx], act[idx])
    ratio = torch.exp(logp - old_logp[idx])
    sur = -torch.min(adv[idx] * ratio, adv[idx] * torch.clamp(ratio, 1 - cfg.clip, 1 + cfg.clip)).mean()
    vl = torch.nn.functional.mse_loss(ret[idx].view(-1, 1), value)
    loss = cfg.pi_coef * sur + cfg.vf_coef * vl + cfg.ent_coef * (-ent.mean())
    loss.backward()
    res = {"mean_abs_err": float((mean_n - mean).abs().max()), "value_abs_err": float((value_n - value.view(-1)).abs().max()),
           "sur": [float(sums[0] / batch), float(sur)], "vl": [float(sums[1] / batch), float(vl)]}
    views = nat._views(nat.grad)
    gerr = {}
    for name, prm in agent.named_parameters():
        ref = prm.grad
        gerr[name] = float((views[name] - ref).norm() / (ref.norm() + 1e-12))
    res["grad_rel_err"] = gerr
    nat.close()
    return res


out["parity_small"] = parity([64, 48], [32], 1024, 256)
print(json.dumps(out["parity_small"]), flush=True)
out["parity_256"] = parity([256, 256, 256], [256, 256, 256], 8192, 4096)
print(json.dumps(out["parity_256"]), flush=True)

# ---------------------------------------------------------------- 3. the reference-generated golden update
z = np.load(os.path.join(ROOT, "tests", "golden", "ppo_update_native.npz"))
for tag in ("plain", "lip"):
    gg = {k[len("plain_"):]: torch.from_numpy(np.asarray(z[k])) for k in z.files if k.startswith("plain_")}   # shared arrays: plain_ only
    gg.update({k[len(tag) + 1:]: torch.from_numpy(np.asarray(z[k])) for k in z.files if k.startswith(tag + "_")})
    init = {k[6:]: v for k, v in gg.items() if k.startswith("init__")}
    final = {k[7:]: v for k, v in gg.items() if k.startswith("final__")}
    buf = types.SimpleNamespace(**{k[5:]: v.cuda() for k, v in gg.items() if k.startswith("buf__")})
    log = {k[5:]: float(v) for k, v in gg.items() if k.startswith("log__")}
    agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32])
    agent.load_state_dict(init)
    agent.cuda()
    cfg = PPOConfig(clip=0.2, target_kl=0.5, max_grad=0.5, epochs=40, train_iters=2, lr=1e-3, pi_coef=1.0, vf_coef=0.5, ent_coef=0.01,
                    lr_ratio=0.3, lr_lp_index=0.7, lr_epoch_index=30, use_lipschitz=(tag == "lip"), lipschitz_para=2.0,
                    lip_ratio=[1.0, 0.3], lip_lp_index=[0.3, 0.7], lip_epoch_index=[5, 30], diff_value=[0.1, 1.0],
                    diff_lp_index=[0.3, 0.7], diff_epoch_index=[5, 30])
    idx = [row.tolist() for row in gg["idx"]]
    nat = NativePPO(agent, len(idx[0]))
    res = nat.update(buf, cfg, int(gg["epoch"]), batch_idx=idx)
    nat.store_to(agent)
    worst, moved = {}, 0.0
    for k, v in agent.state_dict().items():
        worst[k] = float((v.cpu() - final[k]).abs().max())
        moved = max(moved, float((final[k] - init[k]).abs().max()))
    # the same update through the fp32 autograd twin, for scale
    agent2 = TorchActorCritic(26, 4, [64, 48], 26, 64, [32])
    agent2.load_state_dict(init)
    agent2.cuda()
    ppo_update(agent2, make_optimizer(agent2, cfg), buf, cfg, int(gg["epoch"]), batch_idx=idx)
    worst2 = max(float((v.cpu() - final[k]).abs().max()) for k, v in agent2.state_dict().items())
    out["golden_" + tag] = {"max_param_err": max(worst.values()), "worst": {k: v for k, v in worst.items() if v > 2e-5}, "moved": moved,
                            "autograd_twin_err": worst2,
                            "logs": {k: [res[k], log[k]] for k in ("policy_gradient_loss", "value_loss", "entropy_loss", "sum_loss", "approx_kl")},
                            "optim_steps": res["optim_steps"], "sigmas": nat.sigmas().tolist() if tag == "lip" else None}
    print(json.dumps(out["golden_" + tag]), flush=True)
    nat.close()

# ---------------------------------------------------------------- 4. time at the reference's scale
if "--no-time" not in sys.argv:
    H, N, mb, iters = 64, 4096, 4, 4
    agent = TorchActorCritic(26, 4, [256, 256, 256], 26, 64, [256, 256, 256]).cuda()
    gen = torch.Generator(device="cuda").manual_seed(2)
    buf = types.SimpleNamespace(
        obs_buf=torch.randn(H, N, 1, 26, device="cuda", generator=gen) * 0.5, states_buf=torch.randn(H, N, 5, 26, device="cuda", generator=gen) * 0.5,
        act_buf=torch.randn(H, N, 4, device="cuda", generator=gen).clamp(-1, 1), value_buf=torch.zeros(H, N, 1, device="cuda"),
        ret_buf=torch.randn(H, N, 1, device="cuda", generator=gen) * 0.3, adv_buf=torch.randn(H, N, 1, device="cuda", generator=gen))
    with torch.no_grad():
        buf.logp_buf = agent.evaluate(buf.obs_buf.view(-1, 1, 26), buf.states_buf.view(-1, 5, 26), buf.act_buf.view(-1, 4))[0].view(H, N, 1)
    cfg = PPOConfig(train_iters=iters, use_lipschitz=True, lipschitz_para=4.0, target_kl=1e9)
    perm = torch.randperm(H * N, device="cuda").view(mb, -1)
    idx = [perm[i] for i in range(mb)]
    nat = NativePPO(agent, perm.shape[1])
    nat.update(buf, cfg, 0, batch_idx=idx)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 3
    for r in range(reps):
        res = nat.update(buf, cfg, 1 + r, batch_idx=idx)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    opt = make_optimizer(agent, cfg)
    ppo_update(agent, opt, buf, cfg, 0, batch_idx=idx)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ppo_update(agent, opt, buf, cfg, 1, batch_idx=idx)
    torch.cuda.synchronize()
    dt_torch = time.perf_counter() - t0
    out["time"] = {"workload": f"{N} envs x {H} steps, {mb} minibatches x {iters} iterations = {mb * iters} optimiser steps of {perm.shape[1]} samples, "
                               "actor 26-256-256-256-4, critic LSTM 64 + MLP 64-256-256-256-1, spectral projection on",
                   "native_update_s": dt, "native_ms_per_optim_step": dt / (mb * iters) * 1e3, "torch_autograd_update_s": dt_torch,
                   "optim_steps": res["optim_steps"], "kl": res["approx_kl"]}
    print(json.dumps(out["time"]), flush=True)
    nat.close()
with open(os.path.join(ROOT, "gpurun_out", "ppo_native_check.json"), "w") as fh:
    json.dump(out, fh, indent=1)
