"""One native PPO update at the reference's scale (for ncu launch lists / timing).
usage: python tools/ppo_native_time.py [updates] [--no-lip] [--lstm-layers L] [--autograd]
--lstm-layers: stacked LSTM layers of the critic encoder (default 1); --autograd: time the fp32 autograd twin (taco_b200.ppo.ppo_update)
on the same buffer and minibatches instead."""
import os, sys, time, types, json
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from taco_b200.ppo import PPOConfig, TorchActorCritic, make_optimizer, ppo_update
from taco_b200.ppo_native import NativePPO
reps = int(sys.argv[1]) if len(sys.argv) > 1 and sys.argv[1].isdigit() else 1
H, N, mb, iters = 64, 4096, 4, 4
layers = int(sys.argv[sys.argv.index("--lstm-layers") + 1]) if "--lstm-layers" in sys.argv else 1
autograd = "--autograd" in sys.argv
agent = TorchActorCritic(26, 4, [256, 256, 256], 26, 64, [256, 256, 256], lstm_layers=layers).cuda()
gen = torch.Generator(device="cuda").manual_seed(2)
buf = types.SimpleNamespace(
    obs_buf=torch.randn(H, N, 1, 26, device="cuda", generator=gen) * 0.5, states_buf=torch.randn(H, N, 5, 26, device="cuda", generator=gen) * 0.5,
    act_buf=torch.randn(H, N, 4, device="cuda", generator=gen).clamp(-1, 1), value_buf=torch.zeros(H, N, 1, device="cuda"),
    ret_buf=torch.randn(H, N, 1, device="cuda", generator=gen) * 0.3, adv_buf=torch.randn(H, N, 1, device="cuda", generator=gen))
with torch.no_grad():
    buf.logp_buf = agent.evaluate(buf.obs_buf.view(-1, 1, 26), buf.states_buf.view(-1, 5, 26), buf.act_buf.view(-1, 4))[0].view(H, N, 1)
cfg = PPOConfig(train_iters=iters, use_lipschitz="--no-lip" not in sys.argv, lipschitz_para=4.0, target_kl=1e9)
perm = torch.randperm(H * N, device="cuda").view(mb, -1)
idx = [perm[i] for i in range(mb)]
if autograd:
    opt = make_optimizer(agent, cfg)
    update = lambda epoch: ppo_update(agent, opt, buf, cfg, epoch, batch_idx=idx)
else:
    nat = NativePPO(agent, perm.shape[1])
    update = lambda epoch: nat.update(buf, cfg, epoch, batch_idx=idx)
update(0)
torch.cuda.synchronize()
t0 = time.perf_counter()
for r in range(reps):
    res = update(1 + r)
torch.cuda.synchronize()
dt = (time.perf_counter() - t0) / reps
print(json.dumps({"autograd_update_s" if autograd else "native_update_s": dt, "ms_per_optim_step": dt / (mb * iters) * 1e3,
                  "optim_steps": res["optim_steps"], "lstm_layers": layers}))
