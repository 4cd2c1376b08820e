"""The PPO update around the native rollout path (SURVEY.md section 8f row 4).

Mirrors, in the configuration the reference trains with (README.md:60-66: MLP actor, LSTM critic encoder):
  * ``PPO_ActorCritic`` (construction, init, ``evaluate``)   IsaacGymEnvs/algorithms/nets_asymmetry.py:270-377, :41-55, :138-143
  * ``PPO.update`` incl. the three schedules                  IsaacGymEnvs/algorithms/ppo_asymmetry.py:137-258
  * ``PPO.spectral_normalize_actors`` after every optimiser step (:248-249, :398-404) -- here ``taco_spectral_project`` on the
    parameter storage (power iteration on the device, no SVD, no host round trip)
The update itself is PyTorch autograd on the buffers the native rollout filled (``RolloutBuffer``); what this module adds to the
reference is the multi-GPU form of the env-sharded job: gradients are averaged over the ranks with one flat all-reduce per
minibatch, and the KL early-stop decision is taken on the all-reduced KL so that every rank leaves the loop together.
``sync_rollout_nets`` copies the updated weights into the rollout kernels (``ActorMLP`` / ``CriticLSTM``) once per update.
"""
import math
from dataclasses import dataclass, field
from typing import List

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F


class _MLP(nn.Module):
    """nets_asymmetry.py:23-55 (``.layers`` Sequential like the reference, so ``load_module`` / state dicts line up)."""

    def __init__(self, input_size, hidden_size, output_size, output_activation):
        super().__init__()
        self.hidden_size = list(hidden_size)
        sizes = [input_size] + self.hidden_size + [output_size]
        layers = []
        for j in range(len(sizes) - 2):
            layers += [nn.Linear(sizes[j], sizes[j + 1]), nn.ReLU()]
        layers += [nn.Linear(sizes[-2], sizes[-1]), output_activation()]
        self.layers = nn.Sequential(*layers)

    def forward(self, x):
        return self.layers(x.contiguous().view(x.size(0), -1))

    def para_init(self):
        gains = [math.sqrt(2)] * len(self.hidden_size) + [0.01]
        for g, m in zip(gains, (m for m in self.layers if isinstance(m, nn.Linear))):
            nn.init.orthogonal_(m.weight, gain=g)


class _LSTMEncoder(nn.Module):
    """nets_asymmetry.py:128-143."""

    def __init__(self, input_size, output_size, num_layers):
        super().__init__()
        self.layers = nn.LSTM(input_size, output_size, num_layers, batch_first=True)

    def forward(self, x):
        x, _ = self.layers(x)
        return x[:, -1, :]

    def para_init(self):
        for prm in self.layers.parameters():
            if prm.dim() > 1:
                nn.init.xavier_uniform_(prm)
            else:
                nn.init.constant_(prm, 0)


class TorchActorCritic(nn.Module):
    """Autograd twin of ``PPO_ActorCritic`` with ``use_actor_encoder=False, use_critic_encoder=True, critic_encoder_type='LSTM'``;
    parameter names equal the reference's (``actor_mlp.layers.N.*``, ``critic_encoder.layers.*``, ``critic_mlp.layers.N.*``,
    ``log_std``), so state dicts are interchangeable."""

    def __init__(self, obs_dim, act_dim, actor_hidden, state_dim, lstm_hidden, critic_hidden, lstm_layers=1):
        super().__init__()
        self.actor_mlp = _MLP(obs_dim, actor_hidden, act_dim, nn.Tanh)
        self.actor_mlp.para_init()
        self.log_std = nn.Parameter(math.log(1.0) * torch.ones(act_dim))
        self.critic_encoder = _LSTMEncoder(state_dim, lstm_hidden, lstm_layers)
        self.critic_encoder.para_init()
        self.critic_mlp = _MLP(lstm_hidden, critic_hidden, 1, nn.Identity)
        self.critic_mlp.para_init()

    def forward(self, actor_input):
        """nets_asymmetry.py:379-387: the deterministic action mean; what ``export_actor`` traces."""
        return self.actor_mlp(actor_input)

    def evaluate(self, actor_input, critic_input, actor_output):
        """nets_asymmetry.py:356-377.  MultivariateNormal(mean, scale_tril=diag(exp(log_std)^2)) written out: the standard
        deviation is exp(2 log_std) (SURVEY.md quirk 13)."""
        mean = self.actor_mlp(actor_input)
        log_sd = 2.0 * self.log_std
        k = mean.shape[1]
        z = (actor_output - mean) * torch.exp(-log_sd)
        logp = -0.5 * (z * z).sum(dim=1) - log_sd.sum() - 0.5 * k * math.log(2.0 * math.pi)
        entropy = (0.5 * k * (1.0 + math.log(2.0 * math.pi)) + log_sd.sum()).expand(mean.shape[0])
        value = self.critic_mlp(self.critic_encoder(critic_input))
        return logp, entropy, value, mean, self.log_std.repeat(mean.shape[0], 1)


@dataclass
class PPOConfig:
    """Constructor arguments of the reference ``PPO`` that ``update`` reads (ppo_asymmetry.py:26-33; same defaults)."""
    clip: float = 0.2
    target_kl: float = 0.03
    max_grad: float = 0.5
    use_clipped_value_loss: bool = False
    epochs: int = 500
    train_iters: int = 16
    lr: float = 3e-4
    pi_coef: float = 1.0
    vf_coef: float = 0.5
    ent_coef: float = 0.0
    learning_rate_schedule: bool = True
    lr_ratio: float = 0.3
    lr_lp_index: float = 0.7
    lr_epoch_index: int = 350
    use_lipschitz: bool = False
    lipschitz_para: float = 5.0
    lipschitz_schedule: bool = True
    lip_ratio: List[float] = field(default_factory=lambda: [1.0, 0.3])
    lip_lp_index: List[float] = field(default_factory=lambda: [0.3, 0.7])
    lip_epoch_index: List[int] = field(default_factory=lambda: [100, 500])
    difficulty_schedule: bool = True
    diff_value: List[float] = field(default_factory=lambda: [0.1, 1.0])
    diff_lp_index: List[float] = field(default_factory=lambda: [0.3, 0.7])
    diff_epoch_index: List[int] = field(default_factory=lambda: [100, 500])


def make_optimizer(agent, cfg):
    """ppo_asymmetry.py:117."""
    return torch.optim.Adam(filter(lambda p: p.requires_grad, agent.parameters()), lr=cfg.lr, eps=1e-5)


def _ramp(value, index, x):
    if x < index[0]:
        return value[0]
    if x > index[1]:
        return value[1]
    return (value[1] - value[0]) / (index[1] - index[0]) * (x - index[0]) + value[0]


def schedules(cfg, epoch):
    """(learning_rate, lipschitz_para, difficulty) of ``PPO.update`` for this epoch (ppo_asymmetry.py:139-175)."""
    lp = epoch / cfg.epochs
    if cfg.learning_rate_schedule:
        r0 = (cfg.lr_ratio - 1) / cfg.lr_lp_index * lp + 1 if lp < cfg.lr_lp_index else cfg.lr_ratio
        r1 = (cfg.lr_ratio - 1) / cfg.lr_epoch_index * epoch + 1 if epoch < cfg.lr_epoch_index else cfg.lr_ratio
        lr = min(r0, r1) * cfg.lr
    else:
        lr = cfg.lr_ratio * cfg.lr
    if cfg.lipschitz_schedule:
        lip = min(_ramp(cfg.lip_ratio, cfg.lip_lp_index, lp), _ramp(cfg.lip_ratio, cfg.lip_epoch_index, epoch)) * cfg.lipschitz_para
    else:
        lip = cfg.lip_ratio[1] * cfg.lipschitz_para
    if cfg.difficulty_schedule:
        diff = max(_ramp(cfg.diff_value, cfg.diff_lp_index, lp), _ramp(cfg.diff_value, cfg.diff_epoch_index, epoch))
    else:
        diff = cfg.diff_value[1]
    return lr, lip, diff


def _world(group):
    return dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1


def _allreduce_grads(params, group):
    """One flat SUM all-reduce of every gradient, divided by the world size (the env-sharded job's data-parallel step)."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat /= dist.get_world_size(group)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n


def value_log(buffer, idx):
    """``mean_value`` and ``explained_variance`` as PPO.update logs them (ppo_asymmetry.py:252-254,406-423): computed on the old values /
    returns of the LAST evaluated minibatch (numpy, population variance)."""
    idx = idx if isinstance(idx, torch.Tensor) else torch.as_tensor(idx)
    v = buffer.value_buf.reshape(-1)[idx.to(buffer.value_buf.device)].detach().cpu().numpy().flatten()
    r = buffer.ret_buf.reshape(-1)[idx.to(buffer.ret_buf.device)].detach().cpu().numpy().flatten()
    var_y = r.var()
    return float(v.mean()), (float("nan") if var_y == 0 else float(1 - (r - v).var() / var_y))


def ppo_update(agent, optimizer, buffer, cfg, epoch, env=None, batch_idx=None, group=None, project=None):
    """``PPO.update(epoch)`` (ppo_asymmetry.py:137-258) on the tensors of ``buffer`` (a ``RolloutBuffer`` or anything with the
    reference buffer's attributes).  ``batch_idx``: minibatch index lists / tensors (default: ``buffer.batch_idx_generator()``).
    ``project(params, c)``: the spectral projection (default: the device kernel, ``taco_b200.spectral_normalize_``).
    Returns the scalars the reference logs (``log_update``, :438-450)."""
    agent.train()
    torch.cuda.nvtx.range_push("taco.update_autograd") if torch.cuda.is_available() else None
    lr, lip, diff = schedules(cfg, epoch)
    optimizer.param_groups[0]["lr"] = lr
    if env is not None:
        env.difficulty = diff
    if batch_idx is None:
        batch_idx = buffer.batch_idx_generator()
    if project is None and cfg.use_lipschitz:
        from .actor import spectral_normalize_ as project
    world = _world(group)
    params = [p for p in agent.parameters() if p.requires_grad]
    flat = lambda t: t.view(-1, *t.size()[2:])
    obs, states, act = flat(buffer.obs_buf), flat(buffer.states_buf), buffer.act_buf.view(-1, buffer.act_buf.size(-1))
    old_value, ret = buffer.value_buf.view(-1, 1), buffer.ret_buf.view(-1, 1)
    old_logp, adv = buffer.logp_buf.view(-1, 1), buffer.adv_buf.view(-1, 1)
    pg_l, v_l, e_l, s_l, kls = [], [], [], [], []
    keep_going, steps, last_idx = True, 0, None
    for it in range(cfg.train_iters):
        for indices in batch_idx:
            idx = indices if isinstance(indices, torch.Tensor) else torch.as_tensor(indices, device=obs.device)
            last_idx = idx
            logp, entropy, value, _, _ = agent.evaluate(obs[idx], states[idx], act[idx])
            adv_b, old_logp_b, ret_b, old_value_b = adv[idx].squeeze(1), old_logp[idx].squeeze(1), ret[idx], old_value[idx]
            ratio = torch.exp(logp - old_logp_b)
            surrogate_loss = -torch.min(adv_b * ratio, adv_b * torch.clamp(ratio, 1.0 - cfg.clip, 1.0 + cfg.clip)).mean()
            if cfg.use_clipped_value_loss:          # kept as written upstream (:203-207): both terms are the same mse
                value_loss = torch.max(F.mse_loss(value, ret_b), F.mse_loss(ret_b, value)).mean()
            else:
                value_loss = F.mse_loss(ret_b, value)
            entropy_loss = -torch.mean(entropy)
            loss = cfg.pi_coef * surrogate_loss + cfg.vf_coef * value_loss + cfg.ent_coef * entropy_loss
            with torch.no_grad():
                log_ratio = logp - old_logp_b
                kl = torch.mean((torch.exp(log_ratio) - 1) - log_ratio)
                stats = torch.stack([surrogate_loss.detach(), value_loss.detach(), entropy_loss.detach(), loss.detach(), kl]).double()
                if world > 1:
                    dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
                    stats /= world
                pg, vl, el, sl, klv = stats.tolist()     # the reference syncs here too (.item() x 4 + .cpu(), :214-226)
            pg_l.append(pg); v_l.append(vl); e_l.append(el); s_l.append(sl); kls.append(klv)
            if klv > 1.5 * cfg.target_kl and cfg.pi_coef > 0:
                keep_going = False
                break
            optimizer.zero_grad()
            loss.backward()
            if world > 1:
                _allreduce_grads(params, group)
            nn.utils.clip_grad_norm_(agent.parameters(), cfg.max_grad)
            optimizer.step()
            steps += 1
            if cfg.use_lipschitz:
                project(agent.actor_mlp.parameters(), lip)
        if not keep_going:
            break
    agent.eval()
    torch.cuda.nvtx.range_pop() if torch.cuda.is_available() else None
    mean = lambda xs: float(sum(xs) / max(len(xs), 1))
    mean_value, explained_var = value_log(buffer, last_idx) if last_idx is not None else (0.0, float("nan"))
    return {"policy_gradient_loss": mean(pg_l), "value_loss": mean(v_l), "entropy_loss": mean(e_l), "sum_loss": mean(s_l),
            "approx_kl": mean(kls), "learning_rate": lr, "lipschitz_para": lip, "difficulty": diff, "optim_steps": steps,
            "early_stop": not keep_going, "mean_value": mean_value, "explained_variance": explained_var}


def sync_rollout_nets_native(native, actor=None, critic=None):
    """``sync_rollout_nets`` for a ``NativePPO``: the rollout kernels load straight from the trainer's flat device parameter vector
    (device-to-device copies; no torch module, no host round trip)."""
    v = native._views(native.params)
    if actor is not None:
        n = native._cfg.n_actor_hidden + 1
        actor.load([v[f"actor_mlp.layers.{2 * l}.weight"] for l in range(n)], [v[f"actor_mlp.layers.{2 * l}.bias"] for l in range(n)],
                   lipschitz_const=-1.0, log_std=v["log_std"])
    if critic is not None:
        n = native._cfg.n_critic_hidden + 1
        critic.load([tuple(v[f"critic_encoder.layers.{k}_l{l}"] for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")) for l in range(native.lstm_layers)],
                    [v[f"critic_mlp.layers.{2 * l}.weight"] for l in range(n)], [v[f"critic_mlp.layers.{2 * l}.bias"] for l in range(n)])


def sync_rollout_nets(agent, actor=None, critic=None):
    """Copy the trained weights into the rollout kernels: once per update (the stored actor weights are already projected)."""
    if actor is not None:
        actor.load_module(agent.actor_mlp, log_std=agent.log_std, lipschitz_const=-1.0)      # already projected by ppo_update: no norm measurement
    if critic is not None:
        critic.load_modules(agent.critic_encoder, agent.critic_mlp)


# ------------------------------------------------------------------------------------------------ checkpoints / export
def save_checkpoint(path, agent, optimizer=None, epoch=None, env=None, para_only=True, extra=None):
    """``PPO.save`` (ppo_asymmetry.py:452-456): ``para_only=True`` writes ``agent.state_dict()`` exactly like the reference
    (parameter names equal the reference's, so the file loads into a reference ``PPO_ActorCritic`` and vice versa);
    ``para_only=False`` writes a resumable training checkpoint: state dict, optimiser state, epoch and -- which the reference
    never saves (SURVEY.md section 5) -- the complete env state (``FpvVecTask.state_checkpoint``)."""
    if para_only:
        torch.save(agent.state_dict(), path)
        return
    blob = {"agent": agent.state_dict(), "optimizer": optimizer.state_dict() if optimizer is not None else None,
            "epoch": epoch, "extra": extra}
    if env is not None:
        blob["env_state"] = torch.from_numpy(env.state_checkpoint())
        blob["env_difficulty"] = env.difficulty
    torch.save(blob, path)


def load_checkpoint(path, agent, optimizer=None, env=None, map_location=None):
    """Inverse of ``save_checkpoint`` (either form).  Returns the stored epoch (None for a bare state dict)."""
    blob = torch.load(path, map_location=map_location, weights_only=True)
    if "agent" not in blob:                                  # a bare state dict (para_only=True, or a reference model's)
        agent.load_state_dict(blob)
        return None
    agent.load_state_dict(blob["agent"])
    if optimizer is not None and blob.get("optimizer") is not None:
        optimizer.load_state_dict(blob["optimizer"])
    if env is not None and blob.get("env_state") is not None:
        env.load_state_checkpoint(blob["env_state"].numpy())
    return blob.get("epoch")


def export_actor(agent, path, len_obs, num_obs, device="cuda:0"):
    """``PPO.save_actor_as_pt`` (ppo_asymmetry.py:458-468): the deterministic policy (``forward`` = action mean) traced with
    ``torch.jit.trace`` on a zero ``(1, len_obs, num_obs)`` observation and saved as TorchScript -- the file the reference deploys
    (``actor_0.pt`` / ``actor_1.pt``).  Returns (eager output, traced output) on the probe input, which the reference prints."""
    agent.eval()
    obs = torch.zeros((1, len_obs, num_obs), device=device)
    traced = torch.jit.trace(agent, obs)
    traced.save(path)
    with torch.no_grad():
        return agent(obs), traced(torch.zeros((1, len_obs, num_obs), device=device))
