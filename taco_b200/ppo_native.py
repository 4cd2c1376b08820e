"""``PPO.update`` on hand-written sm_100a kernels (SURVEY.md section 8f row 4; ``taco_ppo_*`` in include/taco_b200.h).

``NativePPO`` owns the training state of one ``TorchActorCritic``-shaped agent on the device -- flat fp32 parameters, gradient,
Adam moments -- and runs the reference's update (IsaacGymEnvs/algorithms/ppo_asymmetry.py:137-258) as a stream of kernel launches:
gather -> tcgen05 GEMM forward (actor MLP; critic = 5 LSTM steps per stacked LSTM layer + MLP) -> loss / KL -> device-side early-stop decision ->
GEMM backward (split-K weight gradients, LSTM backward through time) -> gradient norm + clip + Adam -> spectral projection of the
actor weights -> bf16 re-pack.  Nothing synchronises with the host until ``end``: the KL early stop of :223-226 is a device flag.

``ppo_update_native`` has the signature and return value of ``taco_b200.ppo.ppo_update`` (the PyTorch-autograd twin, which stays
as the fp32 parity path).  Under torch.distributed the loss sums and the flat gradient are all-reduced between the phases, one
NCCL call each per minibatch.  There is no fallback: constructing ``NativePPO`` without an sm_100 device raises.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _capi
from .ppo import schedules, value_log


def _linears(mlp):
    return [m for m in mlp.layers if isinstance(m, torch.nn.Linear)]


class NativePPO:
    def __init__(self, agent, batch, device="cuda:0"):
        """``agent``: a ``TorchActorCritic`` (or the reference's ``PPO_ActorCritic`` in the same configuration); ``batch``: samples
        per optimiser step (horizon_len * num_envs / mini_batch_num)."""
        dev = torch.device(device)
        if dev.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("NativePPO runs on CUDA only; there is no CPU path")
        self.device_id = dev.index if dev.index is not None else 0
        self.device = f"cuda:{self.device_id}"
        a_lin, c_lin = _linears(agent.actor_mlp), _linears(agent.critic_mlp)
        lstm = agent.critic_encoder.layers
        if not 1 <= lstm.num_layers <= 4 or lstm.bidirectional:
            raise ValueError("NativePPO: 1 to 4 unidirectional LSTM layers")
        self.lstm_layers = int(lstm.num_layers)
        self.batch = int(batch)
        self.obs_dim, self.act_dim = a_lin[0].in_features, a_lin[-1].out_features
        self.state_dim, self.lstm_hidden = lstm.input_size, lstm.hidden_size
        cfg = _capi.TacoPPOCfg()
        cfg.batch, cfg.obs_dim, cfg.act_dim, cfg.state_dim = self.batch, self.obs_dim, self.act_dim, self.state_dim
        cfg.seq_len = 0                                   # set on the first update from the buffer's states shape
        cfg.lstm_hidden = self.lstm_hidden
        ah, ch = [m.out_features for m in a_lin[:-1]], [m.out_features for m in c_lin[:-1]]
        if len(ah) > 4 or len(ch) > 4:
            raise ValueError("NativePPO: at most 4 hidden layers per MLP")
        cfg.n_actor_hidden, cfg.n_critic_hidden = len(ah), len(ch)
        for i, h in enumerate(ah):
            cfg.actor_hidden[i] = h
        for i, h in enumerate(ch):
            cfg.critic_hidden[i] = h
        self._cfg = cfg
        self._lib = _capi.lib()
        self._h = None
        self._names = (["log_std"] + [f"actor_mlp.layers.{2 * l}.{k}" for l in range(len(a_lin)) for k in ("weight", "bias")] +
                       [f"critic_encoder.layers.{k}_l{l}" for l in range(self.lstm_layers) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")] +
                       [f"critic_mlp.layers.{2 * l}.{k}" for l in range(len(c_lin)) for k in ("weight", "bias")])
        self._pending_agent = agent

    # ------------------------------------------------------------------ construction (needs the sequence length)
    def _create(self, seq_len):
        self._cfg.seq_len = int(seq_len)
        h = C.c_void_p()
        _capi.check(self._lib.taco_ppo_create_layers(self.device_id, C.byref(self._cfg), self.lstm_layers, C.byref(h)), "taco_ppo_create_layers")
        self._h = h
        n = C.c_int64()
        _capi.check(self._lib.taco_ppo_num_params(h, C.byref(n)), "taco_ppo_num_params")
        self.n_params = int(n.value)
        offs = (C.c_int64 * 64)()
        cnt = C.c_int32()
        _capi.check(self._lib.taco_ppo_param_offsets(h, offs, 64, C.byref(cnt)), "taco_ppo_param_offsets")
        assert cnt.value == len(self._names)
        self._offsets = [int(offs[i]) for i in range(cnt.value)]
        ptrs = [C.c_void_p() for _ in range(5)]
        _capi.check(self._lib.taco_ppo_buffers(h, *[C.byref(p) for p in ptrs]), "taco_ppo_buffers")
        w = lambda p, shape, ts: _capi.wrap(p.value, shape, ts, self.device, self)
        self.params, self.grad = w(ptrs[0], (self.n_params,), "<f4"), w(ptrs[1], (self.n_params,), "<f4")
        self.adam_m, self.adam_v = w(ptrs[2], (self.n_params,), "<f4"), w(ptrs[3], (self.n_params,), "<f4")
        self.step = w(ptrs[4], (1,), "<i4")
        acc = C.c_void_p()
        _capi.check(self._lib.taco_ppo_loss_sums(h, C.byref(acc)), "taco_ppo_loss_sums")
        self.loss_sums = w(acc, (8,), "<f8")
        if self._pending_agent is not None:
            self.load_from(self._pending_agent)
            self._pending_agent = None

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device_id).cuda_stream)

    def _views(self, flat):
        return {n: flat[o:o + int(np.prod(s))].view(s) for n, o, s in zip(self._names, self._offsets, self._shapes)}

    # ------------------------------------------------------------------ parameter exchange with the torch module
    def load_from(self, agent, optimizer=None):
        """Copy the module's parameters (and, if given, its torch.optim.Adam moments / step) into the native state."""
        sd = dict(agent.named_parameters())
        self._shapes = [tuple(sd[n].shape) for n in self._names]
        if self._h is None:
            self._pending_agent = agent
            return
        with torch.no_grad():
            for n, v in self._views(self.params).items():
                v.copy_(sd[n].detach().to(self.device, torch.float32))
            if optimizer is not None and len(optimizer.state) > 0:
                m, v2 = self._views(self.adam_m), self._views(self.adam_v)
                step = 0
                for n in self._names:
                    st = optimizer.state.get(sd[n])
                    if st:
                        m[n].copy_(st["exp_avg"]); v2[n].copy_(st["exp_avg_sq"]); step = int(st["step"])
                self.step.fill_(step)
        _capi.check(self._lib.taco_ppo_params_changed(self._h, self._stream()), "taco_ppo_params_changed")

    def store_to(self, agent, optimizer=None):
        """Copy the trained parameters (and Adam state) back into the torch module / optimizer (checkpoints, export, rollout sync)."""
        sd = dict(agent.named_parameters())
        with torch.no_grad():
            for n, v in self._views(self.params).items():
                sd[n].copy_(v)
            if optimizer is not None:
                m, v2 = self._views(self.adam_m), self._views(self.adam_v)
                step = float(self.step.item())
                for n in self._names:
                    st = optimizer.state[sd[n]]
                    st["exp_avg"], st["exp_avg_sq"] = m[n].clone(), v2[n].clone()
                    st["step"] = torch.tensor(step)

    # ------------------------------------------------------------------ one PPO.update
    def update(self, buffer, cfg, epoch, env=None, batch_idx=None, group=None):
        lr, lip, diff = schedules(cfg, epoch)
        if env is not None:
            env.difficulty = diff
        torch.cuda.nvtx.range_push("taco.update")
        try:
            return self._update(buffer, cfg, lr, lip, diff, batch_idx, group)
        finally:
            torch.cuda.nvtx.range_pop()

    def _update(self, buffer, cfg, lr, lip, diff, batch_idx, group):
        flat = lambda t: t.reshape(-1, *t.shape[2:]).contiguous()
        obs, states, act = flat(buffer.obs_buf), flat(buffer.states_buf), buffer.act_buf.reshape(-1, buffer.act_buf.size(-1)).contiguous()
        ret, old_logp, adv = buffer.ret_buf.reshape(-1).contiguous(), buffer.logp_buf.reshape(-1).contiguous(), buffer.adv_buf.reshape(-1).contiguous()
        if self._h is None:
            self._create(states.shape[1])
        # group=False: no collectives even when a process group exists (a rank-local update, e.g. a single-process comparison run)
        world = dist.get_world_size(group) if (group is not False and dist.is_available() and dist.is_initialized()) else 1
        hy = _capi.TacoPPOHyper(lr=lr, clip=cfg.clip, target_kl=cfg.target_kl, max_grad=cfg.max_grad, pi_coef=cfg.pi_coef, vf_coef=cfg.vf_coef,
                                ent_coef=cfg.ent_coef, lipschitz=lip, use_lipschitz=1 if cfg.use_lipschitz else 0, world=world)
        if batch_idx is None:
            batch_idx = buffer.batch_idx_generator()
        idx_dev = []
        for indices in batch_idx:
            t = indices if isinstance(indices, torch.Tensor) else torch.as_tensor(indices)
            t = t.to(self.device, torch.int64).contiguous()
            if t.numel() != self.batch:
                raise ValueError(f"NativePPO was built for minibatches of {self.batch} samples, got {t.numel()}")
            idx_dev.append(t)
        L, s = self._lib, self._stream()
        p = lambda t: C.c_void_p(t.data_ptr())
        obs2 = obs.reshape(obs.shape[0], -1)
        _capi.check(L.taco_ppo_begin_update(self._h, s), "taco_ppo_begin_update")
        for _ in range(cfg.train_iters):
            for t in idx_dev:
                _capi.check(L.taco_ppo_forward_loss(self._h, C.byref(hy), p(obs2), p(states), p(act), p(old_logp), p(adv), p(ret), p(t), s), "taco_ppo_forward_loss")
                if world > 1:
                    dist.all_reduce(self.loss_sums, op=dist.ReduceOp.SUM, group=group)
                _capi.check(L.taco_ppo_decide(self._h, C.byref(hy), s), "taco_ppo_decide")
                _capi.check(L.taco_ppo_backward(self._h, s), "taco_ppo_backward")
                if world > 1:
                    dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=group)
                _capi.check(L.taco_ppo_apply(self._h, C.byref(hy), s), "taco_ppo_apply")
        max_rows = cfg.train_iters * len(idx_dev)
        log = np.zeros((max_rows, 8), dtype=np.float32)
        n_rows, steps, stop = C.c_int32(), C.c_int32(), C.c_int32()
        step_before = getattr(self, "_steps_total", 0)
        _capi.check(L.taco_ppo_end_update(self._h, log.ctypes.data_as(C.c_void_p), max_rows, C.byref(n_rows), C.byref(steps), C.byref(stop), s),
                    "taco_ppo_end_update")
        self._steps_total = int(steps.value)
        log = log[:n_rows.value]
        mean = lambda c: float(log[:, c].mean()) if len(log) else 0.0
        mean_value, explained_var = value_log(buffer, idx_dev[(len(log) - 1) % len(idx_dev)]) if len(log) else (0.0, float("nan"))
        return {"mean_value": mean_value, "explained_variance": explained_var,
                "policy_gradient_loss": mean(0), "value_loss": mean(1), "entropy_loss": mean(2), "sum_loss": mean(3), "approx_kl": mean(4),
                "grad_norm": mean(5), "learning_rate": lr, "lipschitz_para": lip, "difficulty": diff,
                "optim_steps": self._steps_total - step_before, "early_stop": bool(stop.value), "log": log}

    def sigmas(self):
        out = np.zeros(self._cfg.n_actor_hidden + 1, dtype=np.float64)
        _capi.check(self._lib.taco_ppo_sigmas(self._h, out.ctypes.data_as(C.c_void_p)), "taco_ppo_sigmas")
        return out

    def debug_outputs(self):
        m, v = C.c_void_p(), C.c_void_p()
        _capi.check(self._lib.taco_ppo_debug_outputs(self._h, C.byref(m), C.byref(v)), "taco_ppo_debug_outputs")
        return (_capi.wrap(m.value, (self.batch, self.act_dim), "<f4", self.device, self), _capi.wrap(v.value, (self.batch,), "<f4", self.device, self))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.taco_ppo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def ppo_update_native(native, buffer, cfg, epoch, env=None, batch_idx=None, group=None):
    """``ppo_update`` (taco_b200.ppo) on the native kernels; ``native``: a ``NativePPO`` holding the agent's training state."""
    return native.update(buffer, cfg, epoch, env=env, batch_idx=batch_idx, group=group)


def gemm_selftest(a_bf16, b_bf16, splits=1, transposed=False):
    """D = A B^T through the tcgen05 GEMM kernel of the native update; returns fp32 (m, n).  ``transposed=False``: bf16 CUDA tensors A (m, k),
    B (n, k) (K-major operands); ``transposed=True``: the operands are given as At (k, m), Bt (k, n) (the kernel's MN-major mode)."""
    if transposed:
        (k, m), n = a_bf16.shape, b_bf16.shape[1]
    else:
        (m, k), n = a_bf16.shape, b_bf16.shape[0]
    d = torch.empty(m, n, dtype=torch.float32, device=a_bf16.device)
    dev = a_bf16.device.index or 0
    fn = _capi.lib().taco_gemm_selftest_mn if transposed else _capi.lib().taco_gemm_selftest
    _capi.check(fn(dev, C.c_void_p(a_bf16.data_ptr()), C.c_void_p(b_bf16.data_ptr()), C.c_void_p(d.data_ptr()), m, n, k,
                   int(splits), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "taco_gemm_selftest")
    return d
