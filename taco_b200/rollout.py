"""Host-side mirror of the reference rollout buffer, with the return / advantage pass on the device.

Mirrors ``PPOReplayBuffer`` (IsaacGymEnvs/algorithms/buffer_asymmetry.py:9-139): same constructor arguments, same buffer
attributes and shapes (``obs_buf (H,N,Lo,26)``, ``states_buf``, ``act_buf``, ``rew_buf (H,N,1)``, ``done_buf``, ``ret_buf``,
``value_buf``, ``adv_buf``, ``mu_buf``, ``sigma_buf``, ``logp_buf``), ``store``, ``reset``, ``compute_returns_and_advantage``
and ``batch_idx_generator``.  Differences, all on purpose:

  * ``compute_returns_and_advantage`` is two CUDA launches behind the C ABI (``taco_gae_advantages`` / ``taco_gae_normalize``,
    csrc/taco_gae.cu) instead of a Python loop over the horizon plus two full-buffer reductions; under
    ``torch.distributed`` the three float64 moments [sum, sum^2, n] are all-reduced so that every rank normalises with the
    statistics of ALL envs of the job (buffer_asymmetry.py:132 semantics for the sharded rollout);
  * ``store`` accepts ``time_outs``: the bootstrap of truncated episodes (ppo_asymmetry.py:313-324) then happens inside
    the device pass with no ``nonzero().tolist()`` host round trip;
  * obs / states live in a ring of ``horizon_len + 1`` slots (``obs_ring`` / ``states_ring``; ``obs_buf`` / ``states_buf`` are
    the views of the first ``horizon_len`` slots).  ``FpvVecTask.attach_rollout(buffer)`` makes the step kernel write each
    step's observation history, reward, done flag and time-out straight into slot / row ``k`` (``taco_env_attach_rollout``), so
    the per-step ``store`` copies of the reference (2.7 GB per rollout at 262144 envs x 20 steps) disappear; ``store`` then
    takes ``None`` for those fields;
  * ``reset`` only rewinds the write index (the reference re-allocates every buffer each epoch, buffer_asymmetry.py:70-91;
    every slot is overwritten by the next rollout before it is read);
  * ``RolloutEpisodes``: one record per finished training episode and a per-task summary, from one scan of the ring's result
    rows per rollout (``episodes=`` of ``collect_rollout`` / ``GraphedRollout``).
There is no CPU fallback: the buffer lives on a CUDA device.
"""
import ctypes as C

import torch
import torch.distributed as dist

from . import _capi


class RolloutBuffer:
    def __init__(self, num_envs, obs_dim, obs_len, states_dim, states_len, act_dim, horizon_len, mini_batch_num, gamma, lam, device):
        dev = torch.device(device)
        if dev.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("RolloutBuffer runs on CUDA only; there is no CPU path")
        self.num_envs, self.obs_dim, self.obs_len = int(num_envs), int(obs_dim), int(obs_len)
        self.states_dim, self.states_len, self.act_dim = int(states_dim), int(states_len), int(act_dim)
        self.horizon_len, self.mini_batch_num = int(horizon_len), int(mini_batch_num)
        self.gamma, self.lam = float(gamma), float(lam)
        self.device = dev
        self.device_id = dev.index if dev.index is not None else torch.cuda.current_device()
        self._lib = _capi.lib()
        H, N = self.horizon_len, self.num_envs
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)
        self.obs_ring = z(H + 1, N, self.obs_len, self.obs_dim)
        self.states_ring = z(H + 1, N, self.states_len, self.states_dim)
        self.obs_buf = self.obs_ring[:H]
        self.states_buf = self.states_ring[:H]
        self.act_buf = z(H, N, self.act_dim)
        self.rew_buf = z(H, N, 1)
        self.done_buf = z(H, N, 1)
        self.timeout_buf = z(H, N, 1, dtype=torch.uint8)
        self.ret_buf = z(H, N, 1)
        self.value_buf = z(H, N, 1)
        self.adv_buf = z(H, N, 1)
        self.mu_buf = z(H, N, self.act_dim)
        self.sigma_buf = z(H, N, self.act_dim)
        self.logp_buf = z(H, N, 1)
        self.moments = torch.zeros(3, dtype=torch.float64, device=dev)     # [sum adv, sum adv^2, samples], all ranks after the reduce
        self._have_timeouts = False
        self.step = 0

    def store(self, obs, states, act, rew, log_prob, done, value, mu, sigma, time_outs=None):
        """buffer_asymmetry.py:49-68.  ``rew`` is the RAW env reward when ``time_outs`` is given (the bootstrap is applied
        in compute_returns_and_advantage), else the already-augmented reward like the reference."""
        if self.step >= self.horizon_len:
            raise AssertionError("Rollout buffer overflow")
        s = self.step
        if obs is not None:                      # None: the attached env already wrote slot / row s (zero-copy path)
            self.obs_buf[s].copy_(obs)
        if states is not None:
            self.states_buf[s].copy_(states)
        if act is not None and act.data_ptr() != self.act_buf[s].data_ptr():
            self.act_buf[s].copy_(act)
        if rew is not None:
            self.rew_buf[s].copy_(rew.view(-1, 1))
        if done is not None:
            self.done_buf[s].copy_(done.view(-1, 1))
        if value.data_ptr() != self.value_buf[s].data_ptr():
            self.value_buf[s].copy_(value)
        if mu is not None and mu.data_ptr() != self.mu_buf[s].data_ptr():
            self.mu_buf[s].copy_(mu)
        self.sigma_buf[s].copy_(sigma)
        if log_prob is not None and log_prob.data_ptr() != self.logp_buf[s].data_ptr():
            self.logp_buf[s].copy_(log_prob.view(-1, 1))
        if time_outs is True:                    # rows written by the attached env
            self._have_timeouts = True
        elif time_outs is not None:
            self.timeout_buf[s].copy_(time_outs.view(-1, 1))
            self._have_timeouts = True
        elif s == 0:
            self._have_timeouts = False
        self.step += 1

    def reset(self):
        self.step = 0

    def compute_returns_and_advantage(self, last_values, group=None):
        """buffer_asymmetry.py:93-132 on the device; fills ret_buf and the normalised adv_buf.  Asynchronous."""
        last = last_values.detach().to(self.device, torch.float32).contiguous().view(-1)
        if last.numel() != self.num_envs:
            raise ValueError(f"last_values must hold {self.num_envs} values")
        stream = C.c_void_p(torch.cuda.current_stream(self.device_id).cuda_stream)
        p = lambda t: C.c_void_p(t.data_ptr())
        tout = p(self.timeout_buf) if self._have_timeouts else C.c_void_p(0)
        _capi.check(self._lib.taco_gae_advantages(self.device_id, self.horizon_len, self.num_envs, p(self.rew_buf), p(self.done_buf), tout,
                                                  p(self.value_buf), p(last), self.gamma, self.lam, p(self.adv_buf), p(self.ret_buf),
                                                  p(self.moments), stream), "taco_gae_advantages")
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(self.moments, op=dist.ReduceOp.SUM, group=group)          # 3 doubles: the path's second tiny collective
        _capi.check(self._lib.taco_gae_normalize(self.device_id, p(self.adv_buf), self.horizon_len * self.num_envs, p(self.moments), stream),
                    "taco_gae_normalize")
        self._keep = last

    def rows(self, s):
        """Output tensors of step s for ActorMLP.act(out=...): (act_buf[s], scratch for the clipped action, logp_buf[s], mu_buf[s])."""
        if not hasattr(self, "_clipped"):
            self._clipped = torch.empty(self.num_envs, self.act_dim, dtype=torch.float32, device=self.device)
        return self.act_buf[s], self._clipped, self.logp_buf[s].view(-1), self.mu_buf[s]

    def batch_idx_generator(self):
        """buffer_asymmetry.py:134-139."""
        n = self.num_envs * self.horizon_len
        return torch.randperm(n).reshape(self.mini_batch_num, -1).tolist()


class RolloutEpisodes:
    """Training-time episode records and per-task summaries (``taco_env_attach_rollout_episodes``): ``scan()`` -- one launch, run
    by ``collect_rollout`` / ``GraphedRollout`` after the horizon's steps when passed as ``episodes`` -- walks the ring rows the
    step kernel wrote since the last scan and appends one ``ROLLOUT_EPISODE_DTYPE`` record per finished episode (``capacity``
    records on the device; past it they are dropped but counted) and writes the float64 per-task summary of those episodes to
    ``summary_vec``.  Only whole episodes are recorded; the record order is unspecified.  Needs a rollout ring with result rows
    attached at scan time."""

    def __init__(self, env, capacity):
        self.env = env
        self._lib = _capi.lib()
        _capi.check(self._lib.taco_env_attach_rollout_episodes(env._h, int(capacity), self._stream()), "taco_env_attach_rollout_episodes")
        rec, cnt, cap = C.c_void_p(), C.c_void_p(), C.c_int64()
        _capi.check(self._lib.taco_env_rollout_episodes_buffers(env._h, C.byref(rec), C.byref(cnt), C.byref(cap)),
                    "taco_env_rollout_episodes_buffers")
        self.capacity = int(cap.value)
        self._count = _capi.wrap(cnt.value, (1,), "<i8", env.device, self)
        self._records = _capi.wrap(rec.value, (self.capacity * _capi.ROLLOUT_EPISODE_DTYPE.itemsize,), "|u1", env.device, self)
        self.summary_vec = torch.zeros(_capi.EPISODE_SUMMARY_WORDS, dtype=torch.float64, device=env.device)
        self._open = True

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.env.device_id).cuda_stream)

    def scan(self):
        """Scan the ring rows written since the last scan or rewind into records and ``summary_vec`` (asynchronous, capturable)."""
        _capi.check(self._lib.taco_env_scan_rollout_episodes(self.env._h, C.c_void_p(self.summary_vec.data_ptr()), self._stream()),
                    "taco_env_scan_rollout_episodes")
        return self.summary_vec

    @property
    def count(self):
        """Records appended since attach / the last ``clear`` (dropped ones included).  Synchronises."""
        return int(self._count.item())

    @property
    def dropped(self):
        return max(0, self.count - self.capacity)

    def read(self):
        """The records as a numpy structured array (``ROLLOUT_EPISODE_DTYPE``)."""
        n = min(self.count, self.capacity)
        return self._records[:n * _capi.ROLLOUT_EPISODE_DTYPE.itemsize].cpu().numpy().view(_capi.ROLLOUT_EPISODE_DTYPE)

    def clear(self):
        """Rewind the counter; the episodes in progress continue."""
        _capi.check(self._lib.taco_env_rollout_episodes_clear(self.env._h, self._stream()), "taco_env_rollout_episodes_clear")

    def summary(self):
        """Per-task dict of the last scan's summary (all-reduced when the rollout ran under torch.distributed); see
        ``taco_b200.dist.summarise_episode_summary``.  Synchronises."""
        from .dist import summarise_episode_summary
        return summarise_episode_summary(self.summary_vec)

    def close(self):
        if self._open:
            self._open = False
            self._records = self._count = None
            _capi.check(self._lib.taco_env_detach_rollout_episodes(self.env._h), "taco_env_detach_rollout_episodes")

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_warned_fp32 = set()


def _warn_fp32_fallback(actor_tc, critic_tc):
    """The FP32 CUDA-core kernels are the parity path: 70-100x slower than the tcgen05 kernels at large env counts.  Say so once."""
    import warnings
    which = tuple(n for n, ok in (("actor", actor_tc), ("critic", critic_tc)) if not ok)
    if which and which not in _warned_fp32:
        _warned_fp32.add(which)
        warnings.warn(f"taco_b200: the {' and '.join(which)} shape is outside the tcgen05 kernels' envelope (see include/taco_b200.h); "
                      "falling back to the FP32 CUDA-core kernel, which is 70-100x slower at large env counts", RuntimeWarning, stacklevel=3)


def collect_rollout(env, actor, buffer, value_fn, seed=0, tensor_cores=True, group=None, episodes=None):
    """One rollout of ``buffer.horizon_len`` steps: the data-collection loop of ``PPO.run``
    (IsaacGymEnvs/algorithms/ppo_asymmetry.py:305-342) with no host round trip inside it.

    ``env``: FpvVecTask; ``actor``: ActorMLP (weights loaded); ``value_fn``: a ``CriticLSTM`` (the critic kernels write the value
    straight into ``buffer.value_buf[s]``) or any callable ``value_fn(obs, states) -> (N,1)`` (e.g. a PyTorch critic module).
    Per step -- ``agent.act`` of the reference (nets_asymmetry.py:326-352): the actor kernel samples straight into the buffer
    rows, the critic kernel values the state history, the step kernel writes the next observation history into ring slot s+1
    and reward / done / time-out into row s.  The time-out bootstrap, GAE and the advantage normalisation (with the moments
    all-reduced under torch.distributed) run in ``buffer.compute_returns_and_advantage``; episode statistics come from the
    env's device-side vector, all-reduced once.  Returns the (8,) float64 statistics tensor (see taco_b200.dist.STAT_NAMES).
    ``episodes``: a ``RolloutEpisodes`` of ``env``, scanned after the H steps (before GAE); its ``summary_vec`` is all-reduced too."""
    from . import dist as tdist
    from .critic import CriticLSTM
    torch.cuda.nvtx.range_push("taco.rollout")                    # NVTX: rollout / gae / update ranges (SURVEY.md section 5)
    if env.rollout_buffer is not buffer:
        env.attach_rollout(buffer)
    else:
        env.rewind_rollout()
    buffer.reset()
    H = buffer.horizon_len
    sigma = torch.from_numpy(actor.log_std).to(buffer.device).expand(buffer.num_envs, -1)     # act() returns log_std as `sigma`
    native_critic = isinstance(value_fn, CriticLSTM)
    critic_tc = native_critic and tensor_cores and value_fn.tensor_cores_available
    actor_tc = bool(tensor_cores and actor.tensor_cores_available)        # shapes the tcgen05 kernel rejects use the FP32 kernel
    if tensor_cores and not (actor_tc and (critic_tc or not native_critic)):
        _warn_fp32_fallback(actor_tc, critic_tc or not native_critic)
    for s in range(H):
        obs, states = buffer.obs_ring[s], buffer.states_ring[s]
        out = buffer.rows(s)
        actor.act(obs, env.step_count, seed=seed, env_offset=env.env_offset, tensor_cores=actor_tc, out=out)
        if native_critic:
            value = value_fn.forward(states, tensor_cores=critic_tc, out=buffer.value_buf[s])
        else:
            value = value_fn(obs, states)
        env.step(out[1])
        buffer.store(None, None, out[0], None, out[2], None, value, out[3], sigma, time_outs=True)
    if episodes is not None:
        episodes.scan()
    if native_critic:
        last_value = value_fn.forward(buffer.states_ring[H], tensor_cores=critic_tc)
    else:
        last_value = value_fn(buffer.obs_ring[H], buffer.states_ring[H])
    torch.cuda.nvtx.range_pop()
    torch.cuda.nvtx.range_push("taco.gae")
    buffer.compute_returns_and_advantage(last_value, group=group)
    torch.cuda.nvtx.range_pop()
    if episodes is not None:
        tdist.allreduce_episode_summary(episodes.summary_vec, group=group)
    return tdist.allreduce_rollout_stats(env.stats(), group=group)


class GraphedRollout:
    """``collect_rollout`` captured ONCE as a CUDA graph and replayed: rewind -> horizon x (actor.act -> critic -> env.step) -> last
    value -> GAE + normalisation -> statistics are ~3 H + 6 kernel launches that a replay submits with one call, with the critic
    chain as a parallel branch next to the actor -> step chain.  At the reference's
    own scale (4096 envs) the eager loop is bound by Python / launch overhead (~300 us per step against ~65 us of GPU work); the
    replay is not.  The env's step index lives in a device counter while the graph exists (``FpvVecTask.graph_begin``), so every
    replay draws fresh Philox numbers: replays are bit-identical to the eager loop (tests/test_rollout_gpu.py).

    The constructor collects the first rollout eagerly (``first_stats``); every ``run()`` is one more.
    ``critic`` must be a ``CriticLSTM``; weights may be reloaded between replays (``ActorMLP.load`` / ``CriticLSTM.load`` write the
    same device buffers, ``ActorMLP.set_log_std`` the sampler constants the captured kernels read from device memory) and
    ``env.difficulty`` may be set between replays (graph-mode launches read its device copy).  Single-process statistics / advantage normalisation are inside the
    graph; under torch.distributed the two small all-reduces run after the replay.  ``episodes``: a ``RolloutEpisodes`` of ``env``
    whose scan is captured after the H steps; every ``run()`` leaves that rollout's summary in ``episodes.summary_vec``
    (all-reduced under torch.distributed, like the statistics)."""

    def __init__(self, env, actor, buffer, critic, seed=0, tensor_cores=True, group=None, episodes=None):
        from . import dist as tdist
        from .critic import CriticLSTM
        if not isinstance(critic, CriticLSTM):
            raise TypeError("GraphedRollout needs the native critic (CriticLSTM)")
        self.env, self.actor, self.buffer, self.critic, self.group = env, actor, buffer, critic, group
        self.episodes = episodes
        self.seed = int(seed)
        self.tc_actor = bool(tensor_cores and actor.tensor_cores_available)
        self.tc_critic = bool(tensor_cores and critic.tensor_cores_available)
        self._tdist = tdist
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        # The FIRST rollout is collected eagerly, here: it leaves the ring cursor at H (so that the captured rewind contains the
        # slot H -> slot 0 copy), runs every lazy initialisation outside the capture, and its experience is in ``buffer`` like
        # that of any later ``run()``.
        self.first_stats = collect_rollout(env, actor, buffer, critic, seed=self.seed, tensor_cores=tensor_cores, group=group,
                                           episodes=episodes)
        H = buffer.horizon_len
        self.stats = torch.zeros(8, dtype=torch.float64, device=buffer.device)
        self.last_value = torch.empty(buffer.num_envs, 1, dtype=torch.float32, device=buffer.device)
        buffer.rows(0)                                          # allocate the clipped-action scratch outside the capture
        self._side = torch.cuda.Stream(device=buffer.device)    # the critic's branch of the graph
        torch.cuda.synchronize(buffer.device)
        env.graph_begin()
        steps_before = env.step_count
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._body()
        env.step_count = steps_before                           # the capture advanced the host mirrors without running anything
        self.replays = 0

    def _body(self):
        env, buf, H = self.env, self.buffer, self.buffer.horizon_len
        counter = env.step_counter()[0]
        base = env.step_count
        # two branches of the graph: actor -> step -> actor -> ... on the capturing stream, and the critic chain beside it (the value
        # of slot s needs only the state history step s-1 wrote, nothing downstream needs it before GAE).  At small env counts both
        # chains are latency-bound single-wave kernels on disjoint SMs, so they overlap fully.
        main = torch.cuda.current_stream(buf.device)
        side = self._side
        env.rewind_rollout()
        for s in range(H + 1):
            ev = torch.cuda.Event()
            ev.record(main)                                       # slot s is complete (rewind, or step s-1)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                self.critic.forward(buf.states_ring[s], tensor_cores=self.tc_critic, out=buf.value_buf[s] if s < H else self.last_value)
            if s == H:
                break
            out = buf.rows(s)
            self.actor.act(buf.obs_ring[s], env.step_count - base, seed=self.seed, env_offset=env.env_offset, tensor_cores=self.tc_actor,
                           out=out, step_base=counter)
            env.step_raw(out[1])
        if self.episodes is not None:
            self.episodes.scan()                                  # before graph_advance: it reads the counter the steps used
        env.graph_advance(H)
        done = torch.cuda.Event()
        done.record(side)
        main.wait_event(done)                                     # join: every value is written
        buf.step, buf._have_timeouts = H, True
        if self.world == 1:
            buf.compute_returns_and_advantage(self.last_value)
        env.stats(out=self.stats)

    def run(self):
        """One rollout.  Returns the (8,) float64 statistics tensor (all-reduced under torch.distributed)."""
        torch.cuda.nvtx.range_push("taco.rollout_graph")
        self.graph.replay()
        torch.cuda.nvtx.range_pop()
        self.replays += 1
        self.env.step_count += self.buffer.horizon_len
        if self.world > 1:
            self.buffer.compute_returns_and_advantage(self.last_value, group=self.group)
        if self.episodes is not None:
            self._tdist.allreduce_episode_summary(self.episodes.summary_vec, group=self.group)
        return self._tdist.allreduce_rollout_stats(self.stats, group=self.group)

    def close(self):
        """Leave graph mode (the library reads the step index back from the device)."""
        if self.graph is not None:
            self.graph = None
            self.env.graph_end()
