"""Generate tests/golden/*.npz by RUNNING THE REFERENCE'S OWN torch modules (imported
unmodified through oracle/ref_loader.py) on seeded inputs.  TEST INFRASTRUCTURE.

Run in the build container only (needs /root/reference):

    python -m oracle.make_golden

The reference ships no tests / golden vectors for this path (SURVEY.md section 4), so these
files are the pin for the oracle's leaf functions: tests/test_oracle_golden.py checks
oracle/{leaf_math,dynamics,rewards,actor,critic}.py against them on any machine.
"""
import os
import math

import numpy as np
import torch

from . import ref_loader

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _rand_quat(g, n, normalised=True):
    q = torch.randn(n, 4, generator=g)
    if normalised:
        q = q / q.norm(dim=1, keepdim=True)
    return q


def leaf_math(ns):
    g = torch.Generator().manual_seed(1001)
    n = 257
    tu, jit = ns.torch_utils, ns.jit_utils
    a, b = _rand_quat(g, n), _rand_quat(g, n)
    raw = _rand_quat(g, n, normalised=False) * 1.7
    v = torch.randn(n, 3, generator=g) * 5
    eul = (torch.rand(n, 3, generator=g) * 2 - 1) * math.pi
    # gimbal / saturation corner cases for euler extraction
    a[0] = torch.tensor([0.0, math.sqrt(0.5), 0.0, math.sqrt(0.5)])
    a[1] = torch.tensor([0.0, -math.sqrt(0.5), 0.0, math.sqrt(0.5)])
    a[2] = torch.tensor([0.0, 0.0, 0.0, 1.0])
    a[3] = torch.tensor([1.0, 0.0, 0.0, 0.0])
    r, p, y = tu.get_euler_xyz_v1(a)
    out = dict(
        a=a, b=b, raw=raw, v=v, eul=eul,
        quat_mul=tu.quat_mul(a, b),
        quat_conjugate=tu.quat_conjugate(a),
        quat_rotate=tu.quat_rotate(a, v),
        quat_rotate_conj=tu.quat_rotate(tu.quat_conjugate(a), v),
        euler=torch.stack((r, p, y), dim=1),
        quat_from_euler=tu.quat_from_euler_xyz(eul[:, 0], eul[:, 1], eul[:, 2]),
        rotmat=jit.quaternion_to_matrix(raw).reshape(n, 9),
        rotmat_unit=jit.quaternion_to_matrix(a).reshape(n, 9),
        quat_diff_rad=jit.quat_diff_rad(a, b),
        rand_float=tu.torch_rand_float(-math.pi, math.pi, (4, 3), "cpu"),  # shape/API check only
    )
    u = torch.rand(n, generator=g)
    out["u"] = u
    out["rand_range_pi"] = (math.pi - (-math.pi)) * u + (-math.pi)       # torch_utils.py:219 evaluated on given u
    np.savez(os.path.join(OUT, "leaf_math.npz"), **{k: np.asarray(t) for k, t in out.items()})


def dynamics(ns):
    g = torch.Generator().manual_seed(2002)
    n = 64
    dt = float(np.float32(0.001))
    out = {}
    # ---- body-rate PID: 6 consecutive calls, with exact-zero errors mixed in (quirk 9)
    pid = ns.angvel_control.angvel_control(1, 0, n, "cpu", dt)
    sp = (torch.rand(6, n, 3, generator=g) * 2 - 1) * 20
    w = torch.randn(6, n, 3, generator=g) * 8
    w[0, :8] = sp[0, :8]                      # zero error on first call
    w[2, 8:16, 1] = sp[2, 8:16, 1]
    sp[3, 16:20] = 900.0                      # saturate the +-400 error clip
    res, prev = [], []
    for i in range(6):
        res.append(pid.compute(sp[i], w[i]).clone())
        prev.append(pid.previous_error.clone())
    out.update(pid_sp=sp, pid_w=w, pid_out=torch.stack(res), pid_prev=torch.stack(prev))
    # ---- allocator
    alloc = ref_loader.make_allocator(ns)
    u = torch.cat((torch.rand(n, 1, generator=g) * 1000, torch.randn(n, 3, generator=g) * 150), dim=1)
    u[:6, 0] = torch.tensor([0.0, 1000.0, 1000.0, 50.0, 999.0, 500.0])
    u[1, 1:] = torch.tensor([300.0, 300.0, 600.0])
    out["alloc_u"] = u.clone()
    out["alloc_thr"] = alloc.control_allocator(u.clone())
    # ---- battery: 40 calls with time-varying power, random initial charge
    bat = ns.battery_dynamics.Battery_Dynamics(n, "cpu", True, dt)
    bat.E_c[:] = torch.rand(n, 1, generator=g) * 2.2
    pm = torch.rand(40, n, 1, generator=g) * 1500
    pm[0] = 0.0
    out["bat_ec0"] = bat.E_c.clone()
    volts = [bat.sim_process(pm[i]).clone() for i in range(40)]
    out.update(bat_pm=pm, bat_volt=torch.stack(volts), bat_u1=bat.u_1.clone(), bat_ec=bat.E_c.clone(), bat_t=bat.time.clone())
    bat_off = ns.battery_dynamics.Battery_Dynamics(n, "cpu", False, dt)
    out["bat_off_volt"] = bat_off.sim_process(pm[1]).clone()
    # ---- rotor lag with randomised per-env polynomial and response time
    rot = ns.thrust_dynamics.RotorDynamics(n, "cpu", 0.017)
    rot.omega_para = rot.omega_para_init * (0.95 + 0.1 * torch.rand(n, 5, generator=g))
    rot.response_time = 0.016 + 0.002 * torch.rand(n, 4, generator=g)
    volt = 20 + 6 * torch.rand(12, n, 1, generator=g)
    thr = 100 + 900 * torch.rand(12, n, 4, generator=g)
    om = torch.rand(n, 4, generator=g) * 400
    out.update(rot_poly=rot.omega_para.clone(), rot_tau=rot.response_time.clone(), rot_volt=volt, rot_thr=thr, rot_om0=om.clone())
    oms = []
    for i in range(12):
        om = rot.sim_process(volt[i], thr[i], om)
        oms.append(om.clone())
    out["rot_om"] = torch.stack(oms)
    # ---- aero + remap + mechanical power
    aero = ns.thrust_dynamics.AeroDynamics(n, "cpu")
    aero.para_force_torque = aero.para_force_torque_init * (0.95 + 0.1 * torch.rand(n, 2, generator=g))
    aero.para_d = aero.para_d_init * (0.95 + 0.1 * torch.rand(n, 2, generator=g))
    aero.para_t = aero.para_t_init * (0.95 + 0.1 * torch.rand(n, 1, generator=g))
    vb = torch.randn(n, 3, generator=g) * 4
    om = torch.rand(n, 4, generator=g) * 800
    f, tq, bf, bt = aero.sim_process(vb, om)
    out.update(aero_par=torch.cat((aero.para_force_torque, aero.para_d, aero.para_t), dim=1), aero_vb=vb, aero_om=om,
               aero_f=f.clone(), aero_tq=tq.clone(), aero_bf=bf.clone(), aero_bt=bt.clone())
    fs, ts = alloc.sim_process(f.clone(), tq.clone())
    out.update(remap_f=fs, remap_tq=ts)
    out["mech_power"] = torch.sum(400 * (om * 2 * torch.pi / 4500) ** 3, dim=1).unsqueeze(1)   # fpv_asymmetry.py:614 verbatim expression
    np.savez(os.path.join(OUT, "dynamics.npz"), **{k: np.asarray(t) for k, t in out.items()})


def rewards(ns):
    g = torch.Generator().manual_seed(3003)
    n = 128
    tr = ns.task_reward
    rel_body = torch.randn(n, 3, generator=g) * 3
    rel_body[:4] *= 10                                   # dist > 10 -> die
    rel_world = torch.randn(n, 3, generator=g) * 2
    rel_world[5] = torch.tensor([0.0, 0.0, 1.0])         # degenerate horizontal direction (eps path)
    rel_vel = torch.randn(n, 3, generator=g) * 3
    cpos = torch.randn(n, 3, generator=g) + torch.tensor([0.0, 0.0, 2.0])
    cpos[6:10, 2] = torch.tensor([0.05, 0.1, 0.0999, -1.0])
    cq, tq = _rand_quat(g, n), _rand_quat(g, n)
    relq = _rand_quat(g, n)
    cmd_rot = torch.stack((torch.ones(n), (torch.rand(n, generator=g) * 2 - 1) * 6), dim=1)
    cmd_flip = torch.stack((-torch.ones(n), (torch.rand(n, generator=g) * 2 - 1) * 2 * math.pi), dim=1)
    reset = torch.zeros(n, dtype=torch.long)
    prog = torch.randint(0, 1000, (n,), generator=g)
    prog[10:14] = torch.tensor([998, 999, 1000, 997])
    max_len = 1000.0
    rp, xp = tr.compute_pos_reward(rel_body, cpos, cq, tq, reset, prog, max_len)
    rr, xr = tr.compute_rotating_reward(rel_world.clone(), rel_vel, cpos, cq, cmd_rot, reset, prog, max_len)
    rf, xf = tr.compute_flip_reward(rel_body, relq, cpos, cmd_flip, reset, prog, max_len)
    out = dict(rel_body=rel_body, rel_world=rel_world, rel_vel=rel_vel, cpos=cpos, cq=cq, tq=tq, relq=relq,
               cmd_rot=cmd_rot, cmd_flip=cmd_flip, prog=prog, pos_rew=rp, pos_reset=xp, rot_rew=rr, rot_reset=xr,
               flip_rew=rf, flip_reset=xf)
    np.savez(os.path.join(OUT, "rewards.npz"), **{k: np.asarray(t) for k, t in out.items()})


def actor(ns):
    """MLP.forward, PPO_ActorCritic.act (nets_asymmetry.py:23-39,:326-346) and PPO.spectral_normalize_actors
    (ppo_asymmetry.py:398-404) run from the reference's own classes."""
    import types
    import torch.nn as nn
    torch.manual_seed(2024)
    hidden = [64, 128]
    para = {"actor_critic_mlp_dict": {"actor_input_dim": 26, "actor_output_dim": 4, "critic_input_dim": 26 * 5, "critic_output_dim": 1,
                                      "actor_hidden_sizes": hidden, "critic_hidden_sizes": [32], "activation": nn.ReLU},
            "use_actor_encoder": False, "use_critic_encoder": False, "share_encoder": False}
    import io, contextlib
    with contextlib.redirect_stdout(io.StringIO()):        # the constructor prints the net structure
        agent = ns.nets.PPO_ActorCritic(para)
    lin = [m for m in agent.actor_mlp.layers if isinstance(m, nn.Linear)]
    with torch.no_grad():                                   # "trained" weights: orthogonal init + drift, so the sigmas differ
        for i, m in enumerate(lin):
            m.weight += 0.05 * (i + 1) * torch.randn_like(m.weight) * m.weight.abs().mean() * 4
            m.bias.uniform_(-0.2, 0.2)
        agent.log_std.copy_(torch.tensor([-0.5, -0.25, 0.0, 0.1]))
    n = 96
    obs = torch.randn(n, 1, 26) * 0.8
    states = torch.randn(n, 5, 26)
    out = {}
    for i, m in enumerate(lin):
        out[f"w{i}"] = m.weight.detach().clone()
        out[f"b{i}"] = m.bias.detach().clone()
    out["obs"] = obs
    with torch.no_grad():
        out["mean"] = agent.actor_mlp(obs)
        torch.manual_seed(77)
        action, logp, value, mean, log_std = agent.act(obs, states)
    out["act_action"], out["act_logp"], out["act_mean"], out["log_std"] = action, logp, mean, log_std[0]
    e = agent.log_std.detach().exp()
    out["act_eps"] = (action - mean) / (e * e)              # the noise torch drew, recovered for injection into the oracle
    # spectral projection through the reference's own method (needs only self.agent)
    lipschitz = 1.2
    assert ns.ppo is not None, getattr(ns, "ppo_error", None)
    out["sigma_before"] = torch.stack([torch.linalg.matrix_norm(m.weight.detach(), ord=2) for m in lin])
    ns.ppo.PPO.spectral_normalize_actors(types.SimpleNamespace(agent=agent), lipschitz_const=lipschitz)
    for i, m in enumerate(lin):
        out[f"w{i}_proj"] = m.weight.detach().clone()
    out["lipschitz"] = torch.tensor(lipschitz)
    with torch.no_grad():
        out["mean_proj"] = agent.actor_mlp(obs)
    np.savez(os.path.join(OUT, "actor.npz"), **{k: np.asarray(t) for k, t in out.items()})


def critic(ns):
    """LSTMEncoder.forward + critic MLP + the critic branch of PPO_ActorCritic.act (nets_asymmetry.py:128-136,:23-39,:350-352)
    run from the reference's own classes (use_critic_encoder=True, critic_encoder_type=LSTM: the README's training command)."""
    import io, contextlib
    import torch.nn as nn
    out = {}
    for tag, hid, nl, mlp_hidden in (("a", 48, 1, [64, 32]), ("b", 32, 2, [40])):
        torch.manual_seed(4100 + nl)
        para = {"actor_critic_mlp_dict": {"actor_input_dim": 26, "actor_output_dim": 4, "critic_input_dim": 26 * 5, "critic_output_dim": 1,
                                          "actor_hidden_sizes": [32], "critic_hidden_sizes": mlp_hidden, "activation": nn.ReLU},
                "use_actor_encoder": False, "use_critic_encoder": True, "share_encoder": False, "critic_encoder_type": "LSTM",
                "critic_encoder_dict": {"encoder_type": "LSTM", "input_size": 26, "output_size": hid, "num_layers": nl, "bidirectional": False}}
        with contextlib.redirect_stdout(io.StringIO()):
            agent = ns.nets.PPO_ActorCritic(para)
        lstm = agent.critic_encoder.layers
        lin = [m for m in agent.critic_mlp.layers if isinstance(m, nn.Linear)]
        with torch.no_grad():                               # para_init zeroes the LSTM biases: give them values so all four terms count
            for name, prm in lstm.named_parameters():
                if prm.dim() == 1:
                    prm.uniform_(-0.3, 0.3)
            for m in lin:
                m.bias.uniform_(-0.2, 0.2)
            lin[-1].weight.mul_(30.0)                       # gain 0.01 would make the value ~1e-2: scale it into O(1)
        n = 80
        obs = torch.randn(n, 1, 26) * 0.8
        states = torch.randn(n, 5, 26) * 1.5
        for l in range(nl):
            for nm in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                out[f"{tag}_{nm}_l{l}"] = getattr(lstm, f"{nm}_l{l}").detach().clone()
        for i, m in enumerate(lin):
            out[f"{tag}_w{i}"] = m.weight.detach().clone()
            out[f"{tag}_b{i}"] = m.bias.detach().clone()
        out[f"{tag}_states"] = states
        with torch.no_grad():
            out[f"{tag}_enc"] = agent.critic_encoder(states)
            out[f"{tag}_value"] = agent.critic_mlp(agent.critic_encoder(states))
            _, _, value, _, _ = agent.act(obs, states)
        out[f"{tag}_act_value"] = value
    np.savez(os.path.join(OUT, "critic.npz"), **{k: np.asarray(t) for k, t in out.items()})


def ppo_update(ns):
    """PPO.update (ppo_asymmetry.py:137-258) run from the reference's own class on a small fixed buffer: the PPO object is built
    without __init__ (which needs an env and TensorBoard) and given exactly the attributes update() reads; the agent is the
    reference's PPO_ActorCritic (MLP actor, LSTM critic encoder); minibatch indices are fixed.  Two cases: plain, and with the
    spectral projection after every optimiser step."""
    _ppo_update_cases(ns, 6, 16, 3, [32, 24], [20], 16, "ppo_update.npz")
    # shapes the native update (taco_ppo_*, tcgen05 GEMMs) supports: LSTM width 64, hidden widths multiples of 16, minibatches of 256
    _ppo_update_cases(ns, 8, 64, 2, [64, 48], [32], 64, "ppo_update_native.npz")


def _ppo_update_cases(ns, H, N, mb, actor_hidden, critic_hidden, lstm_hidden, file_name):
    import io, contextlib, types
    import torch.nn as nn
    out = {}
    for tag, use_lip in (("plain", False), ("lip", True)):
        torch.manual_seed(900)
        para = {"actor_critic_mlp_dict": {"actor_input_dim": 26, "actor_output_dim": 4, "critic_input_dim": 26 * 5, "critic_output_dim": 1,
                                          "actor_hidden_sizes": list(actor_hidden), "critic_hidden_sizes": list(critic_hidden), "activation": nn.ReLU},
                "use_actor_encoder": False, "use_critic_encoder": True, "share_encoder": False, "critic_encoder_type": "LSTM",
                "critic_encoder_dict": {"encoder_type": "LSTM", "input_size": 26, "output_size": lstm_hidden, "num_layers": 1, "bidirectional": False}}
        with contextlib.redirect_stdout(io.StringIO()):
            agent = ns.nets.PPO_ActorCritic(para)
        with torch.no_grad():                                   # gains that make the projection bite on some layers only
            for i, m in enumerate(mm for mm in agent.actor_mlp.layers if isinstance(mm, nn.Linear)):
                m.weight.mul_(1.0 + 0.6 * i)
        for k, v in agent.state_dict().items():
            out[f"{tag}_init__{k}"] = v.detach().clone()
        g = torch.Generator().manual_seed(901)
        buf = types.SimpleNamespace(
            obs_buf=torch.randn(H, N, 1, 26, generator=g) * 0.7, states_buf=torch.randn(H, N, 5, 26, generator=g) * 0.7,
            act_buf=torch.randn(H, N, 4, generator=g).clamp(-1.5, 1.5), value_buf=torch.randn(H, N, 1, generator=g) * 0.3,
            ret_buf=torch.randn(H, N, 1, generator=g) * 0.5, done_buf=torch.zeros(H, N, 1), logp_buf=torch.randn(H, N, 1, generator=g) * 0.3 - 4.0,
            adv_buf=torch.randn(H, N, 1, generator=g), mu_buf=torch.zeros(H, N, 4), sigma_buf=torch.zeros(H, N, 4))
        with torch.no_grad():                                   # old log-probs of the initial policy + noise, so ratios stay near 1
            lp, _, _, _, _ = agent.evaluate(buf.obs_buf.view(-1, 1, 26), buf.states_buf.view(-1, 5, 26), buf.act_buf.view(-1, 4))
            buf.logp_buf = (lp + 0.02 * torch.randn(lp.shape, generator=g)).view(H, N, 1)
        idx = torch.randperm(H * N, generator=g).reshape(mb, -1).tolist()
        buf.batch_idx_generator = lambda: idx
        ppo = object.__new__(ns.ppo.PPO)
        cfg = dict(clip=0.2, target_kl=0.5, max_grad=0.5, use_clipped_value_loss=False, epochs=40, train_iters=2, lr=1e-3, pi_coef=1.0, vf_coef=0.5,
                   ent_coef=0.01, learning_rate_schedule=True, lr_ratio=0.3, lr_lp_index=0.7, lr_epoch_index=30, use_lipschitz=use_lip,
                   lipschitz_para=2.0, lipschitz_schedule=True, lip_ratio=[1.0, 0.3], lip_lp_index=[0.3, 0.7], lip_epoch_index=[5, 30],
                   difficulty_schedule=True, diff_value=[0.1, 1.0], diff_lp_index=[0.3, 0.7], diff_epoch_index=[5, 30])
        for k, v in cfg.items():
            setattr(ppo, k, v)
        ppo.agent, ppo.replay_buffer, ppo.env = agent, buf, types.SimpleNamespace(difficulty=0.0)
        ppo.optimizer = torch.optim.Adam(filter(lambda p: p.requires_grad, agent.parameters()), lr=cfg["lr"], eps=1e-5)
        ppo.optim_step = 0
        logged = {}
        ppo.writer = types.SimpleNamespace(add_scalar=lambda name, val, step: logged.__setitem__(name, float(val)))
        epoch = 12
        with contextlib.redirect_stdout(io.StringIO()):
            ppo.update(epoch)
        for k, v in agent.state_dict().items():
            out[f"{tag}_final__{k}"] = v.detach().clone()
        for k in ("obs_buf", "states_buf", "act_buf", "value_buf", "ret_buf", "logp_buf", "adv_buf"):
            out[f"{tag}_buf__{k}"] = getattr(buf, k)
        out[f"{tag}_idx"] = torch.tensor(idx)
        out[f"{tag}_epoch"] = torch.tensor(epoch)
        out[f"{tag}_optim_step"] = torch.tensor(ppo.optim_step)
        out[f"{tag}_difficulty"] = torch.tensor(ppo.env.difficulty)
        for name, val in logged.items():
            out[f"{tag}_log__{name.split('/')[1].rstrip(':')}"] = torch.tensor(val)
    if file_name == "ppo_update_native.npz":            # keeps the file under 1 MB: lip_ arrays equal to their plain_ twins are stored once
        out = {k: v for k, v in out.items() if not (k.startswith("lip_") and torch.equal(v, out["plain_" + k[4:]]))}
    np.savez_compressed(os.path.join(OUT, file_name), **{k: np.asarray(t) for k, t in out.items()})


def gae(ns):
    """PPOReplayBuffer.store / compute_returns_and_advantage (buffer_asymmetry.py:49-68,93-132) run from the reference's
    own class, with the time-out bootstrap of ppo_asymmetry.py:313-324 applied to the stored reward."""
    torch.manual_seed(31)
    H, N, gamma, lam = 12, 77, 0.99, 0.95
    buf = ns.buffer.PPOReplayBuffer(N, 26, 1, 26, 5, 4, H, 4, gamma, lam, "cpu")
    rew = torch.rand(H, N) * 0.02
    value = torch.randn(H, N, 1) * 0.3 + 0.5
    done = (torch.rand(H, N) < 0.08).float()
    time_outs = (torch.rand(H, N) < 0.5)
    last_value = torch.randn(N, 1) * 0.3 + 0.5
    rew_aug = rew.clone()
    for s in range(H):
        # ppo_asymmetry.py:313-324: truncated envs get gamma * V(pre-step obs, states) = gamma * value[s]
        ids = (time_outs[s] * done[s]).nonzero(as_tuple=False).squeeze(-1).tolist()
        r = rew[s].clone()
        if ids:
            r[ids] += gamma * value[s, ids].squeeze()
        rew_aug[s] = r
        z = torch.zeros
        buf.store(z(N, 1, 26), z(N, 5, 26), z(N, 4), r, z(N), done[s], value[s], z(N, 4), z(N, 4))
    buf.compute_returns_and_advantage(last_value)
    out = dict(rew=rew, rew_aug=rew_aug, value=value, done=done, time_outs=time_outs.to(torch.uint8), last_value=last_value,
               gamma=torch.tensor(gamma), lam=torch.tensor(lam), adv_norm=buf.adv_buf, ret=buf.ret_buf)
    np.savez(os.path.join(OUT, "gae.npz"), **{k: np.asarray(t) for k, t in out.items()})


def main():
    assert ref_loader.available(), "needs the reference tree (build container only)"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)
    ns = ref_loader.load()
    leaf_math(ns)
    dynamics(ns)
    rewards(ns)
    actor(ns)
    critic(ns)
    ppo_update(ns)
    gae(ns)
    print("golden vectors written to", OUT)
    for f in sorted(os.listdir(OUT)):
        print("  ", f, os.path.getsize(os.path.join(OUT, f)), "bytes")


if __name__ == "__main__":
    main()
