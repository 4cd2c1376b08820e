"""Stacked-LSTM critics (nn.LSTM(in, H, L), L = 2..4) on the tcgen05 critic kernel: one launch per layer over chunks of the batch,
the layers handing h over through a workspace.  GPU only.

Bars, as for the one-layer kernel (tests/test_critic_gpu.py): <= 1.5e-2 absolute on O(1) values against the bf16-operand
emulation of the whole stack (oracle/critic.py: critic_forward_bf16 -- bf16 operands, fp32 bias, gates and cell state, h rounded
to bf16 as the next product's operand, in every layer), <= 6e-2 against the FP32 kernel.  The layers above the bottom add their
bias in fp32 in the epilogue (the bottom layer carries it as a bf16 hi / lo pair inside the MMA).
"""
import warnings

import pytest
import torch

from test_critic_gpu import _random_critic

pytestmark = pytest.mark.gpu

BIG_N = 200_003     # several workspace chunks (4 waves of tile pairs = 151 552 rows on a 148-SM B200), the last one ragged


def _states(n, seq_len, in_dim, seed):
    return torch.randn(n, seq_len, in_dim, generator=torch.Generator().manual_seed(seed)) * 1.2


def _check(c, states, lstm, w, b, tag):
    """tensor-core values against the emulation (a prefix and a suffix of the rows) and the FP32 kernel; returns them"""
    from oracle import critic as oc
    n = states.shape[0]
    v_tc = c.forward(states.cuda(), tensor_cores=True).cpu()
    v_fp = c.forward(states.cuda(), tensor_cores=False).cpu()
    assert torch.isfinite(v_tc).all()
    m = min(n, 4096)                                      # the CPU emulation is slow: check a prefix and a suffix of the rows
    for sl in (slice(0, m), slice(n - m, n)):
        emu = oc.critic_forward_bf16(states[sl], lstm, w, b)
        if n >= 64:
            assert float(emu.abs().mean()) > 0.05
        err = (v_tc[sl] - emu).abs().max().item()
        print(f"stacked critic tc vs bf16 emulation: {tag} n={n} rows {sl.start}:{sl.stop} max|err|={err:.2e} mean|v|={float(emu.abs().mean()):.3f}")
        assert err <= 1.5e-2
    err32 = (v_tc - v_fp).abs().max().item()
    print(f"stacked critic tc vs fp32 kernel: {tag} n={n} max|err|={err32:.2e}")
    assert err32 <= 6e-2
    return v_tc


@pytest.mark.parametrize("mlp_hidden", [[256, 256, 256], [64]])
@pytest.mark.parametrize("hid", [64, 32, 16])
@pytest.mark.parametrize("layers", [2, 3, 4])
def test_tensor_core_path_vs_emulation(layers, hid, mlp_hidden):
    from taco_b200 import CriticLSTM
    lstm, w, b = _random_critic(26, hid, mlp_hidden, seed=10 * layers + hid + len(mlp_hidden), nl=layers)
    c = CriticLSTM(26, 5, hid, mlp_hidden, lstm_layers=layers)
    assert c.tensor_cores_available
    c.load(lstm, w, b)
    for n in (1, 127, 300, 40_000):
        _check(c, _states(n, 5, 26, 7 + n + layers), lstm, w, b, f"L={layers} H={hid} mlp={mlp_hidden}")
    c.close()


@pytest.mark.parametrize("layers", [2, 3])
@pytest.mark.parametrize("in_dim,seq_len,hid", [(26, 1, 64), (26, 8, 32), (30, 5, 64), (2, 3, 16), (2, 8, 64)])
def test_tensor_core_path_other_sequence_shapes(layers, in_dim, seq_len, hid):
    """A single frame, the longest supported history, the widest and the narrowest even input."""
    from taco_b200 import CriticLSTM
    lstm, w, b = _random_critic(in_dim, hid, [64], seed=in_dim * 100 + seq_len + layers, nl=layers)
    c = CriticLSTM(in_dim, seq_len, hid, [64], lstm_layers=layers)
    assert c.tensor_cores_available
    c.load(lstm, w, b)
    _check(c, _states(777, seq_len, in_dim, in_dim + seq_len), lstm, w, b, f"L={layers} in={in_dim} T={seq_len} H={hid}")
    c.close()


@pytest.mark.parametrize("layers,hid", [(3, 32), (3, 64), (4, 64)])
def test_several_chunks_and_launch_shape_invariance(layers, hid):
    """A batch of several workspace chunks with a ragged last one.  Rows computed as part of that batch equal bitwise the same rows
    computed by a 4096-row call (one tile per CTA): rows [0, 4096) (every CTA's first tile), rows of chunk 0 that a CTA runs as its
    second tile pair (tiles 300-331; a layer's last step there stages the slot's next tile while the row's other half may still be
    in its gate math), and the last 4096 rows (second pairs of the ragged last chunk)."""
    from taco_b200 import CriticLSTM
    lstm, w, b = _random_critic(26, hid, [256, 256, 256], seed=41 + hid, nl=layers)
    c = CriticLSTM(26, 5, hid, [256, 256, 256], lstm_layers=layers)
    c.load(lstm, w, b)
    states = _states(BIG_N, 5, 26, 3)
    v_big = _check(c, states, lstm, w, b, f"L={layers} H={hid} several chunks")
    for r0 in (0, 300 * 128, BIG_N - 4096):
        v_small = c.forward(states[r0:r0 + 4096].cuda(), tensor_cores=True).cpu()
        assert torch.equal(v_small, v_big[r0:r0 + 4096]), r0
    c.close()


def test_reload_in_place_equals_a_fresh_handle():
    from taco_b200 import CriticLSTM
    a = _random_critic(26, 64, [256, 256], seed=5, nl=3)
    bw = _random_critic(26, 64, [256, 256], seed=6, nl=3)
    states = _states(50_000, 5, 26, 9).cuda()
    c = CriticLSTM(26, 5, 64, [256, 256], lstm_layers=3)
    c.load(*a)
    v_a = c.forward(states, tensor_cores=True).clone()
    c.load(*bw)
    v_b = c.forward(states, tensor_cores=True).clone()
    fresh = CriticLSTM(26, 5, 64, [256, 256], lstm_layers=3)
    fresh.load(*bw)
    assert torch.equal(v_b, fresh.forward(states, tensor_cores=True))
    assert not torch.equal(v_a, v_b)
    c.close(); fresh.close()


def _rollout_nets(layers, hid, mlp, seed):
    from taco_b200 import ActorMLP, CriticLSTM
    gen = torch.Generator().manual_seed(seed)
    sizes = [26, 64, 64, 4]
    aw = [torch.randn(sizes[i + 1], sizes[i], generator=gen) * 0.25 for i in range(3)]
    ab = [torch.zeros(sizes[i + 1]) for i in range(3)]
    actor, critic = ActorMLP(26, [64, 64], 4), CriticLSTM(26, 5, hid, mlp, lstm_layers=layers)
    actor.load(aw, ab, log_std=torch.full((4,), -0.3))
    return actor, critic


def test_collect_rollout_uses_the_tensor_core_critic():
    import taco_b200.rollout as ro
    from taco_b200 import FpvVecTask, RolloutBuffer, collect_rollout, make_cfg
    n, H = 3000, 6
    actor, critic = _rollout_nets(2, 64, [256, 256, 256], 1)
    critic.load(*_random_critic(26, 64, [256, 256, 256], seed=12, nl=2))
    assert critic.tensor_cores_available
    env = FpvVecTask(make_cfg("flip", n, **{"env.maxEpisodeLength": 9}), seed=3)
    buf = RolloutBuffer(n, 26, 1, 26, 5, 4, H, 1, 0.99, 0.95, "cuda:0")
    ro._warned_fp32.clear()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        collect_rollout(env, actor, buf, critic, seed=4, tensor_cores=True)
        torch.cuda.synchronize()
    assert not [x for x in caught if issubclass(x.category, RuntimeWarning)]
    for s in range(H):
        assert torch.equal(buf.value_buf[s], critic.forward(buf.states_ring[s], tensor_cores=True)), s
    env.close(); actor.close(); critic.close()


def test_graphed_rollout_replays_are_bit_identical_to_the_eager_loop():
    """As the one-layer test in test_rollout_gpu.py, with an L = 2, H = 64 critic whose weights are reloaded between the rollouts:
    the captured graph keeps the handle's images, bias blocks and workspace, which load rewrites in place."""
    from taco_b200 import FpvVecTask, GraphedRollout, RolloutBuffer, collect_rollout, make_cfg
    n, H = 3000, 7
    crit = [_random_critic(26, 64, [256, 256], seed=20 + k, nl=2) for k in range(3)]
    runs = {}
    for mode in ("eager", "graph"):
        env = FpvVecTask(make_cfg("flip", n, **{"env.maxEpisodeLength": 9}), seed=21)
        actor, critic = _rollout_nets(2, 64, [256, 256], 2)
        buf = RolloutBuffer(n, 26, 1, 26, 5, 4, H, 1, 0.99, 0.95, "cuda:0")
        snaps, gr = [], None
        for k in range(3):
            critic.load(*crit[k])
            if mode == "eager":
                stats = collect_rollout(env, actor, buf, critic, seed=4, tensor_cores=True)
            elif k == 0:
                gr = GraphedRollout(env, actor, buf, critic, seed=4, tensor_cores=True)
                assert gr.tc_critic
                stats = gr.first_stats
            else:
                stats = gr.run()
            torch.cuda.synchronize()
            snaps.append([t.clone() for t in (buf.states_ring, buf.act_buf, buf.value_buf, buf.rew_buf, buf.done_buf, buf.ret_buf, buf.adv_buf, stats)])
        if gr is not None:
            gr.close()
        runs[mode] = snaps
        env.close(); actor.close(); critic.close()
    for k, (a, b) in enumerate(zip(runs["eager"], runs["graph"])):
        for j, (ta, tb) in enumerate(zip(a, b)):
            assert torch.equal(ta, tb), (k, j)
    assert not torch.equal(runs["eager"][1][2], runs["eager"][2][2])      # the reload reached the replayed critic


def test_handover_from_the_native_update():
    """sync_rollout_nets_native from a two-layer NativePPO into a tensor-core-eligible CriticLSTM."""
    import copy
    import taco_b200
    from oracle import critic as oc
    from taco_b200.ppo import TorchActorCritic, sync_rollout_nets_native
    from taco_b200.ppo_native import NativePPO
    torch.manual_seed(4)
    agent = TorchActorCritic(26, 4, [64, 64], 26, 64, [256, 256], lstm_layers=2).cuda()
    nat = NativePPO(agent, 256)
    nat._create(5)
    nat.load_from(agent)
    critic = taco_b200.CriticLSTM(26, 5, 64, [256, 256], lstm_layers=2)
    assert critic.tensor_cores_available
    sync_rollout_nets_native(nat, critic=critic)
    states = _states(4096, 5, 26, 11)
    v = critic.forward(states.cuda(), tensor_cores=True).cpu()
    cpu = copy.deepcopy(agent).cpu()
    with torch.no_grad():
        ref = cpu.critic_mlp(cpu.critic_encoder(states))
        lstm = cpu.critic_encoder.layers
        prm = [tuple(getattr(lstm, f"{k}_l{l}") for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")) for l in range(2)]
        lin = [m for m in cpu.critic_mlp.layers if isinstance(m, torch.nn.Linear)]
        emu = oc.critic_forward_bf16(states, prm, [m.weight for m in lin], [m.bias for m in lin])
    assert (v - emu).abs().max().item() <= 1.5e-2
    assert (v - ref).abs().max().item() <= 6e-2
    critic.close(); nat.close()


@pytest.mark.parametrize("hid,mlp_hidden", [(40, [64]), (64, [96, 64])])
def test_stacked_shapes_outside_the_envelope(hid, mlp_hidden):
    from taco_b200 import CriticLSTM
    from oracle import critic as oc
    lstm, w, b = _random_critic(26, hid, mlp_hidden, seed=hid, nl=2)
    c = CriticLSTM(26, 5, hid, mlp_hidden, lstm_layers=2)
    assert not c.tensor_cores_available
    c.load(lstm, w, b)
    states = _states(300, 5, 26, 1)
    with pytest.raises(RuntimeError, match="tensor-core path unavailable"):
        c.forward(states.cuda(), tensor_cores=True)
    torch.testing.assert_close(c.forward(states.cuda()).cpu(), oc.critic_forward(states, lstm, w, b), rtol=0, atol=5e-6)
    c.close()


def test_five_layers_are_rejected():
    from taco_b200 import CriticLSTM
    with pytest.raises(RuntimeError, match="lstm_layers"):
        CriticLSTM(26, 5, 64, [64], lstm_layers=5)
