#!/usr/bin/env python
"""PPO training on the native rollout path -- the loop of the reference's ``train_fpv_asymmetry_ppo.py`` / ``PPO.run``
(IsaacGymEnvs/train/train_fpv_asymmetry_ppo.py:363-538, IsaacGymEnvs/algorithms/ppo_asymmetry.py:260-342) with
  rollout  = GraphedRollout: actor kernel -> critic kernel -> fused env step, zero-copy into the RolloutBuffer, GAE on the device,
             the whole horizon replayed as ONE CUDA graph (--no-graph: the eager collect_rollout loop)
  update   = taco_b200.ppo_native.NativePPO (tcgen05 GEMM forward / backward, device-side KL early stop, Adam and spectral projection
             kernels; loss sums and the flat gradient all-reduced over ranks); --update torch: taco_b200.ppo.ppo_update (PyTorch
             autograd, the fp32 parity path)

    python examples/train_fpv_ppo.py --task pos --num-envs 4096 --epochs 60
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 examples/train_fpv_ppo.py --num-envs 65536

Prints one JSON line per epoch on rank 0 (mean reward per env-step, episode return / length, losses, env-steps/s of the whole loop).
--episode-summary adds, per task, the rollout's finished episodes, survival (time-outs / episodes), mean and std of the return and
the mean length (taco_b200.RolloutEpisodes: one scan of the rollout ring per rollout, all-reduced over ranks).
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--task", default="pos", choices=["pos", "rotate", "flip", "mix"])
    ap.add_argument("--num-envs", type=int, default=4096, help="envs per GPU")
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--epochs", type=int, default=60)
    ap.add_argument("--train-iters", type=int, default=4)
    ap.add_argument("--mini-batch-num", type=int, default=4)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--actor-hidden", default="256,256,256")
    ap.add_argument("--critic-hidden", default="256,256")
    ap.add_argument("--lstm-hidden", type=int, default=64)
    ap.add_argument("--lstm-layers", type=int, default=1, help="stacked LSTM layers of the critic encoder (num_layers of the reference's critic_encoder_dict)")
    ap.add_argument("--lipschitz", type=float, default=4.0, help="README training command: --lipschitz_para=4; 0 disables")
    ap.add_argument("--tensor-cores", default="auto", choices=["auto", "on", "off"])
    ap.add_argument("--update", default="native", choices=["native", "torch"])
    ap.add_argument("--no-graph", action="store_true", help="collect rollouts with the eager loop instead of one CUDA-graph replay per rollout")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--episode-summary", action="store_true", help="log per-task episode counts, survival, return mean / std and mean length")
    ap.add_argument("--save", default=None, help="after training, write the agent's state dict (save_checkpoint(para_only=True)) to this path")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    import taco_b200
    from taco_b200 import dist as tdist
    from taco_b200.ppo import PPOConfig, TorchActorCritic, make_optimizer, ppo_update, save_checkpoint, sync_rollout_nets, sync_rollout_nets_native
    from taco_b200.ppo_native import NativePPO

    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = f"cuda:{local}"
    torch.manual_seed(args.seed)                     # same initial weights on every rank
    n = args.num_envs
    off, n_glob = tdist.shard(rank, world, n)
    env = taco_b200.FpvVecTask(taco_b200.make_cfg(args.task, n, domain_randomization=True), dev, dev, -1, True,
                               env_offset=off, num_envs_global=n_glob, seed=args.seed)
    a_hid = [int(x) for x in args.actor_hidden.split(",")]
    c_hid = [int(x) for x in args.critic_hidden.split(",")]
    agent = TorchActorCritic(26 * env.len_obs, 4, a_hid, 26, args.lstm_hidden, c_hid, lstm_layers=args.lstm_layers).to(dev)
    cfg = PPOConfig(epochs=args.epochs, train_iters=args.train_iters, lr=args.lr, use_lipschitz=args.lipschitz > 0,
                    lipschitz_para=args.lipschitz, lip_epoch_index=[args.epochs // 5, args.epochs],
                    diff_epoch_index=[args.epochs // 5, args.epochs], lr_epoch_index=int(0.7 * args.epochs))
    opt = make_optimizer(agent, cfg)
    native = None
    if args.update == "native":
        native = NativePPO(agent, n * args.horizon // args.mini_batch_num, device=dev)
        native._create(env.len_states)
    actor = taco_b200.ActorMLP(26 * env.len_obs, a_hid, 4, device=dev)
    critic = taco_b200.CriticLSTM(26, env.len_states, args.lstm_hidden, c_hid, lstm_layers=args.lstm_layers, device=dev)
    buf = taco_b200.RolloutBuffer(n, 26, env.len_obs, 26, env.len_states, 4, args.horizon, args.mini_batch_num, 0.99, 0.95, dev)
    # the tensor-core kernels are also the fast path at small env counts (latency of one tile chain: ~12 us actor, ~36 us critic)
    tc = args.tensor_cores != "off" and actor.tensor_cores_available and critic.tensor_cores_available
    env.reset()
    # only the summaries are logged; they count every finished episode, records dropped past the capacity included
    episodes = taco_b200.RolloutEpisodes(env, n) if args.episode_summary else None
    graphed = None
    for epoch in range(args.epochs):
        ts = time.perf_counter()
        if native is not None:
            sync_rollout_nets_native(native, actor, critic)
        else:
            sync_rollout_nets(agent, actor, critic)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if args.no_graph:
            stats = taco_b200.collect_rollout(env, actor, buf, critic, seed=args.seed, tensor_cores=tc, episodes=episodes)
        elif graphed is None:                       # the first rollout runs eagerly inside the constructor, then the loop is one graph
            graphed = taco_b200.GraphedRollout(env, actor, buf, critic, seed=args.seed, tensor_cores=tc, episodes=episodes)
            stats = graphed.first_stats
        else:
            stats = graphed.run()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        n_s = n * args.horizon
        idx = torch.randperm(n_s, device=dev).view(args.mini_batch_num, -1)
        if native is not None:
            out = native.update(buf, cfg, epoch, env=env, batch_idx=list(idx))
        else:
            out = ppo_update(agent, opt, buf, cfg, epoch, env=env, batch_idx=list(idx))
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        if rank == 0:
            s = tdist.summarise(stats)
            line = {"epoch": epoch, "mean_reward": s["mean_reward"], "episode_return": s["mean_episode_return"],
                    "episode_length": s["mean_episode_length"], "difficulty": out["difficulty"], "lipschitz": out["lipschitz_para"],
                    "pg_loss": out["policy_gradient_loss"], "value_loss": out["value_loss"], "kl": out["approx_kl"],
                    "optim_steps": out["optim_steps"], "sync_s": t0 - ts, "rollout_s": t1 - t0, "update_s": t2 - t1,
                    "rollout_env_steps_per_s": world * n_s / (t1 - t0), "loop_env_steps_per_s": world * n_s / (t2 - ts),
                    "tensor_cores": bool(tc), "update": args.update, "early_stop": out["early_stop"], "world": world}
            if episodes is not None:
                line["episodes_by_task"] = {task: {k: e[k] for k in ("episodes", "survival", "ret_mean", "ret_std", "length_mean")}
                                            for task, e in episodes.summary().items()}
            print(json.dumps(line), flush=True)
    if graphed is not None:
        graphed.close()
    if episodes is not None:
        episodes.close()
    if native is not None:
        native.store_to(agent, opt)                 # the torch module / optimiser hold the trained state again (checkpoints, export)
        native.close()
    if args.save and rank == 0:
        save_checkpoint(args.save, agent, para_only=True)         # loads with examples/eval_fpv_policy.py --checkpoint
    env.close(); actor.close(); critic.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
