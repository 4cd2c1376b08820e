#!/usr/bin/env python
"""Test-mode evaluation of a trained policy on the device -- what the reference's ``--train_mode=testmodel``
(train_fpv_asymmetry_ppo.py:328-356) does with its ``Logger`` (CTRL/logger.py), at evaluation scale:

  * the checkpoint (``save_checkpoint`` / ``PPO.save``: a bare state dict, or a training checkpoint) is loaded into
    ``TorchActorCritic`` and its actor into the rollout kernel (``ActorMLP``);
  * the env runs in test mode: maxEpisodeLength = 1000, difficulty 1, domain randomisation switches from the flags;
  * ``evaluate_policy`` drives it with the deterministic policy (the action mean), replayed as CUDA graphs, until ``--episodes``
    whole episodes are recorded by the env's episode log;
  * one JSON line per task summary is printed; ``--record`` envs' trajectories go to ``--out`` (one .npy and .csv per episode).

    python examples/train_fpv_ppo.py --task pos --epochs 60 --save m.pt
    python examples/eval_fpv_policy.py --checkpoint m.pt --task pos --num-envs 65536 --episodes 100000 --record 0 --out traj
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--checkpoint", required=True)
    ap.add_argument("--task", default="pos", choices=["pos", "rotate", "flip", "mix"])
    ap.add_argument("--num-envs", type=int, default=4096)
    ap.add_argument("--episodes", type=int, default=10000, help="whole episodes to record before stopping")
    ap.add_argument("--max-steps", type=int, default=100000)
    ap.add_argument("--record", default="", help="comma-separated env ids whose trajectories are recorded, e.g. 0,1")
    ap.add_argument("--out", default="eval_out", help="directory of the trajectory files")
    ap.add_argument("--tensor-cores", default="auto", choices=["auto", "on", "off"])
    ap.add_argument("--no-dr", action="store_true", help="turn the domain randomisation switches off (make_cfg default set)")
    ap.add_argument("--steps-per-replay", type=int, default=64)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()

    import torch
    import taco_b200
    from taco_b200.ppo import TorchActorCritic, load_checkpoint

    dev = "cuda:0"
    blob = torch.load(args.checkpoint, map_location="cpu", weights_only=True)
    sd = blob["agent"] if "agent" in blob else blob
    lin = sorted({int(k.split(".")[2]) for k in sd if k.startswith("actor_mlp.layers.") and k.endswith(".weight")})
    a_sizes = [sd[f"actor_mlp.layers.{lin[0]}.weight"].shape[1]] + [sd[f"actor_mlp.layers.{j}.weight"].shape[0] for j in lin]
    clin = sorted({int(k.split(".")[2]) for k in sd if k.startswith("critic_mlp.layers.") and k.endswith(".weight")})
    c_hidden = [sd[f"critic_mlp.layers.{j}.weight"].shape[0] for j in clin][:-1]
    lstm_layers = len([k for k in sd if k.startswith("critic_encoder.layers.weight_ih_l")])
    lstm_hidden = sd["critic_encoder.layers.weight_hh_l0"].shape[1]
    agent = TorchActorCritic(a_sizes[0], a_sizes[-1], a_sizes[1:-1], sd["critic_encoder.layers.weight_ih_l0"].shape[1], lstm_hidden,
                             c_hidden, lstm_layers=lstm_layers)
    load_checkpoint(args.checkpoint, agent, map_location="cpu")

    cfg = taco_b200.make_cfg(args.task, args.num_envs, domain_randomization=not args.no_dr, difficulty=1.0, seed=args.seed)
    cfg["env"]["maxEpisodeLength"] = 1000                        # train_fpv_asymmetry_ppo.py:342
    env = taco_b200.FpvVecTask(cfg, dev, dev, -1, True)
    if a_sizes[0] != 26 * env.len_obs:
        raise SystemExit(f"the checkpoint's actor reads {a_sizes[0]} features, the env gives {26 * env.len_obs}")
    actor = taco_b200.ActorMLP(a_sizes[0], a_sizes[1:-1], a_sizes[-1], device=dev)
    actor.load_module(agent.actor_mlp, log_std=agent.log_std, lipschitz_const=-1.0)
    tc = args.tensor_cores != "off" and actor.tensor_cores_available
    if args.tensor_cores == "on" and not tc:
        raise SystemExit("--tensor-cores on: the tcgen05 actor kernel does not support this shape")
    record = [int(x) for x in args.record.split(",") if x.strip()] or None

    t0 = time.perf_counter()
    records, traj, summary = taco_b200.evaluate_policy(env, actor, args.episodes, args.max_steps, tensor_cores=tc, graph=not args.no_graph,
                                                       record_env_ids=record, steps_per_replay=args.steps_per_replay)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    steps = int(records["end_step"].max()) + 1 if len(records) else 0
    for s in summary.values():
        print(json.dumps(dict(s, checkpoint=os.path.basename(args.checkpoint), num_envs=args.num_envs, tensor_cores=bool(tc))), flush=True)
    files = taco_b200.save_trajectories(traj, args.out) if traj is not None else []
    print(json.dumps({"episodes": int(len(records)), "steps": steps, "seconds": dt, "trajectory_files": len(files),
                      "out": os.path.abspath(args.out) if files else None}), flush=True)
    actor.close()
    env.close()


if __name__ == "__main__":
    main()
