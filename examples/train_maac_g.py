#!/usr/bin/env python
"""MAAC / MAAC-G / MAAC-R training on the GPU-resident batched environment (BASELINE.json configs[4]).

    python examples/train_maac_g.py --envs 4096 --episodes 5
    python examples/train_maac_g.py --envs 1024 --episodes 5 --method MAAC-R --replay     # PER + PMI training
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 examples/train_maac_g.py --envs 32768
    python examples/train_maac_g.py --envs 4096 --episodes 5 --eval-episodes 4 --greedy     # train, then evaluate
    python examples/train_maac_g.py --envs 65536 --eval-episodes 2 --actor run/actor/actor_weights_4.pth   # evaluate only

Environments are sharded over ranks (no data-path collective); gradients are all-reduced by DDP, episode
statistics by one small all-reduce.  The learner is stock PyTorch (reference architecture and update rule).
"""
import argparse
import os
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config, shard_envs  # noqa: E402
from marl_uavs_targets_tracking_b200 import PMINetwork  # noqa: E402
from marl_uavs_targets_tracking_b200.rollout import (BatchedActorCritic, evaluate_batched, operate_epoch_batched,  # noqa: E402
                                                     train_batched)


def evaluate(cfg, env, agent, pmi, args, rank, world):
    """Per-environment return and average coverage over --eval-episodes episodes: mean, standard deviation and the
    5 / 50 / 95 percentiles over every environment-episode of every rank."""
    t0 = time.perf_counter()
    summaries, per_env = evaluate_batched(cfg, env, agent, pmi, args.eval_episodes, args.steps, greedy=args.greedy)
    for key in ("return", "average_covered_targets"):
        v = per_env[key].reshape(-1)
        if world > 1:  # shards differ by at most one environment: gather as objects
            parts = [None] * world
            dist.all_gather_object(parts, v.cpu())
            v = torch.cat(parts)
        if rank == 0:
            q = torch.quantile(v.double().cpu(), torch.tensor([0.05, 0.5, 0.95], dtype=torch.float64))
            print("evaluate (%s, %d episodes x %d envs): %s mean %.4f std %.4f  p5 %.4f p50 %.4f p95 %.4f" % (
                "greedy" if args.greedy else "sampled", args.eval_episodes, args.envs, key, float(v.mean()),
                float(v.std()) if v.numel() > 1 else 0.0, *q.tolist()))
    if rank == 0:
        print("evaluate: episode returns %s  (%.1f s)" % (" ".join("%.4f" % s["return"] for s in summaries),
                                                         time.perf_counter() - t0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096, help="total environments over all ranks")
    ap.add_argument("--episodes", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--n-uav", type=int, default=10)
    ap.add_argument("--m-targets", type=int, default=10)
    ap.add_argument("--method", default="MAAC-G", choices=["MAAC", "MAAC-G", "MAAC-R"])
    ap.add_argument("--replay", action="store_true",
                    help="reference loop: device prioritized replay + |TD| priorities (+ PMI training for MAAC-R)")
    ap.add_argument("--buffer", type=int, default=1 << 22, help="replay capacity (transitions)")
    ap.add_argument("--minibatch", type=int, default=1 << 20, help="transitions per update")
    ap.add_argument("--eval-episodes", type=int, default=0,
                    help="after training, evaluate the policy over this many episodes of every environment")
    ap.add_argument("--greedy", action="store_true", help="evaluate with the most probable action instead of a draw")
    ap.add_argument("--actor", help="actor checkpoint (BatchedActorCritic.save): evaluate it without training")
    ap.add_argument("--critic", help="critic checkpoint to load with --actor")
    args = ap.parse_args()
    if args.actor:
        for path in (args.actor, args.critic):
            if path and not os.path.exists(path):
                ap.error("checkpoint not found: %s" % path)
        args.episodes = 0
        args.eval_episodes = args.eval_episodes or 1
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    cfg = default_config(args.method, args.n_uav, args.m_targets)
    n_local, offset = shard_envs(args.envs, rank, world)
    env = BatchedEnvironment(args.n_uav, args.m_targets, 2000, 2000, 12, n_envs=n_local, device=device,
                             env_id_offset=offset, seed=cfg["seed"], num_steps=args.steps)
    torch.manual_seed(cfg["seed"])
    agent = BatchedActorCritic(12, 128, 12, 1e-4, 5e-4, 0.95, device, ddp=world > 1)  # src/configs/MAAC-G.yaml:30-36
    if args.actor:
        agent.load(args.actor, args.critic)
    pmi = PMINetwork(hidden_dim=128).to(device) if args.method == "MAAC-R" else None  # src/configs/MAAC-R.yaml:38-41
    if (args.replay or pmi is not None) and args.episodes:
        cfg.setdefault("actor_critic", {}).update(buffer_size=args.buffer, sample_size=min(args.minibatch, args.buffer))
        cfg.setdefault("pmi", {}).setdefault("batch_size", 128)
        t0 = time.perf_counter()

        def report(ep, s):
            if rank == 0:
                print("episode %d  return %.4f  covered avg %.2f  actor %.4f critic %.4f%s  (%.1f s)" % (
                    ep, s["return"], s["average_covered_targets"], s["actor_loss"], s["critic_loss"],
                    "  pmi %.4f" % s["avg_pmi_loss"] if "avg_pmi_loss" in s else "", time.perf_counter() - t0))
        train_batched(cfg, env, agent, pmi, args.episodes, args.steps, on_episode=report)
        args.episodes = 0
    for ep in range(args.episodes):
        t0 = time.perf_counter()
        env.reset(cfg)
        tr, summary = operate_epoch_batched(cfg, env, agent, None, args.steps)
        torch.cuda.synchronize(device)
        t1 = time.perf_counter()
        B = tr["states"].shape[0]
        idx = torch.randint(0, B, (min(args.minibatch, B),), device=device)
        a_loss, c_loss, _ = agent.update(tr["states"][idx], tr["actions"][idx], tr["rewards"][idx], tr["next_states"][idx])
        torch.cuda.synchronize(device)
        if rank == 0:
            print("episode %d  return %.4f  tracking %.4f  covered avg %.2f max %d  rollout %.2f M agent-steps/s  "
                  "actor %.4f critic %.4f" % (ep, summary["return"], summary["target_tracking_return"],
                                               summary["average_covered_targets"], summary["max_covered_targets"],
                                               args.envs * args.n_uav * args.steps / (t1 - t0) / 1e6, float(a_loss), float(c_loss)))
    if args.eval_episodes:
        evaluate(cfg, env, agent, pmi.eval() if pmi is not None else None, args, rank, world)
    env.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
