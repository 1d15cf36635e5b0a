#!/usr/bin/env python
"""Learned-policy rollout: ms per step of the per-step loop driven from Python (bind_obs, bind_actions,
fused_policy_sample, step_device and a copy of reward plane 0, i.e. what operate_epoch_batched did per step) against one
uavsim_run_policy call per episode (env.run_policy with obs / action / reward trajectories, then the copy of plane 0
that operate_epoch_batched makes).  Whole 200-step episodes timed with CUDA events, after a warm-up episode of each
path; the two paths alternate in one process, each on its own environment (same seed, so episode k starts from the
same state on both), and every pair of episodes is checked to give identical episode statistics and final state.
Policy: 12 -> 128 -> 12.  Prints the GPU name and power limit with the table.

    python tools/policy_loop_timing.py [--reps R] [--steps T] [--json FILE] [--only NAME]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from marl_uavs_targets_tracking_b200 import BatchedEnvironment, PMINetwork, default_config  # noqa: E402
from marl_uavs_targets_tracking_b200.rollout import PolicyNet, fused_policy_sample  # noqa: E402

# (name, n_uav, m_targets, environments, method)
WORKLOADS = [
    ("10x10-4k-G", 10, 10, 4096, "MAAC-G"),
    ("10x10-16k-G", 10, 10, 16384, "MAAC-G"),
    ("10x10-64k-G", 10, 10, 65536, "MAAC-G"),
    ("10x10-16k-R", 10, 10, 16384, "MAAC-R"),
    ("64x64-16k-G", 64, 64, 16384, "MAAC-G"),
    ("64x64-64k-G", 64, 64, 65536, "MAAC-G"),
]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # the table is still worth having; the missing field says why
        info["power_limit"] = "unknown (%s)" % exc
    return info


def per_step_episode(env, cfg, pmi, net, seed, c0, T, traj, acts, rews):
    E, n = env.n_envs, env.n_uav
    home_obs, home_act = env._obs, env.actions
    traj[0].copy_(home_obs)
    for k in range(T):
        cfg["step"] = k + 1
        env.bind_obs(traj[k + 1])
        env.bind_actions(acts[k])
        fused_policy_sample(net, traj[k].view(E * n, 12), seed, c0 + k, out=acts[k].view(-1))
        _, rew4, _ = env.step_device(cfg, pmi)
        rews[k].copy_(rew4[0].reshape(E * n))
    home_obs.copy_(traj[T])
    env.bind_obs(home_obs)
    env.bind_actions(home_act)


def device_loop_episode(env, cfg, pmi, net, seed, c0, T, traj, acts, rew4, rews):
    env.run_policy(cfg, pmi, net, seed, c0, T, obs=traj, actions=acts, rew4=rew4)
    rews.copy_(rew4[:, 0].reshape(T, -1))


def measure(name, n, m, E, method, T, reps):
    dev = torch.device("cuda:0")
    cfg = default_config(method, n, m)
    pmi = None
    if method == "MAAC-R":
        torch.manual_seed(1)
        pmi = PMINetwork(hidden_dim=128).eval()
    envs = [BatchedEnvironment(n, m, 2000, 2000, 12, n_envs=E, device=dev, seed=5, num_steps=T) for _ in range(2)]
    torch.manual_seed(0)
    net = PolicyNet(12, 128, 12).to(dev)
    traj = torch.empty((T + 1, E, n, 12), dtype=torch.float32, device=dev)
    acts = torch.empty((T, E, n), dtype=torch.int32, device=dev)
    rew4 = torch.empty((T, 4, E, n), dtype=torch.float32, device=dev)
    rews = torch.empty((T, E * n), dtype=torch.float32, device=dev)
    runs = [lambda e, c0: per_step_episode(e, cfg, pmi, net, 9, c0, T, traj, acts, rews),
            lambda e, c0: device_loop_episode(e, cfg, pmi, net, 9, c0, T, traj, acts, rew4, rews)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = [[], []]
    identical = True
    for rep in range(reps + 1):  # rep 0: warm-up
        ends = []
        for p in (0, 1) if rep % 2 == 0 else (1, 0):  # alternate which path goes first
            env = envs[p]
            env.reset(cfg)
            torch.cuda.synchronize()
            ev[0].record()
            runs[p](env, 1 + rep * T)
            ev[1].record()
            torch.cuda.synchronize()
            if rep:
                ms[p].append(ev[0].elapsed_time(ev[1]) / T)
            ends.append((p, env.episode_stats(), {k: v.clone() for k, v in env.get_state().items()}))
        ends.sort(key=lambda x: x[0])
        identical = identical and ends[0][1] == ends[1][1] and all(torch.equal(ends[0][2][k], ends[1][2][k]) for k in ends[0][2])
    for e in envs:
        e.close()
    del traj, acts, rew4, rews
    torch.cuda.empty_cache()
    row = {"workload": name, "n_uav": n, "m_targets": m, "envs": E, "method": method, "steps": T, "reps": reps,
           "identical": identical}
    for key, v in (("per_step", ms[0]), ("run_policy", ms[1])):
        row[key + "_ms"] = statistics.median(v)
        row[key + "_ms_min"], row[key + "_ms_max"] = min(v), max(v)
    row["speedup"] = row["per_step_ms"] / row["run_policy_ms"]
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=6, help="timed episodes per path")
    ap.add_argument("--steps", type=int, default=200, help="episode length")
    ap.add_argument("--json", help="also write the rows and the GPU info to this file")
    ap.add_argument("--only", help="one workload by name")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("policy_loop_timing needs a CUDA device")
    info = gpu_info()
    print("GPU: %s, power limit %s, max SM clock %s" % (info["name"], info.get("power_limit"), info.get("max_sm_clock")))
    rows = []
    print("%-12s %8s %-7s | %-27s | %-27s | %7s %s" % ("workload", "envs", "method", "per-step loop ms/step (range)",
                                                      "run_policy ms/step (range)", "speedup", "identical"))
    for w in WORKLOADS:
        if args.only and w[0] != args.only:
            continue
        r = measure(*w, args.steps, args.reps)
        rows.append(r)
        print("%-12s %8d %-7s | %.4f (%.4f-%.4f)          | %.4f (%.4f-%.4f)          | %6.2fx %s" % (
            r["workload"], r["envs"], r["method"], r["per_step_ms"], r["per_step_ms_min"], r["per_step_ms_max"],
            r["run_policy_ms"], r["run_policy_ms_min"], r["run_policy_ms_max"], r["speedup"], r["identical"]), flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump({"gpu": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
