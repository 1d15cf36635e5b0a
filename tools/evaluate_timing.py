#!/usr/bin/env python
"""Policy evaluation: ms per step of one uavsim_evaluate_policy episode (sampled and greedy: reset, policy + step +
per-environment accumulation per step, the row output) against reset + one uavsim_run_policy call without a trajectory
(the same episode with the episode statistics only).  Whole 200-step episodes timed with CUDA events, the reset
included on both sides, after a warm-up episode of each path; the three paths alternate in one process, each on its own
environment.  The sampled evaluation and run_policy draw the same actions (same seeds and counters), so each pair of
their episodes is checked to end in the same state with the same episode statistics.  Policy: 12 -> 128 -> 12.  Prints
the GPU name and power limit with the table.

    python tools/evaluate_timing.py [--reps R] [--steps T] [--json FILE] [--only NAME]"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from marl_uavs_targets_tracking_b200 import BatchedEnvironment, PMINetwork, default_config  # noqa: E402
from marl_uavs_targets_tracking_b200.rollout import PolicyNet  # noqa: E402

from policy_loop_timing import gpu_info  # noqa: E402

# (name, n_uav, m_targets, environments, method)
WORKLOADS = [
    ("10x10-4k-G", 10, 10, 4096, "MAAC-G"),
    ("10x10-64k-G", 10, 10, 65536, "MAAC-G"),
    ("10x10-16k-R", 10, 10, 16384, "MAAC-R"),
    ("64x64-16k-G", 64, 64, 16384, "MAAC-G"),
    ("64x64-64k-G", 64, 64, 65536, "MAAC-G"),
]
PATHS = ("run_policy", "evaluate", "evaluate_greedy")


def measure(name, n, m, E, method, T, reps):
    dev = torch.device("cuda:0")
    cfg = default_config(method, n, m)
    pmi = None
    if method == "MAAC-R":
        torch.manual_seed(1)
        pmi = PMINetwork(hidden_dim=128).eval()
    envs = [BatchedEnvironment(n, m, 2000, 2000, 12, n_envs=E, device=dev, seed=5, num_steps=T) for _ in PATHS]
    torch.manual_seed(0)
    net = PolicyNet(12, 128, 12).to(dev)

    def run(p, c0):
        env = envs[p]
        if p == 0:
            env.reset(cfg)
            env.run_policy(cfg, pmi, net, 9, c0, T)
        else:
            env.evaluate_policy(cfg, pmi, net, 1, T, greedy=p == 2, first_counter=c0, policy_seed=9)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = [[] for _ in PATHS]
    identical = True
    for rep in range(reps + 1):  # rep 0: warm-up
        order = list(range(len(PATHS)))
        order = order[rep % len(order):] + order[:rep % len(order)]  # rotate which path goes first
        ends = {}
        for p in order:
            torch.cuda.synchronize()
            ev[0].record()
            run(p, 1 + rep * T)
            ev[1].record()
            torch.cuda.synchronize()
            if rep:
                ms[p].append(ev[0].elapsed_time(ev[1]) / T)
            if p < 2:
                ends[p] = (envs[p].episode_stats(), {k: v.clone() for k, v in envs[p].get_state().items()})
        identical = identical and ends[0][0] == ends[1][0] and all(torch.equal(ends[0][1][k], ends[1][1][k])
                                                                    for k in ends[0][1])
    for e in envs:
        e.close()
    torch.cuda.empty_cache()
    row = {"workload": name, "n_uav": n, "m_targets": m, "envs": E, "method": method, "steps": T, "reps": reps,
           "identical": identical}
    for key, v in zip(PATHS, ms):
        row[key + "_ms"] = statistics.median(v)
        row[key + "_ms_min"], row[key + "_ms_max"] = min(v), max(v)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=6, help="timed episodes per path")
    ap.add_argument("--steps", type=int, default=200, help="episode length")
    ap.add_argument("--json", help="also write the rows and the GPU info to this file")
    ap.add_argument("--only", help="one workload by name")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("evaluate_timing needs a CUDA device")
    info = gpu_info()
    print("GPU: %s, power limit %s, max SM clock %s" % (info["name"], info.get("power_limit"), info.get("max_sm_clock")))
    print("%-12s %6s %-7s | %-25s | %-25s | %-25s | %s" % ("workload", "envs", "method", "run_policy ms/step (range)",
                                                           "evaluate ms/step (range)", "greedy ms/step (range)",
                                                           "identical"))
    rows = []
    for w in WORKLOADS:
        if args.only and w[0] != args.only:
            continue
        r = measure(*w, args.steps, args.reps)
        rows.append(r)
        print("%-12s %6d %-7s | %s | %s" % (r["workload"], r["envs"], r["method"], " | ".join(
            "%.4f (%.4f-%.4f)%s" % (r[p + "_ms"], r[p + "_ms_min"], r[p + "_ms_max"], " " * 4) for p in PATHS),
            r["identical"]), flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump({"gpu": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
