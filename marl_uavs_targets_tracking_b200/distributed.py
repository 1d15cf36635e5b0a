"""Rank sharding of environments and the episode-statistics reduce (SURVEY.md section 8e).

Environments are independent, so rank r of R owns the contiguous global ids
[r*E/R, (r+1)*E/R) and the data path has no collective.  The only exchange is one all-reduce of
<= 8 doubles per episode (the sums src/train.py:181-192 accumulates): NCCL over NVLink on GPUs,
gloo in the CPU tests.
"""
import os

import torch
import torch.distributed as dist

_SUM_KEYS = ("rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment",
             "covered_sum", "env_steps", "pmi_rows_out_of_range")


def shard_envs(total_envs, rank, world_size):
    """-> (n_local, global id of the first local env); sizes differ by at most one."""
    lo = total_envs * rank // world_size
    hi = total_envs * (rank + 1) // world_size
    return hi - lo, lo


def reduce_episode_stats(stats, device=None, group=None):
    """All-reduce the dict returned by BatchedEnvironment.episode_stats(): SUM for the sums, MAX for
    covered_max.  Returns a new dict; a no-op when torch.distributed is not initialised."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return dict(stats)
    dev = device if device is not None else ("cuda" if dist.get_backend(group) == "nccl" else "cpu")
    keys = [k for k in _SUM_KEYS if k in stats]  # (every rank passes the same keys)
    s = torch.tensor([stats[k] for k in keys], dtype=torch.float64, device=dev)
    mx = torch.tensor([stats["covered_max"]], dtype=torch.float64, device=dev)
    dist.all_reduce(s, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    out = {k: float(v) for k, v in zip(keys, s.tolist())}
    out["covered_max"] = float(mx.item())
    return out


def episode_summary(stats, n_uav):
    """The per-episode scalars src/train.py:187-192 logs, from (reduced) statistics."""
    agent_steps = max(stats["env_steps"] * n_uav, 1.0)
    return {"return": stats["rewards"] / agent_steps,
            "target_tracking_return": stats["target_tracking_reward"] / agent_steps,
            "boundary_punishment_return": stats["boundary_punishment"] / agent_steps,
            "duplicate_tracking_punishment_return": stats["duplicate_tracking_punishment"] / agent_steps,
            "average_covered_targets": stats["covered_sum"] / max(stats["env_steps"], 1.0),
            "max_covered_targets": stats["covered_max"]}


def bind_host_to_gpu(device_index):
    """Pin this process to the CPUs NVML reports as local to the GPU (same NUMA node / PCIe root), so pinned host
    buffers allocated afterwards are first-touched next to the link they are copied over.  With one process per GPU
    and host-buffer steps (`uavsim_step_host`) every rank otherwise stages through whichever node the scheduler
    picked.  Returns (previous affinity, new affinity) or None when NVML / the affinity call is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(device_index).uuid)
        try:
            handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + uuid)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        before = os.sched_getaffinity(0)
        cpus &= before
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return before, cpus
    except Exception:
        return None
