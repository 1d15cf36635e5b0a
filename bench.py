#!/usr/bin/env python
"""bench.py -- agent-steps/s of the batched environment step on B200 (one JSON line on rank 0).

    python bench.py --gpus N --steps K --warmup W              # this repo (CUDA)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm: oracle port, all host threads

A "step" is one Environment.step over every environment of the workload (one launch of the fused
kernel).  Default workload = BASELINE.json configs[3], the one the north_star target is quoted on:
64 UAVs x 64 targets, 65 536 environments per GPU, MAAC-G reward (neighbour mean, cooperative 0.3),
random-policy actions resident in HBM.  Environments are independent, so N GPUs run N shards with no
data-path collective ("scaling": "weak": 65 536 environments per GPU); the only exchange is the episode
statistics all-reduce (<= 8 doubles), done once after the timed region.

value     = env x n_uav x K / device time (CUDA events, max over ranks), inputs resident in HBM.
e2e       = same metric through BatchedEnvironment.step_host (the C-ABI call with HOST buffers):
            pinned host actions in, observations / 4 reward planes / covered counts out, every step.
roofline  = algorithmic bytes per launch (SURVEY.md section 8d: 124 n + 48 m + 4 per env-step) / mean launch time
            against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
cpu_baseline = the CPU oracle (C port of the reference loop, oracle/) on a bounded sample, all host threads.
             cpu_baseline.python_reference times the reference's own Python step; it needs the copy of the
             reference that __graft_entry__.build() makes from $UAVSIM_REFERENCE_SRC and is null without it.

--dump-outputs DIR writes what the last timed step returned (observations, reward planes, covered counts; a fixed
sample of environments when the workload is large) as .npy files.  The inputs depend only on the arguments, so two
builds of the project can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n_uav, m_targets, envs per GPU, method, description)
    "swarm64": (64, 64, 65536, "MAAC-G", "configs[3]: 64 UAV x 64 targets, 65536 envs/GPU, MAAC-G reward, random policy"),
    "swarm64_self": (64, 64, 65536, "MAAC", "configs[3] with MAAC (cooperative=0) reward"),
    "default4096": (10, 10, 4096, "MAAC", "configs[1]: default 10x10 scenario, 4096 envs, random policy, step+reward"),
    "default_pmi16384": (10, 10, 16384, "MAAC-R", "configs[2]: default 10x10, 16384 envs, MAAC-R PMI reward (H=128)"),
    "swarm64_pmi": (64, 64, 16384, "MAAC-R", "64x64, 16384 envs, MAAC-R PMI reward (H=128)"),
}
EPISODE = 200  # src/main.py:128 --num_steps default


def alg_bytes_per_env_step(n, m):
    """SURVEY.md section 8d: fp64 x,y,h in+out, int32 last action in+out... = 124 n + 48 m + 4 bytes."""
    return 124 * n + 48 * m + 4


def workload_config(name, E):
    """The `config` object of the JSON line: identical in the native and the reference arm."""
    n, m, _, method, desc = WORKLOADS[name]
    return {"workload": name, "description": desc, "n_uav": n, "m_targets": m, "envs_per_gpu": E, "method": method}


def python_reference_rate(budget_s=6.0):
    """The reference's own Python `Environment.step` (baseline/_ref/src, unmodified) timed on this box: one process, one
    environment -- the way the reference runs (src/environment.py:120) -- for 64x64 and 10x10, MAAC-G reward, random
    actions.  A few steps each (bounded by `budget_s`); None when the copy of the reference is absent."""
    try:
        import random
        import numpy as np
        import torch
        import baseline
        if not baseline.available():
            return None
        ref = baseline.import_reference()
        torch.set_num_threads(1)
        out = {"source": "baseline/_ref/src Environment.step (unmodified reference), 1 process, 1 thread", "cases": {}}
        for n, m in ((64, 64), (10, 10)):
            cfg = baseline.load_yaml_config("MAAC-G")
            cfg["environment"].update(n_uav=n, m_targets=m)
            random.seed(0)
            env = ref.environment.Environment(n_uav=n, m_targets=m, x_max=2000, y_max=2000, na=12)
            env.reset(cfg)
            rng = np.random.RandomState(0)
            acts = [[int(a) for a in rng.randint(0, 12, size=n)] for _ in range(400)]
            env.step(cfg, None, acts[0])
            t0, k = time.perf_counter(), 0
            while k < 399 and time.perf_counter() - t0 < budget_s / 2:
                env.step(cfg, None, acts[k + 1])
                k += 1
            dt = time.perf_counter() - t0
            out["cases"]["%dx%d" % (n, m)] = {"value": n * k / dt, "unit": "agent-steps/s", "steps": k, "seconds": dt}
        return out
    except Exception as exc:  # noqa: BLE001  (a reported baseline must never take the GPU line down)
        return {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}


def link_probe(torch, device, h2d_bytes, d2h_bytes, reps=5):
    """Bare pinned-memory copies of the e2e step's byte counts (no kernels): what the host link gives this process."""
    h_in = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
    h_out = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
    d_in, d_out = torch.empty_like(h_in, device=device), torch.empty_like(h_out, device=device)
    s_in, s_out = torch.cuda.Stream(device), torch.cuda.Stream(device)
    for _ in range(2):
        d_in.copy_(h_in, non_blocking=True)
        h_out.copy_(d_out, non_blocking=True)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(reps):  # both directions at once, like the pipelined step
        with torch.cuda.stream(s_in):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s_out):
            h_out.copy_(d_out, non_blocking=True)
    torch.cuda.synchronize(device)
    dt = (time.perf_counter() - t0) / reps
    return {"ms": dt * 1e3, "gbs": (h2d_bytes + d2h_bytes) / dt / 1e9}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """Summarise the samples that arrived inside [t_begin, t_end] (the timed region); if the region was too short
        for nvidia-smi to report inside it, fall back to every sample since start() (warm-up + timed region)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        window = "timed region"
        rows = [ln for (ts, ln) in self.lines if t_begin is None or (t_begin <= ts <= (t_end or ts) + 0.15)]
        if not rows:
            rows, window = [ln for (_, ln) in self.lines], "warm-up + timed region"
        sm, mx, reasons, pw = [], [], set(), []
        for ln in rows:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "window": window, "reasons": sorted(reasons)}


DUMP_BYTES = 32 << 20  # --dump-outputs: above this, a seeded sample of the environments is written


def dump_outputs(out_dir, obs, rew4, covered):
    """Write one step's outputs as returned by step_device -- obs [E,n,12] and rew4 [4,E,n] float32, covered [E] (as
    float64) -- to out_dir/<name>.npy.  When all E environments exceed DUMP_BYTES, a fixed seeded sample of them is
    written in ascending order; env_index.npy (float64) says which environments the rows are."""
    import numpy as np
    import torch
    E, n = obs.shape[0], obs.shape[1]
    k = min(E, DUMP_BYTES // ((12 + 4) * n * 4 + 2 * 8))
    idx = np.arange(E) if k == E else np.sort(np.random.RandomState(0).choice(E, k, replace=False))
    sel = torch.from_numpy(idx).to(obs.device)
    arrays = {"obs": obs.index_select(0, sel).float(), "rew4": rew4.index_select(1, sel).float(),
              "covered": covered.index_select(0, sel).double(), "env_index": torch.from_numpy(idx).double()}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def make_pmi(torch, hidden=128):
    from marl_uavs_targets_tracking_b200 import PMINetwork
    torch.manual_seed(42)
    pmi = PMINetwork(hidden_dim=hidden)
    for bn in (pmi.bn_comm, pmi.bn_obs, pmi.bn_boundary_state, pmi.bn1):  # SURVEY 8d config 3
        bn.running_mean.normal_(0, 0.3)
        bn.running_var.uniform_(0.5, 1.5)
    return pmi.eval()


def cpu_oracle_rate(n, m, method, budget_s, threads, seed=0):
    """Time the CPU oracle (oracle/, C port of the reference's loops) on a bounded sample of the workload."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from gpu_util import oracle_params_from_config, oracle_pmi_from_module
    from philox_ref import reset_reference
    from marl_uavs_targets_tracking_b200 import default_config
    from oracle import Oracle
    cfg = default_config(method, n, m)
    P = oracle_params_from_config(cfg, n, m)
    mode = {"MAAC": 0, "MAAC-G": 1, "MAAC-R": 2}[method]
    pmi = oracle_pmi_from_module(make_pmi(torch)) if method == "MAAC-R" else None
    orc = Oracle()
    E = max(threads * 16, 32)
    st = reset_reference(seed, E, n, m, 12, 2000, 2000)
    st = {k: np.ascontiguousarray(v) for k, v in st.items()}
    rng = np.random.RandomState(seed)
    acts = rng.randint(0, 12, size=(E, n)).astype(np.int32)
    t0 = time.perf_counter()
    orc.step_batch(P, mode, float(cfg["cooperative"]), pmi, st, acts, nthreads=threads, want_tracker=False)
    one = max(time.perf_counter() - t0, 1e-4)
    steps = int(max(3, min(100000, budget_s / one)))
    t0 = time.perf_counter()
    for _ in range(steps):
        acts = rng.randint(0, 12, size=(E, n)).astype(np.int32)
        orc.step_batch(P, mode, float(cfg["cooperative"]), pmi, st, acts, nthreads=threads, want_tracker=False)
    dt = time.perf_counter() - t0
    return E * n * steps / dt, "%d envs x %d steps of %dx%d %s, %d threads, %.1f s" % (E, steps, n, m, method, threads, dt), E, steps, dt


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (the Python
    reference itself cannot travel to the GPU box), all host threads, same metric / config / unit."""
    if rank != 0:
        return
    n, m, E, method, desc = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from gpu_util import oracle_params_from_config, oracle_pmi_from_module
    from philox_ref import reset_reference
    from marl_uavs_targets_tracking_b200 import default_config
    from oracle import Oracle
    cfg = default_config(method, n, m)
    P = oracle_params_from_config(cfg, n, m)
    mode = {"MAAC": 0, "MAAC-G": 1, "MAAC-R": 2}[method]
    pmi = oracle_pmi_from_module(make_pmi(torch)) if method == "MAAC-R" else None
    orc = Oracle()
    # bounded sample: enough envs to keep every thread busy; one probe step sizes it so that K+W steps take ~1.5 x --cpu-seconds
    # (more environments per call when the steps are short, so thread start-up does not dominate; fewer when long)
    Es = max(threads * 8, 16)
    probe = {k: np.ascontiguousarray(v) for k, v in reset_reference(0, Es, n, m, 12, 2000, 2000).items()}
    rng = np.random.RandomState(0)
    acts = rng.randint(0, 12, size=(Es, n)).astype(np.int32)
    orc.step_batch(P, mode, float(cfg["cooperative"]), pmi, probe, acts, nthreads=threads, want_tracker=False)  # page-in
    t0 = time.perf_counter()
    orc.step_batch(P, mode, float(cfg["cooperative"]), pmi, probe, acts, nthreads=threads, want_tracker=False)
    one = max(time.perf_counter() - t0, 1e-6)
    total = max(args.steps + args.warmup, 1)
    scale = 1.5 * args.cpu_seconds / (one * total)   # default --cpu-seconds 12 -> ~18 s of CPU work
    if scale >= 2:
        Es *= int(min(scale, 256))
    else:
        while Es > threads and one * total > 120:
            Es //= 2
            one /= 2
    Es = min(Es, E)
    st = {k: np.ascontiguousarray(v) for k, v in reset_reference(0, Es, n, m, 12, 2000, 2000).items()}
    # random-policy actions drawn BEFORE the timed loop, one [Es,n] array per step -- exactly what the native arm does
    # with its resident action bank: both arms time the environment step and nothing else
    bank = [rng.randint(0, 12, size=(Es, n)).astype(np.int32) for _ in range(args.warmup + args.steps)]
    for i in range(args.warmup):
        orc.step_batch(P, mode, float(cfg["cooperative"]), pmi, st, bank[i], nthreads=threads, want_tracker=False)
    t0 = time.perf_counter()
    for i in range(args.steps):
        orc.step_batch(P, mode, float(cfg["cooperative"]), pmi, st, bank[args.warmup + i], nthreads=threads, want_tracker=False)
    dt = time.perf_counter() - t0
    value = Es * n * args.steps / dt
    sample = "%d envs (sample of %d x %d GPUs) x %d steps of %dx%d %s" % (Es, E, args.gpus, args.steps, n, m, method)
    out = {"impl": "reference", "metric": "agent-steps/s", "value": value, "unit": "agent-steps/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": workload_config(args.workload, E),
           "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": threads, "kind": "port", "sample": sample},
           "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0,
           "note": "CPU oracle (C restatement of the reference's Python loops, pinned to the reference by tests/golden); "
                   "the Python reference itself is timed by the native arm (cpu_baseline.python_reference)"}
    print(json.dumps(out), flush=True)


def measure_workload(torch, dist, env_cls, args, name, rank, world, device, steps, warmup, with_e2e, e2e_steps):
    from marl_uavs_targets_tracking_b200 import default_config
    n, m, E, method, desc = WORKLOADS[name]
    if args.envs_per_gpu and name == args.workload:
        E = args.envs_per_gpu
    cfg = default_config(method, n, m)
    pmi = make_pmi(torch) if method == "MAAC-R" else None
    sampler = ClockSampler(device.index)
    sampler.start()  # early: nvidia-smi needs a moment to start streaming; only timed-region samples are reported
    env = env_cls(n, m, 2000, 2000, 12, n_envs=E, device=device, env_id_offset=rank * E, seed=42, num_steps=EPISODE)
    sp = getattr(args, "step_path", 0)
    if sp == 1 or (sp in (2, 3) and (n, m) == (64, 64)) or (sp == 4 and max(n, m) <= 16):
        env.set_step_path(sp)  # A/B timing (1: generic; 64 x 64: 2 per-UAV walks, 3 all-pairs tiles; small swarms: 4)
    env.reset(cfg)
    # random-policy actions resident in HBM: one pre-drawn [E,n] tensor per step of an episode (a short bank that
    # repeats would make every UAV fly the same few turns in a loop instead of a random walk), rebound per step
    # (the headline workload keeps a whole episode of them, 3.4 GB at 64 x 64 x 65 536, for the per-episode figure)
    NB = EPISODE if with_e2e else min(EPISODE, steps + warmup)
    bank = torch.empty((NB, E, n), dtype=torch.int32, device=device)
    for b in range(NB):
        env.bind_actions(bank[b])
        env.random_actions(seed=4242, step=b)
    torch.cuda.synchronize(device)

    def one_step(i):
        if i % EPISODE == 0 and i > 0:
            env.reset(cfg)
        env.bind_actions(bank[i % NB])
        return env.step_device(cfg, pmi)

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for i in range(warmup):
        one_step(i)
    barrier()
    l0 = env.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.time()
    ev0.record(torch.cuda.current_stream(device))
    marks = []
    for i in range(steps):
        last = one_step(warmup + i)
        if args.trace_every and (i + 1) % args.trace_every == 0:
            e = torch.cuda.Event(enable_timing=True)
            e.record(torch.cuda.current_stream(device))
            marks.append(e)
    ev1.record(torch.cuda.current_stream(device))
    barrier()
    clocks = sampler.stop(t_begin, time.time())
    if args.dump_outputs and name == args.workload and rank == 0:
        dump_outputs(args.dump_outputs, *last)  # before the legs below overwrite the output buffers
    ms = ev0.elapsed_time(ev1)
    launches = env.launch_count() - l0
    trace = None
    if marks:  # ms per step over consecutive windows of the timed region (diagnostic only)
        pts = [ev0] + marks
        trace = [round(pts[k].elapsed_time(pts[k + 1]) / args.trace_every, 4) for k in range(len(marks))]
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    res = {"name": name, "desc": desc, "n": n, "m": m, "E": E, "method": method, "ms": ms, "steps": steps,
           "launches": launches, "clocks": clocks, "value": E * world * n * steps / (ms * 1e-3), "trace": trace}

    # the same random-policy rollout queued from C (uavsim_run_random_policy: action draw + step per iteration, no
    # interpreter between steps): what a small batch needs, where one step is shorter than a Python-level call
    env.reset(cfg)
    env.run_random_policy(cfg, pmi, 4242, 0, warmup)
    barrier()
    ev0.record(torch.cuda.current_stream(device))
    env.run_random_policy(cfg, pmi, 4242, warmup, steps)
    ev1.record(torch.cuda.current_stream(device))
    barrier()
    ms_loop = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms_loop], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_loop = float(t.item())
    res["device_loop"] = {"value": E * world * n * steps / (ms_loop * 1e-3), "unit": "agent-steps/s",
                          "ms_per_step": ms_loop / steps, "api": "uavsim_run_random_policy (actions drawn on the device)"}

    if with_e2e:
        # ms per step over one whole 200-step episode (the timed window above sits where the driver's --steps /
        # --warmup put it: right after the reset, when the swarm is densest)
        env.reset(cfg)
        NBe = min(EPISODE, NB)
        barrier()
        ev0.record(torch.cuda.current_stream(device))
        for i in range(EPISODE):
            env.bind_actions(bank[i % NBe])
            env.step_device(cfg, pmi)
        ev1.record(torch.cuda.current_stream(device))
        barrier()
        ms_ep = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms_ep], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_ep = float(t.item())
        res["episode"] = {"steps": EPISODE, "ms_per_step": ms_ep / EPISODE, "value": E * world * n * EPISODE / (ms_ep * 1e-3),
                          "unit": "agent-steps/s", "actions": "bank of %d pre-drawn steps" % NBe}
        NH = min(NB, e2e_steps + 2)
        h_act = torch.empty((NH, E, n), dtype=torch.int32).pin_memory()
        h_act.copy_(bank[:NH].cpu())
        h_obs = torch.empty((E, n, 12), dtype=torch.float32).pin_memory()
        h_rew = torch.empty((4, E, n), dtype=torch.float32).pin_memory()
        h_cov = torch.empty((E,), dtype=torch.int32).pin_memory()
        for i in range(2):
            env.step_host(cfg, pmi, h_act[i % NH], h_obs, h_rew, h_cov, chunks=args.chunks)
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            env.step_host(cfg, pmi, h_act[(i + 2) % NH], h_obs, h_rew, h_cov, chunks=args.chunks)
        torch.cuda.synchronize(device)
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        res["e2e"] = {"value": E * world * n * e2e_steps / dt, "unit": "agent-steps/s",
                      "h2d_bytes_per_step": E * n * 4, "d2h_bytes_per_step": E * n * 12 * 4 + 4 * E * n * 4 + E * 4,
                      "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3, "chunks": args.chunks,
                      "api": "BatchedEnvironment.step_host -> uavsim_step_host (pinned host buffers)"}
        res["checksum"] = float(h_rew[0].double().sum())
        # The same steps queued one ahead (uavsim_step_host_async / _wait, two sets of host output buffers): the download
        # of step t overlaps upload + kernels of step t+1.  Only for callers that hold the next actions already (as this
        # random policy does); the closed-loop number above stays the headline.
        try:
            h_obs2, h_rew2, h_cov2 = torch.empty_like(h_obs).pin_memory(), torch.empty_like(h_rew).pin_memory(), torch.empty_like(h_cov).pin_memory()
            outs = ((h_obs, h_rew, h_cov), (h_obs2, h_rew2, h_cov2))
            for i in range(2):  # both buffer sets and the other chunk count once before the clock starts
                env.step_host_wait(env.step_host_async(cfg, pmi, h_act[i % NH], *outs[i & 1], chunks=2))
            barrier()
            t0 = time.perf_counter()
            acc = 0.0
            pch = 2  # measured best for the queued variant (tools/e2e_timing.py): fewer, larger copies; overlap comes from the next step
            tk = env.step_host_async(cfg, pmi, h_act[2 % NH], *outs[0], chunks=pch)
            for i in range(1, e2e_steps):
                tk2 = env.step_host_async(cfg, pmi, h_act[(i + 2) % NH], *outs[i & 1], chunks=pch)
                env.step_host_wait(tk)
                acc += float(outs[(i - 1) & 1][1][0, 0, 0])   # the step's result is read on the host
                tk = tk2
            env.step_host_wait(tk)
            acc += float(outs[(e2e_steps - 1) & 1][1][0, 0, 0])
            torch.cuda.synchronize(device)
            dtp = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dtp], dtype=torch.float64, device=device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dtp = float(t.item())
            res["e2e"]["pipelined"] = {"value": E * world * n * e2e_steps / dtp, "unit": "agent-steps/s", "ms_per_step": dtp / e2e_steps * 1e3, "chunks": pch,
                                       "api": "step_host_async / step_host_wait, next step queued before this one's outputs are read"}
        except Exception as ex:  # noqa: BLE001
            res["e2e"]["pipelined"] = {"error": str(ex)[:200]}
        try:
            lp = link_probe(torch, device, res["e2e"]["h2d_bytes_per_step"], res["e2e"]["d2h_bytes_per_step"])
            if world > 1:
                t = torch.tensor([lp["ms"]], dtype=torch.float64, device=device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                lp["ms"] = float(t.item())
                lp["gbs"] = (res["e2e"]["h2d_bytes_per_step"] + res["e2e"]["d2h_bytes_per_step"]) / (lp["ms"] * 1e-3) / 1e9
            res["e2e"]["link_ms_per_step"] = lp["ms"]
            res["e2e"]["link_gbs"] = lp["gbs"]     # per GPU, all ranks copying at the same time
            res["e2e"]["link_frac"] = lp["ms"] / res["e2e"]["ms_per_step"]  # share of the e2e step the bare copies take
        except Exception as exc:  # noqa: BLE001
            res["e2e"]["link_probe_error"] = str(exc)[:120]
    # the one collective of the path: episode statistics (<= 8 doubles), outside the timed region
    from marl_uavs_targets_tracking_b200 import reduce_episode_stats
    res["episode_stats"] = reduce_episode_stats(env.episode_stats(), device=device)
    env.close()
    return res


def measure_training(torch, dist, env_cls, rank, world, device, steps=25, envs=65536):
    """BASELINE configs[4]: MAAC-G rollout with the GPU-resident environment feeding the torch actor / critic
    (one [E*n,12] actor forward + on-device categorical sample + one step launch per step), then the reference loop's
    replay add / prioritized sample / actor-critic update / priority write-back (src/train.py:232-262)."""
    from marl_uavs_targets_tracking_b200 import PrioritizedReplayBuffer, default_config
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, operate_epoch_batched
    n = m = 10
    cfg = default_config("MAAC-G", n, m)
    env = env_cls(n, m, 2000, 2000, 12, n_envs=envs, device=device, env_id_offset=rank * envs, seed=42, num_steps=steps)
    torch.manual_seed(42)
    agent = BatchedActorCritic(12, 128, 12, 1e-4, 5e-4, 0.95, device, ddp=world > 1)
    buf = PrioritizedReplayBuffer(1 << 24, device=device, seed=42)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    res = {}
    for it in range(3):  # the first passes warm the allocator and cuBLAS up; the last one is reported
        env.reset(cfg)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)
        ev[0].record()
        tr, summary = operate_epoch_batched(cfg, env, agent, None, steps)
        ev[1].record()
        buf.add(tr)
        sample, idx, _ = buf.sample(1 << 20)
        a_loss, c_loss, td = agent.update(sample["states"], sample["actions"], sample["rewards"], sample["next_states"])
        buf.update_priorities(idx, td.abs())
        ev[2].record()
        torch.cuda.synchronize(device)
        t = torch.tensor([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res = {"value": envs * world * n * steps / (float(t[0]) * 1e-3), "unit": "agent-steps/s (rollout incl. policy)",
               "rollout_ms_per_step": float(t[0]) / steps, "learn_ms": float(t[1]), "envs_per_gpu": envs, "n_uav": n,
               "m_targets": m, "method": "MAAC-G", "steps": steps, "update_batch": 1 << 20,
               "replay_launches": buf.launches, "return": summary["return"]}
        del tr, sample
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="swarm64", choices=sorted(WORKLOADS))
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--chunks", type=int, default=8, help="env ranges the host-buffer step is pipelined over")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU time spent on the cpu_baseline sample")
    ap.add_argument("--trace-every", type=int, default=0, help="also report ms/step per window of this many steps")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary workloads and the CPU baseline")
    ap.add_argument("--step-path", type=int, default=0, help="step kernel: 0 default, 1 generic, 2 per-UAV walks (64x64), 3 all-pairs tiles (64x64), 4 small-swarm")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0's environments) "
                    "as DIR/<name>.npy: obs, rew4, covered, env_index")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native step")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    # host buffers of the e2e leg next to this GPU's PCIe root (one process per GPU); undone before the CPU baseline
    from marl_uavs_targets_tracking_b200 import bind_host_to_gpu
    affinity = None if os.environ.get("UAVSIM_NO_BIND") else bind_host_to_gpu(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)

    main_res = measure_workload(torch, dist, BatchedEnvironment, args, args.workload, rank, world, device, args.steps,
                                args.warmup, True, args.e2e_steps)
    extras = {}
    if not args.no_extras:
        # secondary workloads never take the headline line down with them: a failure is recorded, not raised
        # (every rank runs the same code, so an exception is raised on all ranks or none)
        for name in ("swarm64_self", "default4096", "default_pmi16384", "swarm64_pmi"):
            if name == args.workload:
                continue
            try:
                r = measure_workload(torch, dist, BatchedEnvironment, args, name, rank, world, device,
                                     min(args.steps, 100), 5, False, 0)
                extras[name] = {"value": r["value"], "unit": "agent-steps/s", "ms_per_step": r["ms"] / r["steps"],
                                "envs_per_gpu": r["E"], "n_uav": r["n"], "m_targets": r["m"], "method": r["method"],
                                "device_loop": r["device_loop"],
                                "roofline_frac": r["value"] / world * alg_bytes_per_env_step(r["n"], r["m"]) / r["n"] / (hbm_peak()[0] * 1e9),
                                # small batches: the Python loop above is bound by the interpreter (~19 us per call), the
                                # rollout loop below the FFI is what the kernels deliver
                                "roofline_frac_device_loop": r["device_loop"]["value"] / world * alg_bytes_per_env_step(r["n"], r["m"]) / r["n"] / (hbm_peak()[0] * 1e9)}
            except Exception as exc:  # noqa: BLE001
                extras[name] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
        try:
            extras["train_maac_g"] = measure_training(torch, dist, BatchedEnvironment, rank, world, device)
        except Exception as exc:  # noqa: BLE001
            extras["train_maac_g"] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}

    if rank == 0:
        n, m, E = main_res["n"], main_res["m"], main_res["E"]
        peak, peak_src = hbm_peak()
        bytes_per_launch = E * alg_bytes_per_env_step(n, m)
        # launches in the timed region = `steps` step kernels (+ a reset pair per episode boundary)
        ms_per_step = main_res["ms"] / main_res["steps"]
        achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get(args.workload)
            except Exception:
                traffic = None
        out = {"metric": "agent-steps/s", "value": main_res["value"], "unit": "agent-steps/s", "n_gpus": world,
               "steps": main_res["steps"], "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": workload_config(args.workload, E),
               "timing": {"episode_len": EPISODE, "window": "steps %d..%d after a reset" % (args.warmup, args.warmup + main_res["steps"] - 1),
                          "l2": "per-step working set %.0f MB > 126 MB L2 (inputs larger than L2, no flush needed)" % (bytes_per_launch / 1e6)},
               "clocks": main_res["clocks"], "e2e": main_res["e2e"], "gpu_launches": main_res["launches"],
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "traffic": traffic,
                            "traffic_source": "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full "
                                              "capture of this kernel (committed with the round; not measured by this run)",
                            "peak_source": peak_src, "kernel": "uavsim_step_fast_kernel<64,64>" if (n, m) == (64, 64) else "uavsim_step_kernel",
                            "bytes_per_launch": bytes_per_launch,
                            "bytes_per_agent_step": alg_bytes_per_env_step(n, m) / n},
               "device_loop": main_res["device_loop"], "episode": main_res.get("episode"),
               "episode_stats": main_res["episode_stats"], "other_workloads": extras}
        if main_res.get("trace"):
            out["ms_per_step_trace"] = {"every": args.trace_every, "ms": main_res["trace"]}
        if affinity:
            os.sched_setaffinity(0, affinity[0])
        out["host_affinity"] = None if not affinity else {"cpus": len(affinity[1]), "of": len(affinity[0])}
        if not args.no_extras:  # rank 0 at every N (the other ranks wait at the closing barrier)
            try:
                v, sample, _, _, _ = cpu_oracle_rate(n, m, main_res["method"], args.cpu_seconds, os.cpu_count() or 1)
                out["cpu_baseline"] = {"value": v, "unit": "agent-steps/s", "cores": os.cpu_count() or 1, "kind": "port",
                                       "sample": sample}
            except Exception as exc:  # noqa: BLE001  (the oracle is test infrastructure: never lose the GPU line to it)
                out["cpu_baseline"] = {"value": None, "unit": "agent-steps/s", "cores": os.cpu_count() or 1, "kind": "port",
                                       "sample": "failed: %s" % str(exc)[:200]}
            out["cpu_baseline"]["python_reference"] = python_reference_rate()
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
