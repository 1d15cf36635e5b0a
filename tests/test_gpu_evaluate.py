"""Policy evaluation: uavsim_evaluate_policy / BatchedEnvironment.evaluate_policy / rollout.evaluate_batched, and the greedy
form of the fused policy kernel (uavsim_policy_greedy / fused_policy_greedy).

The evaluation call must equal the loop it replaces (reset + run_policy per episode, or reset + fused_policy_greedy +
step_device per step) bit for bit, and its per-environment rows must be the fixed-point sums of the reward planes that loop
records: counts of 2^-22 of (v + 3.0f) as int32 minus 0x40400000, summed as int64, and the covered count summed and
maximised.  Summed over environments they are the episode statistics exactly."""
import ctypes as C
import os
import re

import pytest
import torch

from conftest import ROOT

from marl_uavs_targets_tracking_b200 import _cabi

from test_gpu_policy_kernel import BAD_SIZES, _weights, make_inputs, make_net, reference
from test_gpu_policy_loop import alloc_traj, assert_same_env, make_env, make_pmi, make_policy, snapshot

DEV = "cuda:0"


# ------------------------------------------------------------------------------------------------ CPU checks
_CTYPES = {"int": C.c_int, "int64_t": C.c_int64, "uint64_t": C.c_uint64, "double": C.c_double}


def _header_argtypes(name):
    """The ctypes argument list a declaration of include/uavsim.h maps to: pointers to the library's structs and to
    uint64_t as typed pointers, every other pointer as c_void_p, the handle as c_void_p."""
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "uavsim.h")).read(), flags=re.S)
    m = re.search(r"\b%s\s*\(([^)]*)\)" % name, hdr)
    assert m, name
    out = []
    for arg in m.group(1).split(","):
        t = re.sub(r"\bconst\b", "", arg).strip()
        t = t[:t.rfind("*") + 1] if "*" in t else t.rsplit(None, 1)[0]
        t = " ".join(t.replace("*", " *").split())
        if t == "UavSimPolicyWeights *":
            out.append(C.POINTER(_cabi.UavSimPolicyWeights))
        elif t == "uint64_t *":
            out.append(C.POINTER(C.c_uint64))
        elif t.endswith("*"):
            out.append(C.c_void_p)
        else:
            out.append(_CTYPES[t])
    return out


@pytest.mark.parametrize("name", ["uavsim_policy_greedy", "uavsim_evaluate_policy"])
def test_argtypes_match_the_header(name):
    res, args = _cabi.SYMBOLS[name]
    assert res is C.c_int
    assert args == _header_argtypes(name)
    lib = _cabi.load()
    assert list(getattr(lib, name).argtypes) == args


def _greedy(lib, obs, rows, w):
    return lib.uavsim_policy_greedy(C.c_void_p(obs), rows, C.byref(w) if w is not None else None, C.c_void_p(0x5000),
                                    None, 0, None)


def test_policy_greedy_refuses_unsupported_weights():
    """With rows = 0 these are refused before anything else could happen, so the call is safe with or without a device."""
    lib = _cabi.load()
    for kw in BAD_SIZES:
        assert _greedy(lib, 0x100, 0, _weights(**kw)) == -3, kw
    assert _greedy(lib, 0x100, 0, _weights(null=True)) == -1
    assert _greedy(lib, 0x100, 0, None) == -1
    assert b"uavsim_policy_greedy" in lib.uavsim_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="fake pointers: must never reach a launch")
def test_policy_greedy_argument_checks_come_before_the_device():
    lib = _cabi.load()
    for kw in BAD_SIZES:
        assert _greedy(lib, 0x100, 8, _weights(**kw)) == -3, kw
    assert _greedy(lib, 0x100, 8, _weights(null=True)) == -1
    assert _greedy(lib, 0, 8, _weights()) == -1                   # NULL obs
    assert _greedy(lib, 0x100, 0, _weights()) == 0                # nothing to do
    for off in (4, 8, 12):
        assert _greedy(lib, 0x100 + off, 8, _weights()) == -1, off
        assert b"aligned" in lib.uavsim_last_error()
    assert _greedy(lib, 0x100, 8, _weights()) > 0                 # valid arguments: the missing device is reported


def test_evaluate_policy_refuses_a_null_handle():
    lib = _cabi.load()
    assert lib.uavsim_evaluate_policy(None, 1, 0.3, C.byref(_weights()), 0, 1, 1, None, 0, 0, None, None) == -1
    assert b"NULL handle" in lib.uavsim_last_error()


# ------------------------------------------------------------------------------------------------ GPU helpers
def fx_rows(rew4, covered):
    """Per-environment rows of one episode from its recorded planes [T,4,E,n] f32 and covered counts [T,E] i32, with the
    library's fixed-point rule, exact: float64 [E,6]."""
    T, _, E, _ = rew4.shape
    acc = torch.zeros((E, 6), dtype=torch.int64, device=rew4.device)
    if T:
        fx = ((rew4 + 3.0).view(torch.int32) - 0x40400000).to(torch.int64)
        acc[:, :4] = fx.sum(dim=(0, 3)).T
        acc[:, 4] = covered.to(torch.int64).sum(0)
        acc[:, 5] = covered.to(torch.int64).amax(0)
    return acc.double() * torch.tensor([2.0 ** -22] * 4 + [1.0, 1.0], dtype=torch.float64, device=rew4.device)


def check_identity(rows, stats):
    """The sums over environments of an episode's rows are its episode statistics, bit for bit; the maximum is covered_max."""
    s = rows[:, :5].sum(0).tolist()
    want = [stats[k] for k in ("rewards", "target_tracking_reward", "boundary_punishment",
                               "duplicate_tracking_punishment", "covered_sum")]
    assert s == want, (s, want)
    assert (float(rows[:, 5].max()) if rows.shape[0] else 0.0) == stats["covered_max"]


def sampled_reference(ref, cfg, pmi, net, pseed, c0, K, T):
    """reset + run_policy per episode with rew4 / covered recorded: rows [K,E,6] and the episode statistics per episode."""
    rows, stats = [], []
    for k in range(K):
        ref.reset(cfg)
        tr = alloc_traj(ref, T, ("rew4", "covered"))
        ref.run_policy(cfg, pmi, net, pseed, c0 + k * T, T, **tr)
        rows.append(fx_rows(tr["rew4"], tr["covered"]))
        stats.append(ref.episode_stats())
    return rows, stats


def greedy_reference(ref, cfg, pmi, net, K, T):
    """reset + (fused_policy_greedy, step_device) per step, the Python loop the greedy evaluation replaces."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_greedy
    rows, stats = [], []
    E, n = ref.n_envs, ref.n_uav
    for k in range(K):
        ref.reset(cfg)
        rew4 = torch.empty((T, 4, E, n), dtype=torch.float32, device=DEV)
        cov = torch.empty((T, E), dtype=torch.int32, device=DEV)
        for t in range(T):
            fused_policy_greedy(net, ref.get_states().view(-1, 12), out=ref.actions.view(-1))
            ref.step_device(cfg, pmi)
            rew4[t].copy_(ref._rew4)
            cov[t].copy_(ref._covered)
        rows.append(fx_rows(rew4, cov))
        stats.append(ref.episode_stats())
    return rows, stats


def run_eval(n, m, E, method, K, T, greedy=False, step_path=0, pmi=None, pmi_path=0, num_steps=0, hidden=64,
             expect_kernels=()):
    """The reference loop on one environment, evaluate_policy on a twin; asserts everything equal.  Returns both."""
    ref, cfg = make_env(n, m, E, method, num_steps, step_path, pmi_path)
    env, _ = make_env(n, m, E, method, num_steps, step_path, pmi_path)
    net = make_policy(hidden)
    pseed, c0 = 11, 5
    l_ref0 = ref.launch_count()
    if greedy:
        rows_ref, stats_ref = greedy_reference(ref, cfg, pmi, net, K, T)
    else:
        rows_ref, stats_ref = sampled_reference(ref, cfg, pmi, net, pseed, c0, K, T)
    # the reference's launches without its K episode_stats reductions; the handle does not count fused_policy_greedy
    ref_launches = ref.launch_count() - l_ref0 - K + (K * T if greedy else 0)
    l_env0 = env.launch_count()
    call = lambda: env.evaluate_policy(cfg, pmi, net, K, T, greedy=greedy, first_counter=c0, policy_seed=pseed)  # noqa
    if expect_kernels:
        from test_gpu_policy_loop import cuda_kernels
        box = []
        names = cuda_kernels(lambda: box.append(call()))
        for k in expect_kernels:
            assert k in names, (k, names)
        rows = box[0]
    else:
        rows = call()
    # the loop's launches, plus one accumulation per step and one row output per episode
    assert env.launch_count() - l_env0 == ref_launches + K * (T + 1)
    assert rows.shape == (K, E, 6) and rows.dtype == torch.float64
    for k in range(K):
        assert torch.equal(rows[k], rows_ref[k]), k
        check_identity(rows[k], stats_ref[k])
    assert env._episode == ref._episode
    if K:
        assert_same_env(ref, env)
        check_identity(rows[-1], env.episode_stats())
    return ref, env, cfg, net, rows


# ------------------------------------------------------------------------------------------------ 1 + 2: sampled evaluation
@pytest.mark.gpu
@pytest.mark.parametrize("n,m,E,step_path,kernel", [
    (10, 10, 301, 0, "uavsim_step_small_kernel"),
    (10, 10, 301, 1, "uavsim_step_kernel<"),
    (10, 10, 32768, 0, "uavsim_step_kernel<"),        # beyond ~2.5 waves of small-kernel CTAs: the automatic choice
    (64, 64, 96, 0, "uavsim_step_fast_kernel"),
    (64, 64, 96, 3, "uavsim_step_tile_kernel"),
    (7, 5, 9, 1, "uavsim_step_kernel<"),
    (7, 5, 9, 0, "uavsim_step_small_kernel"),
], ids=["small-10x10", "generic-10x10", "generic-auto-10x10", "fast-64x64", "tile-64x64", "generic-7x5", "small-7x5"])
def test_every_step_kernel(n, m, E, step_path, kernel):
    T = 25 if E <= 1024 else 6
    ref, env, _, _, _ = run_eval(n, m, E, "MAAC-G", 3, T, step_path=step_path, num_steps=T - 3,
                                 expect_kernels=(kernel, "uavsim_policy_kernel<12, true>",
                                                 "uavsim_env_stats_kernel", "uavsim_env_stats_finish_kernel"))
    assert int(env.done.min()) == 1
    ref.close()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("method,pmi_hidden,kernel", [
    ("MAAC", 0, None), ("MAAC-G", 0, None),
    ("MAAC-R", 128, "uavsim_pmi_tc_kernel"),
    ("MAAC-R", 32, "uavsim_pmi_kernel<"),
], ids=["MAAC", "MAAC-G", "MAAC-R-tensor-h128", "MAAC-R-cudacore-h32"])
def test_every_reward_mode(method, pmi_hidden, kernel):
    pmi = make_pmi(pmi_hidden) if pmi_hidden else None
    ref, env, _, _, _ = run_eval(10, 10, 301, method, 3, 25, pmi=pmi, hidden=128,
                                 expect_kernels=(kernel,) if kernel else ())
    ref.close()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 1, 3])
@pytest.mark.parametrize("T", [0, 1, 25])
def test_episode_and_step_counts(K, T):
    ref, env, _, _, _ = run_eval(10, 10, 37, "MAAC-G", K, T, num_steps=20)
    ref.close()
    env.close()


@pytest.mark.gpu
def test_no_episode_queues_nothing():
    env, cfg = make_env(10, 10, 37, "MAAC-G")
    before, launches = snapshot(env), env.launch_count()
    rows = env.evaluate_policy(cfg, None, make_policy(), 0, 25)
    assert rows.shape == (0, 37, 6) and env.launch_count() == launches
    for k, v in snapshot(env).items():
        assert torch.equal(v, before[k]), k
    env.close()


# ------------------------------------------------------------------------------------------------ 3: the greedy kernel
GREEDY_CASES = [(A, (1, 128, 385, 512)[i % 4], (1, 3, 513, 4099, 100_003)[i % 5]) for i, A in enumerate(range(2, 17))]


@pytest.mark.gpu
@pytest.mark.parametrize("A,H,rows", GREEDY_CASES, ids=["A%d-H%d-rows%d" % c for c in GREEDY_CASES])
def test_greedy_kernel_is_the_argmax_of_its_probabilities(A, H, rows):
    """actions == torch.argmax(probs) exactly; the chosen action's fp64 probability is within the rounding bound of the
    fp64 maximum; the probability output equals the sampling kernel's and does not change the actions."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_greedy, fused_policy_sample
    net = make_net(H, A, "fc2x8" if A % 2 else "fresh", seed=17 * H + A)
    x = make_inputs("obs" if A % 3 else "randn", rows, seed=H + A)
    act, probs = fused_policy_greedy(net, x, want_probs=True)
    assert act.dtype == torch.int32 and act.shape == (rows,)
    assert torch.equal(act.long(), probs.argmax(1))
    assert torch.equal(act, fused_policy_greedy(net, x)[0])
    assert torch.equal(probs, fused_policy_sample(net, x, 99, 5, want_probs=True)[1])
    p64, bound = reference(net, x)
    a = act.long()[:, None]
    best = p64.argmax(1, keepdim=True)
    gap = p64.gather(1, best) - p64.gather(1, a)
    assert bool((gap <= bound.gather(1, a) + bound.gather(1, best)).all())


@pytest.mark.gpu
@pytest.mark.parametrize("A", [2, 5, 12, 16])
def test_greedy_ties_take_the_first_index(A):
    """Identical fc2 rows give identical logits: the first of them wins.  All rows equal: action 0."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_greedy
    net = make_net(128, A, seed=A)
    x = make_inputs("obs", 4099, seed=A)
    with torch.no_grad():
        hot = [A - 1, A // 2, 0] if A > 2 else [1, 0]
        for j in hot[1:]:
            net.fc2.weight[j] = net.fc2.weight[hot[0]]
            net.fc2.bias[j] = net.fc2.bias[hot[0]]
        net.fc2.bias[hot] += 50.0      # the tied actions dominate every row
    act, probs = fused_policy_greedy(net, x, want_probs=True)
    assert bool((probs[:, hot] == probs[:, hot[:1]]).all())
    assert bool((act == min(hot)).all())
    assert torch.equal(act.long(), probs.argmax(1))
    with torch.no_grad():
        net.fc2.weight.zero_()
        net.fc2.bias.zero_()
    act, probs = fused_policy_greedy(net, x, want_probs=True)
    assert bool((act == 0).all()) and torch.equal(act.long(), probs.argmax(1))


# ------------------------------------------------------------------------------------------------ 4: greedy evaluation
@pytest.mark.gpu
@pytest.mark.parametrize("n,m,E,step_path,method", [
    (10, 10, 301, 0, "MAAC-G"), (10, 10, 301, 1, "MAAC-R"), (64, 64, 96, 0, "MAAC-G"), (7, 5, 9, 0, "MAAC"),
], ids=["small-10x10", "generic-10x10-MAAC-R", "fast-64x64", "small-7x5-MAAC"])
def test_greedy_evaluation_equals_the_python_loop(n, m, E, step_path, method):
    pmi = make_pmi(128) if method == "MAAC-R" else None
    ref, env, _, _, _ = run_eval(n, m, E, method, 2, 25, greedy=True, step_path=step_path, pmi=pmi,
                                 expect_kernels=("uavsim_policy_greedy_kernel<12, true>",))
    ref.close()
    env.close()


# ------------------------------------------------------------------------------------------------ 5: sharding
@pytest.mark.gpu
def test_greedy_rows_do_not_depend_on_sharding():
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    E, K, T = 64, 2, 25
    cfg = default_config("MAAC-G", 10, 10)
    net = make_policy(128)
    parts = []
    for count, offset in ((E, 0), (E // 2, 0), (E // 2, E // 2)):
        env = BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=count, device=DEV, env_id_offset=offset, seed=9)
        parts.append(env.evaluate_policy(cfg, None, net, K, T, greedy=True))
        env.close()
    assert torch.equal(parts[0], torch.cat(parts[1:], dim=1))


# ------------------------------------------------------------------------------------------------ 6: evaluate_batched
@pytest.mark.gpu
@pytest.mark.parametrize("greedy", [False, True], ids=["sampled", "greedy"])
def test_evaluate_batched_fused_is_one_call(greedy):
    """The fused agent: one evaluate_policy call with the agent's seed and counters; summaries are episode_summary of the
    episode statistics (the last one checked against the environment's own), per-environment tensors are the rows
    normalised as episode_summary normalises."""
    from marl_uavs_targets_tracking_b200.distributed import episode_summary
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, evaluate_batched
    E, K, T = 301, 3, 25
    env, cfg = make_env(10, 10, E, "MAAC-G", num_steps=T)
    twin, _ = make_env(10, 10, E, "MAAC-G", num_steps=T)
    torch.manual_seed(0)
    agent = BatchedActorCritic(12, 128, 12, 1e-3, 1e-3, 0.95, torch.device(DEV), seed=7)
    agent._calls = 40
    summaries, per_env = evaluate_batched(cfg, env, agent, None, K, T, greedy=greedy)
    assert agent._calls == 40 + (0 if greedy else K * T) and cfg["step"] == T
    rows = twin.evaluate_policy(cfg, None, agent.actor, K, T, greedy=greedy, first_counter=41, policy_seed=agent.seed)
    assert len(summaries) == K and set(per_env) == set(summaries[0])
    assert summaries[-1] == episode_summary(env.episode_stats(), 10)
    for q, key in enumerate(("return", "target_tracking_return", "boundary_punishment_return",
                             "duplicate_tracking_punishment_return", "average_covered_targets", "max_covered_targets")):
        assert per_env[key].shape == (K, E)
        d = (T * 10, T * 10, T * 10, T * 10, T, 1)[q]
        # (tensor / tensor: an IEEE division like episode_summary's; torch divides by a Python scalar via its reciprocal)
        assert torch.equal(per_env[key], rows[:, :, q] / torch.full_like(rows[:, :, q], d)), key
    env.close()
    twin.close()


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["MAAC-G", "MAAC-R"])
def test_stock_greedy_path_matches_the_fused_one(method):
    """Stock agent (torch forward, argmax, per-environment sums in torch) and fused agent with the same weights give the
    same per-environment rows.  An environment may differ only where some step had a row whose two largest fp64
    probabilities are within the rounding bound (the two forwards round differently); those environments are found from
    the fused run's own observations."""
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, evaluate_batched, fused_policy_greedy
    E, K, T, n = 128, 2, 25, 10
    pmi = make_pmi(128) if method == "MAAC-R" else None
    out, agents = [], []
    for fused in (False, True):
        env, cfg = make_env(n, n, E, method, num_steps=T)
        torch.manual_seed(0)
        agent = BatchedActorCritic(12, 128, 12, 1e-3, 1e-3, 0.95, torch.device(DEV), seed=7, fused=fused)
        assert agent.fused is fused
        out.append(evaluate_batched(cfg, env, agent, pmi, K, T, greedy=True))
        agents.append(agent)
        env.close()
    assert agents[0]._calls == agents[1]._calls == 0
    (s0, p0), (s1, p1) = out
    # near ties along the fused trajectories
    env, cfg = make_env(n, n, E, method, num_steps=T)
    net = agents[1].actor
    near = torch.zeros((K, E), dtype=torch.bool, device=DEV)
    for k in range(K):
        env.reset(cfg)
        for t in range(T):
            x = env.get_states().view(-1, 12)
            p64, bound = reference(net, x)
            top = p64.topk(2, dim=1)
            bnd = 2 * bound.gather(1, top.indices).sum(1)  # (twice: torch's forward rounds in its own order)
            near[k] |= ((top.values[:, 0] - top.values[:, 1]) <= bnd).view(E, n).any(1)
            fused_policy_greedy(net, x, out=env.actions.view(-1))
            env.step_device(cfg, pmi)
    env.close()
    for key in p0:
        same = (p0[key] == p1[key]) | near
        assert bool(same.all()), (key, int((~same).sum()))
    print("%s: %d of %d environment-episodes had a near tie" % (method, int(near.sum()), K * E))
    if not bool(near.any()):
        assert s0 == s1


# ------------------------------------------------------------------------------------------------ 7: errors
def _raw_call(env, w, K=2, T=4, greedy=0, seeds="ok", out="ok", mode=1, coop=0.3):
    seeds_arr = (C.c_uint64 * 2)(1, 2) if seeds == "ok" else None
    buf = torch.zeros(2 * env.n_envs * 6 + 1, dtype=torch.float64, device=DEV)
    ptr = {"ok": buf.data_ptr(), "null": None, "misaligned": buf.data_ptr() + 4}[out]
    rc = env._lib.uavsim_evaluate_policy(env._h, mode, coop, C.byref(w), greedy, 1, 1, seeds_arr, K, T,
                                         C.c_void_p(ptr) if ptr else None,
                                         C.c_void_p(torch.cuda.current_stream().cuda_stream))
    return rc, buf


@pytest.mark.gpu
@pytest.mark.parametrize("case,code", [
    ("episodes<0", -1), ("nsteps<0", -1), ("null-seeds", -1), ("null-out", -1), ("misaligned-out", -1),
    ("greedy=2", -1), ("bad-mode", -1), ("null-weights", -1), ("hidden0", -3), ("n_actions", -1), ("no-pmi", -4),
    ("pmi-path", -3), ("unbound", -2),
])
def test_errors_enqueue_nothing(case, code):
    """Each validation error returns its code with nothing queued: the state, the step counter, the launch count, the
    episode count and the output are unchanged, and a following step on the twin environments gives identical results."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample, policy_weights
    E = 6
    ref, cfg = make_env(10, 10, E, "MAAC-G")
    env, _ = make_env(10, 10, E, "MAAC-G")
    net = make_policy()
    w, _params = policy_weights(net, 12)
    launches, steps = env.launch_count(), env._lib.uavsim_step_count(env._h)
    kw = {}
    if case == "episodes<0":
        kw = dict(K=-1)
    elif case == "nsteps<0":
        kw = dict(T=-1)
    elif case == "null-seeds":
        kw = dict(seeds=None)
    elif case == "null-out":
        kw = dict(out="null")
    elif case == "misaligned-out":
        kw = dict(out="misaligned")
    elif case == "greedy=2":
        kw = dict(greedy=2)
    elif case == "bad-mode":
        kw = dict(mode=7)
    elif case == "null-weights":
        w.w2 = None
    elif case == "hidden0":
        w.hidden = 0
    elif case == "n_actions":
        w, _params = policy_weights(make_policy(na=5), 12)
    elif case == "no-pmi":
        kw = dict(mode=2)
    elif case == "pmi-path":  # the tensor path selected before weights it cannot serve were uploaded
        _cabi.check(env._lib.uavsim_set_pmi_path(env._h, 2), "uavsim_set_pmi_path")
        env.set_pmi(make_pmi(32))
        kw = dict(mode=2)
    if case == "unbound":
        from marl_uavs_targets_tracking_b200 import default_config, params_from_config
        p = params_from_config(default_config("MAAC-G"), 10, 10, 2000, 2000, 12)
        h = C.c_void_p()
        _cabi.check(env._lib.uavsim_create(C.byref(p), 8, 0, 0, C.byref(h)), "uavsim_create")
        seeds = (C.c_uint64 * 1)(1)
        buf = torch.zeros(8 * 6, dtype=torch.float64, device=DEV)
        try:
            rc = env._lib.uavsim_evaluate_policy(h, 1, 0.3, C.byref(w), 0, 1, 1, seeds, 1, 4, C.c_void_p(buf.data_ptr()),
                                                 None)
            assert env._lib.uavsim_launch_count(h) == 0 and env._lib.uavsim_step_count(h) == 0
        finally:
            env._lib.uavsim_destroy(h)
        assert rc == code
    else:
        rc, buf = _raw_call(env, w, **kw)
        assert rc == code, (case, rc, env._lib.uavsim_last_error())
    torch.cuda.synchronize()
    assert bool((buf == 0).all())
    assert env.launch_count() == launches and env._lib.uavsim_step_count(env._h) == steps
    assert_same_env(ref, env)
    for e in (ref, env):
        fused_policy_sample(net, e.get_states().view(-1, 12), 2, 2, out=e.actions.view(-1))
        e.step_device(cfg, None)
    assert_same_env(ref, env)
    ref.close()
    env.close()
