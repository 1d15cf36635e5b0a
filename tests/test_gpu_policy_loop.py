"""uavsim_run_policy / BatchedEnvironment.run_policy: a learned-policy episode queued in one library call is bit-identical
to driving the same steps from Python (bind_obs, bind_actions, fused_policy_sample, step_device) in every output."""
import ctypes as C
import os
import subprocess

import pytest
import torch

from conftest import ROOT

from marl_uavs_targets_tracking_b200 import _cabi

FIELDS = ("obs", "actions", "rew4", "covered")


def test_trajectory_struct_layout_matches_the_header(tmp_path):
    """sizeof() and field offsets of UavSimTrajectory seen by the C compiler == the ctypes layout."""
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "uavsim.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
           ' sizeof(UavSimTrajectory), offsetof(UavSimTrajectory, obs), offsetof(UavSimTrajectory, actions),'
           ' offsetof(UavSimTrajectory, rew4), offsetof(UavSimTrajectory, covered));return 0;}')
    exe = str(tmp_path / "uavsim_traj_sizeof")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    got = list(map(int, subprocess.check_output([exe]).split()))
    T = _cabi.UavSimTrajectory
    assert got == [C.sizeof(T)] + [getattr(T, f).offset for f in FIELDS]


# ------------------------------------------------------------------------------------------------ GPU helpers
DEV = "cuda:0"


def make_env(n, m, E, method, num_steps=0, step_path=0, pmi_path=0, seed=3):
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    cfg = default_config(method, n, m)
    env = BatchedEnvironment(n, m, 2000, 2000, 12, n_envs=E, device=DEV, seed=seed, num_steps=num_steps)
    if step_path:
        env.set_step_path(step_path)
    if pmi_path:
        env.set_pmi_path(pmi_path)
    env.reset(cfg)
    return env, cfg


def make_policy(hidden=64, na=12, seed=0):
    from marl_uavs_targets_tracking_b200.rollout import PolicyNet
    torch.manual_seed(seed)
    return PolicyNet(12, hidden, na).to(DEV)


def make_pmi(hidden):
    from marl_uavs_targets_tracking_b200 import PMINetwork
    torch.manual_seed(hidden)
    return PMINetwork(hidden_dim=hidden).eval()


def alloc_traj(env, T, fields):
    """Trajectory tensors filled with NaN / -7: a slot neither path writes makes the comparison fail."""
    E, n = env.n_envs, env.n_uav
    shapes = {"obs": ((T + 1, E, n, 12), torch.float32), "actions": ((T, E, n), torch.int32),
              "rew4": ((T, 4, E, n), torch.float32), "covered": ((T, E), torch.int32)}
    return {f: torch.full(shapes[f][0], float("nan") if shapes[f][1] == torch.float32 else -7, dtype=shapes[f][1],
                          device=DEV) for f in fields}


def reference_loop(env, cfg, pmi, net, seed, c0, T, obs=None, actions=None, rew4=None, covered=None):
    """The per-step loop run_policy replaces: step k draws with counter c0 + k from slot k (or the bound buffers)."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    E, n = env.n_envs, env.n_uav
    home_obs, home_act = env._obs, env.actions
    if obs is not None:
        obs[0].copy_(home_obs)
    for k in range(T):
        if obs is not None:
            env.bind_obs(obs[k + 1])
        if actions is not None:
            env.bind_actions(actions[k])
        states = (obs[k] if obs is not None else home_obs).view(E * n, 12)
        fused_policy_sample(net, states, seed, c0 + k, out=env.actions.view(-1))
        env.step_device(cfg, pmi)
        if rew4 is not None:
            rew4[k].copy_(env._rew4)
        if covered is not None:
            covered[k].copy_(env._covered)
    if obs is not None:
        if T:
            home_obs.copy_(obs[T])
        env.bind_obs(home_obs)
    if actions is not None:
        if T:
            home_act.copy_(actions[T - 1])
        env.bind_actions(home_act)


def snapshot(env):
    d = {k: v.clone() for k, v in env.get_state().items()}
    d.update(obs=env.get_states().clone(), actions=env.actions.clone(), rew4=env._rew4.clone(),
             covered=env._covered.clone(), done=env.done.clone())
    return d


def assert_same_env(a, b):
    sa, sb = snapshot(a), snapshot(b)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert a.episode_stats() == b.episode_stats()
    assert a._lib.uavsim_step_count(a._h) == b._lib.uavsim_step_count(b._h)


def cuda_kernels(fn):
    """Names of the kernels `fn` launches (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " | ".join(e.key for e in prof.key_averages())


def run_both(n, m, E, method, T, fields=FIELDS, step_path=0, pmi=None, pmi_path=0, hidden=64, num_steps=0,
             expect_kernels=(), seed=11, c0=5):
    """Reference loop on one environment, run_policy on a twin; asserts every output equal.  Returns both."""
    ref, cfg = make_env(n, m, E, method, num_steps, step_path, pmi_path)
    env, _ = make_env(n, m, E, method, num_steps, step_path, pmi_path)
    net = make_policy(hidden)
    tr_ref, tr = alloc_traj(ref, T, fields), alloc_traj(env, T, fields)
    reference_loop(ref, cfg, pmi, net, seed, c0, T, **tr_ref)
    launches0 = env.launch_count()
    call = lambda: env.run_policy(cfg, pmi, net, seed, c0, T, **tr)  # noqa: E731
    if expect_kernels:
        names = cuda_kernels(call)
        for k in expect_kernels:
            assert k in names, (k, names)
    else:
        call()
    # one policy launch per step, counted; the step and PMI launches are the reference's
    assert env.launch_count() - launches0 - T == ref.launch_count() - launches0
    for f in fields:
        assert torch.equal(tr_ref[f], tr[f]), f
    assert_same_env(ref, env)
    return ref, env, cfg, net


# ------------------------------------------------------------------------------------------------ step kernels
@pytest.mark.gpu
@pytest.mark.parametrize("n,m,E,step_path,kernel", [
    (10, 10, 301, 0, "uavsim_step_small_kernel"),     # 100 full groups of 3 and a partial one
    (10, 10, 301, 1, "uavsim_step_kernel<"),
    (10, 10, 32768, 0, "uavsim_step_kernel<"),        # beyond ~2.5 waves of small-kernel CTAs: the automatic choice
    (64, 64, 96, 0, "uavsim_step_fast_kernel"),
    (64, 64, 96, 3, "uavsim_step_tile_kernel"),
    (7, 5, 9, 1, "uavsim_step_kernel<"),
    (7, 5, 9, 0, "uavsim_step_small_kernel"),         # groups of 4: a partial last group, E*n % 4 != 0
], ids=["small-10x10", "generic-10x10", "generic-auto-10x10", "fast-64x64", "tile-64x64", "generic-7x5", "small-7x5"])
def test_every_step_kernel(n, m, E, step_path, kernel):
    T = 25 if E <= 1024 else 6
    ref, env, _, _ = run_both(n, m, E, "MAAC-G", T, step_path=step_path, num_steps=T - 3,
                              expect_kernels=(kernel, "uavsim_policy_kernel<12, true>"))
    assert int(env.done.min()) == 1  # the episode length was reached inside the call
    ref.close()
    env.close()


# ------------------------------------------------------------------------------------------------ reward modes
@pytest.mark.gpu
@pytest.mark.parametrize("method,pmi_hidden,kernel", [
    ("MAAC", 0, None), ("MAAC-G", 0, None),
    ("MAAC-R", 128, "uavsim_pmi_tc_kernel"),   # tensor-core PMI path
    ("MAAC-R", 32, "uavsim_pmi_kernel<"),      # CUDA-core PMI path
], ids=["MAAC", "MAAC-G", "MAAC-R-tensor-h128", "MAAC-R-cudacore-h32"])
def test_every_reward_mode(method, pmi_hidden, kernel):
    pmi = make_pmi(pmi_hidden) if pmi_hidden else None
    ref, env, _, _ = run_both(10, 10, 301, method, 25, pmi=pmi, hidden=128, expect_kernels=(kernel,) if kernel else ())
    ref.close()
    env.close()


@pytest.mark.gpu
def test_pmi_reward_on_the_generic_kernel():
    ref, env, _, _ = run_both(10, 10, 301, "MAAC-R", 12, step_path=1, pmi=make_pmi(128))
    ref.close()
    env.close()


# ------------------------------------------------------------------------------------------------ trajectory shapes
@pytest.mark.gpu
@pytest.mark.parametrize("T", [0, 1, 25])
@pytest.mark.parametrize("fields", [FIELDS, (), ("obs",), ("actions",), ("rew4",), ("covered",)],
                         ids=["all", "none", "obs", "actions", "rew4", "covered"])
def test_trajectory_fields(fields, T):
    ref, env, _, _ = run_both(10, 10, 37, "MAAC-G", T, fields=fields, num_steps=20)
    ref.close()
    env.close()


@pytest.mark.gpu
def test_null_trajectory_steps_in_place():
    """traj = NULL in the C call: everything in the bound buffers, as the in-place reference loop."""
    from marl_uavs_targets_tracking_b200 import MODE_MEAN
    from marl_uavs_targets_tracking_b200.rollout import policy_weights
    ref, cfg = make_env(10, 10, 37, "MAAC-G")
    env, _ = make_env(10, 10, 37, "MAAC-G")
    net = make_policy()
    reference_loop(ref, cfg, None, net, 3, 1, 9)
    w, _params = policy_weights(net, 12)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _cabi.check(env._lib.uavsim_run_policy(env._h, MODE_MEAN, float(cfg["cooperative"]), C.byref(w), 3, 1, 9, None,
                                           stream), "uavsim_run_policy")
    assert_same_env(ref, env)
    ref.close()
    env.close()


# ------------------------------------------------------------------------------------------------ continuation
@pytest.mark.gpu
@pytest.mark.parametrize("fields", [FIELDS, ()], ids=["trajectory", "in-place"])
def test_a_python_step_continues_the_episode(fields):
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    T, seed, c0 = 25, 11, 5
    ref, env, cfg, net = run_both(10, 10, 301, "MAAC-G", T, fields=fields)
    for e in (ref, env):
        fused_policy_sample(net, e.get_states().view(-1, 12), seed, c0 + T, out=e.actions.view(-1))
        e.step_device(cfg, None)
    assert_same_env(ref, env)
    ref.close()
    env.close()


# ------------------------------------------------------------------------------------------------ operate_epoch_batched
def reference_operate(config, env, agent, pmi, num_steps, keep_transitions):
    """operate_epoch_batched driven step by step from Python (the fused-policy loop it replaces)."""
    from marl_uavs_targets_tracking_b200.distributed import episode_summary, reduce_episode_stats
    E, n = env.n_envs, env.n_uav
    if keep_transitions:
        home_obs, home_act = env._obs, env.actions
        traj = torch.empty((num_steps + 1, E, n, 12), dtype=torch.float32, device=env.device)
        acts = torch.empty((num_steps, E, n), dtype=torch.int32, device=env.device)
        rews = torch.empty((num_steps, E * n), dtype=torch.float32, device=env.device)
        traj[0].copy_(env._obs)
        for step in range(num_steps):
            config["step"] = step + 1
            env.bind_obs(traj[step + 1])
            env.bind_actions(acts[step])
            agent.take_actions(traj[step].view(E * n, 12), out=acts[step].view(-1))
            _, rew4, _ = env.step_device(config, pmi)
            rews[step].copy_(rew4[0].reshape(E * n))
        home_obs.copy_(traj[num_steps])
        env.bind_obs(home_obs)
        env.bind_actions(home_act)
        transitions = {"states": traj[:-1].reshape(num_steps * E * n, 12), "actions": acts.reshape(-1),
                       "rewards": rews.reshape(-1), "next_states": traj[1:].reshape(num_steps * E * n, 12)}
    else:
        for step in range(num_steps):
            config["step"] = step + 1
            agent.take_actions(env._obs.view(E * n, 12), out=env.actions.view(-1))
            env.step_device(config, pmi)
        transitions = None
    stats = reduce_episode_stats(env.episode_stats(), device=env.device)
    return transitions, episode_summary(stats, n)


@pytest.mark.gpu
@pytest.mark.parametrize("keep", [True, False], ids=["keep", "no-transitions"])
@pytest.mark.parametrize("method", ["MAAC-G", "MAAC-R"])
def test_operate_epoch_batched_makes_one_call_with_the_same_result(keep, method):
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, operate_epoch_batched
    E, T = 301, 25
    pmi = make_pmi(128) if method == "MAAC-R" else None
    out = []
    for driver in (reference_operate, operate_epoch_batched):
        env, cfg = make_env(10, 10, E, method, num_steps=T)
        torch.manual_seed(0)
        agent = BatchedActorCritic(12, 128, 12, 1e-3, 1e-3, 0.95, torch.device(DEV), seed=7)
        agent._calls = 40  # a later episode: the counters continue
        tr, summary = driver(cfg, env, agent, pmi, T, keep_transitions=keep)
        out.append((tr, summary, agent._calls, cfg["step"], snapshot(env), env.launch_count(), env))
    (tr0, s0, c0, st0, sn0, l0, e0), (tr1, s1, c1, st1, sn1, l1, e1) = out
    assert (tr0 is None) == (tr1 is None) == (not keep)
    if keep:
        for k in tr0:
            assert tr1[k].shape == tr0[k].shape and tr1[k].dtype == tr0[k].dtype, k
            assert torch.equal(tr0[k], tr1[k]), k
        assert tr1["next_states"].data_ptr() == tr1["states"].data_ptr() + E * 10 * 12 * 4
    assert s0 == s1
    assert c0 == c1 == 40 + T and st0 == st1 == T
    for k in sn0:
        if k != "actions" or not keep:  # (the per-step loop leaves the bound action buffer as it found it)
            assert torch.equal(sn0[k], sn1[k]), k
    assert l1 == l0 + T  # the policy launches, counted by the library
    e0.close()
    e1.close()


# ------------------------------------------------------------------------------------------------ errors
@pytest.mark.gpu
def test_unbound_handle_is_refused():
    from marl_uavs_targets_tracking_b200 import default_config, params_from_config
    from marl_uavs_targets_tracking_b200.rollout import policy_weights
    lib = _cabi.load()
    p = params_from_config(default_config("MAAC-G"), 10, 10, 2000, 2000, 12)
    h = C.c_void_p()
    _cabi.check(lib.uavsim_create(C.byref(p), 8, 0, 0, C.byref(h)), "uavsim_create")
    w, _params = policy_weights(make_policy(), 12)
    try:
        assert lib.uavsim_run_policy(h, 1, 0.3, C.byref(w), 1, 1, 5, None, None) == -2  # UAVSIM_ERR_UNBOUND
        assert lib.uavsim_launch_count(h) == 0 and lib.uavsim_step_count(h) == 0
    finally:
        lib.uavsim_destroy(h)


@pytest.mark.gpu
@pytest.mark.parametrize("case,code", [("n_actions", -1), ("hidden0", -3), ("hidden513", -3), ("nsteps", -1),
                                       ("misaligned", -3)])
def test_errors_enqueue_nothing_and_leave_the_binding(case, code):
    """Each validation error returns its code with nothing queued: the state, the step counter, the launch count and the
    bound pointers are unchanged (a following Python step on the twin environments gives identical results)."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample, policy_weights
    n = 64 if case == "misaligned" else 10
    E, T = 6, 4
    ref, cfg = make_env(n, n, E, "MAAC-G", step_path=2 if case == "misaligned" else 0)
    env, _ = make_env(n, n, E, "MAAC-G", step_path=2 if case == "misaligned" else 0)
    net = make_policy()
    tr = alloc_traj(env, T, FIELDS)
    launches, steps = env.launch_count(), env._lib.uavsim_step_count(env._h)
    if case == "misaligned":  # a contiguous action trajectory 4 bytes off a 16-byte boundary
        tr["actions"] = torch.full((T * E * n + 1,), -7, dtype=torch.int32, device=DEV)[1:].view(T, E, n)
    if case in ("n_actions", "nsteps", "misaligned"):
        pol = make_policy(na=5) if case == "n_actions" else net
        with pytest.raises(_cabi.UavSimError, match=r"code %d\)" % code):
            env.run_policy(cfg, None, pol, 1, 1, -1 if case == "nsteps" else T, **({} if case == "nsteps" else tr))
    else:
        w, _params = policy_weights(net, 12)
        w.hidden = 0 if case == "hidden0" else 513
        traj = _cabi.UavSimTrajectory(*(t.data_ptr() for t in tr.values()))
        rc = env._lib.uavsim_run_policy(env._h, 1, 0.3, C.byref(w), 1, 1, T, C.byref(traj),
                                        C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == code
    assert env.launch_count() == launches and env._lib.uavsim_step_count(env._h) == steps
    for f, t in tr.items():  # nothing was written to the trajectory
        assert bool((t.isnan() if t.dtype == torch.float32 else t == -7).all()), f
    assert_same_env(ref, env)
    for e in (ref, env):
        fused_policy_sample(net, e.get_states().view(-1, 12), 2, 2, out=e.actions.view(-1))
        e.step_device(cfg, None)
    assert_same_env(ref, env)
    ref.close()
    env.close()
