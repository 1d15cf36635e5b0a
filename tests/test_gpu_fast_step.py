"""The two 64 x 64 step kernels -- the all-pairs tile kernel (csrc/step_tile_kernel.cuh, step path 3, the default for
this shape) and the per-UAV fast kernel (csrc/step_fast_kernel.cuh, step path 2) -- against the CPU oracle and against
the generic kernel.

The fast kernel classifies every pair in fp32 with a two-sided guard and sends a UAV to the fp64 path only when a
pair falls inside the guard band; these tests pin (i) both template instances (plain, and with masks / per-target
counts) to the oracle and (ii) the two kernels to each other on every integer output.  Pairs placed exactly on the
thresholds, for these and the other step kernels, are in test_gpu_pair_thresholds.py.
"""
import numpy as np
import pytest
import torch

from gpu_util import MASKS, max_scaled_err, oracle_params_from_config

pytestmark = pytest.mark.gpu

TOL = 1e-5        # contract
TOL_TIGHT = 2e-6  # fp32 outputs of fp32 pair sums


def _env(n, m, cfg, E, **kw):
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment
    e = cfg["environment"]
    return BatchedEnvironment(n, m, e["x_max"], e["y_max"], e["na"], n_envs=E, device="cuda:0", **kw)


PATHS = [3, 2]


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("method,T", [("MAAC-G", 200), ("MAAC", 40)])
def test_plain_instance_matches_the_oracle(oracle, method, T, path):
    """No masks, no per-target counts: the instance the benchmark runs.  Whole episode, Philox reset and policy."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 64
    cfg = default_config(method, n, m)
    E = 80
    env = _env(n, m, cfg, E, seed=77)
    env.set_step_path(path)
    env.reset(cfg)
    P = oracle_params_from_config(cfg, n, m)
    st = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    omode = {"MAAC": 0, "MAAC-G": 1}[method]
    wo = wr = wp = 0.0
    for t in range(T):
        a = env.random_actions(11, t).cpu().numpy().copy()
        obs, rew4, cov = env.step_device(cfg, None)
        ref = oracle.step_batch(P, omode, float(cfg["cooperative"]), None, st, a, nthreads=8)
        assert np.array_equal(cov.cpu().numpy(), ref["covered"]), t
        wo = max(wo, max_scaled_err(obs.double().cpu().numpy(), ref["obs"]))
        wr = max(wr, max_scaled_err(rew4.double().cpu().numpy(), ref["rew4"]))
        got = env.get_state()
        for k in ("ux", "uy", "uh", "tx", "ty", "th"):
            wp = max(wp, max_scaled_err(got[k].cpu().numpy(), st[k]))
        assert np.array_equal(got["ua"].cpu().numpy(), st["ua"])
    print(method, "obs %.1e rew %.1e state %.1e" % (wo, wr, wp))
    assert wo <= TOL_TIGHT and wr <= TOL_TIGHT and wp <= 1e-9
    s = env.episode_stats()
    assert s["env_steps"] == E * T
    env.close()


@pytest.mark.parametrize("fast_path", PATHS)
def test_fast_and_generic_kernels_agree(fast_path):
    """Same seeds through both kernels: every integer output identical (masks, counts, coverage, last actions), state
    equal to 1e-9 (the kernels use different sine routines, each within 2 ulp), floats within the tight tolerance."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 64
    cfg = default_config("MAAC-G", n, m)
    E = 150
    envs = []
    for path in (1, fast_path):
        env = _env(n, m, cfg, E, seed=5, record_masks=True, track_counts=True)
        env.set_step_path(path)
        env.reset(cfg)
        envs.append(env)
    g, f = envs
    for t in range(120):
        g.random_actions(3, t)
        f.random_actions(3, t)
        og, rg, cg = g.step_device(cfg, None)
        of, rf, cf = f.step_device(cfg, None)
        assert torch.equal(cg, cf), t
        assert torch.equal(g.tracker_counts, f.tracker_counts), t
        for k in MASKS:
            assert torch.equal(g.masks[k], f.masks[k]), (t, k)
        assert max_scaled_err(of.double().cpu().numpy(), og.double().cpu().numpy()) <= TOL_TIGHT
        assert max_scaled_err(rf.double().cpu().numpy(), rg.double().cpu().numpy()) <= TOL_TIGHT
        sg, sf = g.get_state(), f.get_state()
        for k in ("ux", "uy", "uh", "tx", "ty", "th"):
            assert max_scaled_err(sf[k].cpu().numpy(), sg[k].cpu().numpy()) <= 1e-9, (t, k)
    a, b = g.episode_stats(), f.episode_stats()
    assert a["covered_sum"] == b["covered_sum"] and a["covered_max"] == b["covered_max"]
    for k in ("rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment"):
        assert abs(a[k] - b[k]) <= 1e-6 * max(1.0, abs(a[k]))
    g.close()
    f.close()


@pytest.mark.parametrize("path", PATHS)
def test_wide_swarms_fall_back_to_fp64_per_environment(oracle, path):
    """Beyond r_fast (about 33 x min(dp, dc) from the map centre) the fp32 offsets would cost more than 2e-6 in the
    observation: such an environment takes the fp64 path as a whole, its neighbours in the batch stay fast."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 64
    cfg = default_config("MAAC-G", n, m)
    E = 6
    env = _env(n, m, cfg, E, seed=4, track_counts=True)
    env.set_step_path(path)
    env.reset(cfg)
    st = env.get_state()
    st["ux"][1, :] += 2.0e4
    st["tx"][1, :] += 2.0e4
    st["ux"][3, 7] = -9.0e3          # one UAV outside r_fast, inside the prefilter radius of the generic kernel
    st["ty"][4, 2] = 6.0e4
    env.set_state(cfg, *(st[k] for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    P = oracle_params_from_config(cfg, n, m)
    host = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    for t in range(5):
        a = env.random_actions(3, t).cpu().numpy().copy()
        obs, rew4, cov = env.step_device(cfg, None)
        ref = oracle.step_batch(P, 1, float(cfg["cooperative"]), None, host, a, nthreads=4)
        assert np.array_equal(cov.cpu().numpy(), ref["covered"])
        assert np.array_equal(env.tracker_counts.cpu().numpy(), ref["tracker_cnt"])
        assert max_scaled_err(obs.double().cpu().numpy(), ref["obs"]) <= TOL_TIGHT
        assert max_scaled_err(rew4.double().cpu().numpy(), ref["rew4"]) <= TOL_TIGHT
    env.close()


def test_fast_path_is_refused_for_other_shapes():
    from marl_uavs_targets_tracking_b200 import UavSimError, default_config
    cfg = default_config("MAAC", 10, 10)
    env = _env(10, 10, cfg, 4)
    env.reset(cfg)
    for path in PATHS:
        with pytest.raises(UavSimError):
            env.set_step_path(path)
    env.close()


@pytest.mark.parametrize("n,m,method", [(10, 10, "MAAC-G"), (10, 10, "MAAC-R"), (7, 5, "MAAC-G"), (16, 16, "MAAC"),
                                         (1, 1, "MAAC-G"), (3, 16, "MAAC-G"), (16, 2, "MAAC-R")])
def test_small_swarm_and_generic_kernels_agree(n, m, method):
    """The two-warp small-swarm kernel (csrc/step_small_kernel.cuh, step path 4) against the generic kernel (path 1) on
    the same seeds: masks, per-target counts, coverage and last actions identical; for MAAC-R also the neighbour sets
    handed to the PMI kernel (through the final reward); state to 1e-9 (different sine routines), floats tight.  Ragged
    group sizes: E = 37 is not a multiple of any group."""
    from marl_uavs_targets_tracking_b200 import PMINetwork, default_config
    cfg = default_config(method, n, m)
    pmi = None
    if method == "MAAC-R":
        torch.manual_seed(5)
        pmi = PMINetwork(hidden_dim=128)
        pmi.eval()
    E = 37
    envs = []
    for path in (1, 4):
        env = _env(n, m, cfg, E, seed=9, record_masks=True, track_counts=True)
        env.set_step_path(path)
        env.reset(cfg)
        envs.append(env)
    g, f = envs
    for t in range(60):
        g.random_actions(3, t)
        f.random_actions(3, t)
        og, rg, cg = g.step_device(cfg, pmi)
        of, rf, cf = f.step_device(cfg, pmi)
        assert torch.equal(cg, cf), t
        assert torch.equal(g.tracker_counts, f.tracker_counts), t
        for k in MASKS:
            assert torch.equal(g.masks[k], f.masks[k]), (t, k)
        assert max_scaled_err(of.double().cpu().numpy(), og.double().cpu().numpy()) <= TOL_TIGHT
        assert max_scaled_err(rf.double().cpu().numpy(), rg.double().cpu().numpy()) <= TOL_TIGHT
        sg, sf = g.get_state(), f.get_state()
        for k in ("ux", "uy", "uh", "tx", "ty", "th"):
            assert max_scaled_err(sf[k].cpu().numpy(), sg[k].cpu().numpy()) <= 1e-9, (t, k)
        assert torch.equal(sg["ua"], sf["ua"])
    a, b = g.episode_stats(), f.episode_stats()
    assert a["covered_sum"] == b["covered_sum"] and a["covered_max"] == b["covered_max"] and a["env_steps"] == b["env_steps"]
    for k in ("rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment"):
        assert abs(a[k] - b[k]) <= 1e-6 * max(1.0, abs(a[k]))
    g.close()
    f.close()


def test_small_swarm_rollout_loop_draws_the_same_actions():
    """uavsim_run_random_policy on the small-swarm kernel draws the policy inside the step kernel (one launch per step,
    programmatic dependent launch): same Philox draws, same results as random_actions + step, step by step."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 10
    cfg = default_config("MAAC-G", n, m)
    E = 500
    a = _env(n, m, cfg, E, seed=21)
    b = _env(n, m, cfg, E, seed=21)
    for env in (a, b):
        env.set_step_path(4)
        env.reset(cfg)
    T = 25
    for t in range(T):
        a.random_actions(77, t)
        oa, ra, ca = a.step_device(cfg, None)
    ob, rb, cb = b.run_random_policy(cfg, None, 77, 0, T)
    assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(ca, cb)
    assert torch.equal(a.actions, b.actions)
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert a.episode_stats() == b.episode_stats()
    a.close()
    b.close()


def test_64x64_kernels_hand_the_same_neighbour_sets_to_the_pmi_kernel():
    """MAAC-R at 64 x 64: the step kernels export raw rewards and neighbour bit sets, the PMI kernel finishes the reward.
    Generic (1), per-UAV (2) and tile (3) kernels on the same seeds: final rewards within the tight tolerance, every other
    output as in the MAAC-G comparison."""
    from marl_uavs_targets_tracking_b200 import PMINetwork, default_config
    n = m = 64
    cfg = default_config("MAAC-R", n, m)
    torch.manual_seed(11)
    pmi = PMINetwork(hidden_dim=128)
    pmi.eval()
    E = 24
    envs = []
    for path in (1, 2, 3):
        env = _env(n, m, cfg, E, seed=13)
        env.set_step_path(path)
        env.reset(cfg)
        envs.append(env)
    for t in range(25):
        outs = []
        for env in envs:
            env.random_actions(5, t)
            o, r, c = env.step_device(cfg, pmi)
            outs.append((o.double().cpu().numpy(), r.double().cpu().numpy(), c.cpu().numpy()))
        for k in (1, 2):
            assert np.array_equal(outs[0][2], outs[k][2]), (t, k)
            assert max_scaled_err(outs[k][0], outs[0][0]) <= TOL_TIGHT, (t, k)
            assert max_scaled_err(outs[k][1], outs[0][1]) <= TOL_TIGHT, (t, k)
    for env in envs:
        env.close()


def test_counter_scheduled_launch_is_reproducible_and_complete():
    """The fast kernel hands environments beyond the first wave of CTAs out from a launch-wide counter, so which CTA
    steps which environment depends on timing.  With more environments than resident CTAs (8 192 > 148 x 14), two runs
    of the same seeds must still give identical outputs, identical state and IDENTICAL statistics (fixed-point sums),
    every environment must be stepped exactly once per launch (env_steps, and the generic kernel as the witness), and
    the counter must be back at zero for the next launch."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 64
    cfg = default_config("MAAC-G", n, m)
    E, T = 8192, 12
    runs = []
    for path in (2, 2, 1):
        env = _env(n, m, cfg, E, seed=31)
        env.set_step_path(path)
        env.reset(cfg)
        for t in range(T):
            env.random_actions(5, t)
            obs, rew4, cov = env.step_device(cfg, None)
        runs.append((obs.clone(), rew4.clone(), cov.clone(), {k: v.clone() for k, v in env.get_state().items()}, env.episode_stats()))
        env.close()
    a, b, g = runs
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    for k in a[3]:
        assert torch.equal(a[3][k], b[3][k]), k
    assert a[4] == b[4], (a[4], b[4])
    assert a[4]["env_steps"] == E * T
    assert torch.equal(a[2], g[2]) and torch.equal(a[3]["ua"], g[3]["ua"])
    assert max_scaled_err(a[0].double().cpu().numpy(), g[0].double().cpu().numpy()) <= TOL_TIGHT
    assert max_scaled_err(a[1].double().cpu().numpy(), g[1].double().cpu().numpy()) <= TOL_TIGHT
    assert a[4]["covered_sum"] == g[4]["covered_sum"] and a[4]["covered_max"] == g[4]["covered_max"]
    for k in ("rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment"):
        assert abs(a[4][k] - g[4][k]) <= 1e-6 * max(1.0, abs(g[4][k])), k


def test_rollout_loop_and_stepwise_route_agree_between_the_kernel_ranges():
    """Between ~2.5 and ~10 waves of the small-swarm kernel's CTAs the rollout loop below the FFI (policy drawn inside the
    small-swarm kernel) and the step-by-step route (random_actions + step: generic kernel) run DIFFERENT kernels on the
    same Philox draws: every integer output and the state's last actions must be identical, floats within 2e-6."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 10
    cfg = default_config("MAAC-G", n, m)
    E, T = 20000, 15
    a, b = _env(n, m, cfg, E, seed=41), _env(n, m, cfg, E, seed=41)
    a.reset(cfg); b.reset(cfg)
    for t in range(T):
        a.random_actions(13, t)
        oa, ra, ca = a.step_device(cfg, None)
    ob, rb, cb = b.run_random_policy(cfg, None, 13, 0, T)
    assert torch.equal(ca, cb)
    sa, sb = a.get_state(), b.get_state()
    assert torch.equal(sa["ua"], sb["ua"])
    for k in ("ux", "uy", "uh", "tx", "ty", "th"):
        assert max_scaled_err(sa[k].cpu().numpy(), sb[k].cpu().numpy()) <= 1e-9, k
    assert max_scaled_err(oa.double().cpu().numpy(), ob.double().cpu().numpy()) <= TOL_TIGHT
    assert max_scaled_err(ra.double().cpu().numpy(), rb.double().cpu().numpy()) <= TOL_TIGHT
    x, y = a.episode_stats(), b.episode_stats()
    assert x["covered_sum"] == y["covered_sum"] and x["covered_max"] == y["covered_max"] and x["env_steps"] == y["env_steps"] == E * T
    for k in ("rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment"):
        assert abs(x[k] - y[k]) <= 1e-6 * max(1.0, abs(x[k])), k
    a.close(); b.close()
