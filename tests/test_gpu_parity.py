"""GPU parity: the CUDA path (through the C ABI) against the golden vectors recorded from the
reference and against the CPU oracle on seeded batches.

Bars (BASELINE.json north_star): integer / index outputs bit-exact -- the five range masks, the
covered count, per-target tracker counts, the done flag; float state and rewards within 1e-5.
Tolerance rule: |got - ref| <= TOL * max(|ref|, 1) for observations and rewards (they cross zero),
true relative error for positions.  TOL = 1e-5 is the contract; the observed error is ~1e-7 (outputs
are stored as fp32) and the tests also assert a tighter 2e-6 so regressions are caught early.
"""
import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden
from gpu_util import (MASKS, golden_config, golden_pmi_module, max_scaled_err, oracle_params_from_config,
                      oracle_pmi_from_module)

pytestmark = pytest.mark.gpu

TOL = 1e-5         # contract
TOL_TIGHT = 2e-6   # what fp32 outputs of an fp64 computation should achieve
TOL_PMI = 1e-5     # MAAC-R reward (fp32 MLP, different summation order)


def _env(n, m, cfg, E, **kw):
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment
    e = cfg["environment"]
    return BatchedEnvironment(n, m, e["x_max"], e["y_max"], e["na"], n_envs=E, device="cuda:0", **kw)


@pytest.mark.parametrize("name", golden_names())
def test_cuda_matches_reference_golden(name):
    """Replayed reset + recorded actions, E=3 identical environments (so one CTA holds several)."""
    g = load_golden(name)
    cfg = golden_config(g)
    n, m, T = int(g["params_i"][0]), int(g["params_i"][1]), int(g["params_i"][3])
    mode = int(g["params_i"][5])
    pmi = golden_pmi_module(g)
    E = 3
    env = _env(n, m, cfg, E, record_masks=True, track_counts=True, num_steps=T)
    rep = lambda a: np.broadcast_to(np.asarray(a), (E,) + np.asarray(a).shape).copy()  # noqa: E731
    env.set_state(cfg, *(rep(g[k + "0"]) for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    obs0 = env.get_states().double().cpu().numpy()
    assert max_scaled_err(obs0[0], g["obs0"]) <= TOL_TIGHT
    worst = {}
    for t in range(T):
        a = torch.as_tensor(rep(g["actions"][t]), device="cuda:0")
        obs, rew, cov = env.step(cfg, pmi, a)
        st = {k: v.cpu().numpy() for k, v in env.get_state().items()}
        for e in range(E):
            # integer outputs: bit-exact
            for k in MASKS:
                assert np.array_equal(env.masks[k][e].cpu().numpy().astype(bool), g[k][t]), (name, t, k, e)
            assert int(cov[e]) == int(g["covered"][t]), (name, t, "covered")
            assert np.array_equal(env.tracker_counts[e].cpu().numpy(), g["cover_mask"][t].sum(0)), (name, t, "tracker")
            assert np.array_equal(st["ua"][e], g["actions"][t])
            assert int(env.done[e]) == int(t + 1 == T)
        for k in ("ux", "uy", "uh", "tx", "ty", "th"):
            err = float(np.max(np.abs(st[k][0] - g[k][t]) / np.maximum(np.abs(g[k][t]), 1e-300)))
            if k in ("uh", "th"):  # headings cross zero: scale by max(|ref|, 1)
                err = max_scaled_err(st[k][0], g[k][t])
            worst[k] = max(worst.get(k, 0.0), err)
            assert np.array_equal(st[k][0], st[k][E - 1])  # replicas agree bit for bit
        o = obs.double().cpu().numpy()
        worst["obs"] = max(worst.get("obs", 0.0), max_scaled_err(o[0], g["obs"][t]))
        for key, gk in (("rewards", "rewards"), ("target_tracking_reward", "tt"), ("boundary_punishment", "bp"),
                        ("duplicate_tracking_punishment", "dup")):
            r = rew[key].double().cpu().numpy()
            worst[gk] = max(worst.get(gk, 0.0), max_scaled_err(r[0], g[gk][t]))
            assert np.array_equal(r[0], r[E - 1])
    print(name, {k: "%.1e" % v for k, v in worst.items()})
    for k in ("ux", "uy", "uh", "tx", "ty", "th"):
        assert worst[k] <= 1e-9, (k, worst[k])       # fp64 state: far inside the 1e-5 bar
    for k in ("obs", "tt", "bp", "dup"):
        assert worst[k] <= TOL_TIGHT, (k, worst[k])
    assert worst["rewards"] <= (TOL_PMI if mode == 2 else TOL_TIGHT), worst["rewards"]
    env.close()


@pytest.mark.parametrize("n,m,method,E,T", [(10, 10, "MAAC", 256, 200), (10, 10, "MAAC-G", 256, 200),
                                             (10, 10, "MAAC-R", 128, 200), (64, 64, "MAAC-G", 64, 200),
                                             (64, 64, "MAAC-R", 16, 60), (64, 64, "MAAC", 64, 60),
                                             (128, 40, "MAAC-G", 5, 30), (3, 200, "MAAC-R", 7, 30)])
def test_cuda_matches_oracle_on_seeded_batches(oracle, n, m, method, E, T):
    """Philox reset + Philox random policy on the GPU; the oracle replays the same state and actions."""
    from marl_uavs_targets_tracking_b200 import PMINetwork, default_config
    cfg = default_config(method, n, m)
    coop = float(cfg["cooperative"])
    pmi = None
    if method == "MAAC-R":
        torch.manual_seed(1)
        pmi = PMINetwork(hidden_dim=128)
        for bn in (pmi.bn_comm, pmi.bn_obs, pmi.bn_boundary_state, pmi.bn1):
            bn.running_mean.normal_(0, 0.3)
            bn.running_var.uniform_(0.5, 1.5)
        pmi.eval()
    env = _env(n, m, cfg, E, track_counts=True, seed=123)
    env.reset(cfg)
    P = oracle_params_from_config(cfg, n, m)
    opmi = oracle_pmi_from_module(pmi) if pmi is not None else None
    omode = {"MAAC": 0, "MAAC-G": 1, "MAAC-R": 2}[method]
    st = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    worst = {"obs": 0.0, "rew": 0.0, "terms": 0.0, "pos": 0.0}
    for t in range(T):
        acts = env.random_actions(seed=99, step=t)
        a_host = acts.cpu().numpy().copy()
        assert a_host.min() >= 0 and a_host.max() < cfg["environment"]["na"]
        obs, rew4, cov = env.step_device(cfg, pmi)
        ref = oracle.step_batch(P, omode, coop, opmi, st, a_host, nthreads=8)
        assert np.array_equal(cov.cpu().numpy(), ref["covered"]), (t, "covered")
        assert np.array_equal(env.tracker_counts.cpu().numpy(), ref["tracker_cnt"]), (t, "tracker")
        worst["obs"] = max(worst["obs"], max_scaled_err(obs.double().cpu().numpy(), ref["obs"]))
        r = rew4.double().cpu().numpy()
        worst["rew"] = max(worst["rew"], max_scaled_err(r[0], ref["rew4"][0]))
        worst["terms"] = max(worst["terms"], max_scaled_err(r[1:], ref["rew4"][1:]))
        for k in ("ux", "uy", "tx", "ty"):
            worst["pos"] = max(worst["pos"], float(np.max(np.abs(env.get_state()[k].cpu().numpy() - st[k]) / np.maximum(np.abs(st[k]), 1.0))))
    print(n, m, method, {k: "%.1e" % v for k, v in worst.items()})
    assert worst["pos"] <= 1e-9
    assert worst["obs"] <= TOL_TIGHT and worst["terms"] <= TOL_TIGHT
    assert worst["rew"] <= (TOL_PMI if method == "MAAC-R" else TOL_TIGHT)
    # episode statistics accumulated on the device == sums of the per-step outputs (only last step checked here)
    env.close()


def test_origin_corner_in_the_warp_uniform_kernel(oracle):
    """64x64 kernel (warp = 32 UAVs of one environment): a UAV inside the 4 m x 4 m origin corner switches its
    whole warp to the exact per-row path; results must still match the oracle (weight quirk, uav.py:162-186)."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 64
    cfg = default_config("MAAC-G", n, m)
    env = _env(n, m, cfg, 6, track_counts=True, seed=9)
    env.reset(cfg)
    st = env.get_state()
    st["ux"][1, 5], st["uy"][1, 5] = 0.5, 0.7
    st["ux"][2, 40], st["uy"][2, 40] = -1.0, 1.5
    st["ux"][2, 41], st["uy"][2, 41] = 30.0, 40.0     # a partner within dc of the corner UAV
    st["tx"][1, 3], st["ty"][1, 3] = 50.0, 60.0        # a target within dp of it
    st["uh"][1, 5] = 0.0  # moves +20 m in x: out of the corner after the first step, in it before
    st["ux"][4, 7], st["uy"][4, 7], st["uh"][4, 7] = -19.5, 0.3, 0.0   # lands in the corner after the move
    env.set_state(cfg, *(st[k] for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    P = oracle_params_from_config(cfg, n, m)
    host = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    for t in range(4):
        a = env.random_actions(3, t).cpu().numpy().copy()
        obs, rew4, cov = env.step_device(cfg, None)
        ref = oracle.step_batch(P, 1, float(cfg["cooperative"]), None, host, a, nthreads=4)
        assert np.array_equal(cov.cpu().numpy(), ref["covered"])
        assert np.array_equal(env.tracker_counts.cpu().numpy(), ref["tracker_cnt"])
        assert max_scaled_err(obs.double().cpu().numpy(), ref["obs"]) <= TOL_TIGHT
        assert max_scaled_err(rew4.double().cpu().numpy(), ref["rew4"]) <= TOL_TIGHT
    env.close()


@pytest.mark.parametrize("case", range(6))
def test_origin_corner_under_random_scenarios(oracle, case):
    """The exact per-row path (UAVs inside the 4 m x 4 m origin corner, weight quirk of uav.py:162-186) with random
    scenario constants, small maps (many entities near the corner) and the shape-specialised kernels."""
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    rng = np.random.RandomState(300 + case)
    n, m = [(64, 64), (10, 10), (7, 33), (40, 3), (100, 9), (64, 64)][case]
    method = ("MAAC", "MAAC-G")[case % 2]
    cfg = default_config(method, n, m)
    side = float(rng.choice([40.0, 300.0, 2000.0]))
    cfg["environment"].update(x_max=side, y_max=side, na=int(rng.randint(2, 13)))
    cfg["uav"].update(v_max=float(rng.uniform(0.5, 8)), dt=float(rng.choice([0.5, 1.0])), dc=float(rng.uniform(0.1, 0.9) * side),
                      dp=float(rng.uniform(0.05, 0.6) * side))
    cfg["target"].update(v_max=float(rng.uniform(0.1, 3)))
    cfg["cooperative"] = 0.4 if method == "MAAC-G" else 0.0
    E = 9
    e = cfg["environment"]
    env = BatchedEnvironment(n, m, e["x_max"], e["y_max"], e["na"], n_envs=E, device="cuda:0", track_counts=True, seed=case)
    env.reset(cfg)
    st = env.get_state()
    for env_i in range(E):
        for _ in range(int(rng.randint(0, 4))):        # some environments keep no corner UAV
            i = int(rng.randint(0, n))
            st["ux"][env_i, i], st["uy"][env_i, i] = float(rng.uniform(-2.5, 2.5)), float(rng.uniform(-2.5, 2.5))
        if rng.rand() < 0.5:                           # a target and a partner close to the corner
            st["tx"][env_i, int(rng.randint(0, m))], st["ty"][env_i, int(rng.randint(0, m))] = float(rng.uniform(0, 5)), float(rng.uniform(0, 5))
            j = int(rng.randint(0, n))
            st["ux"][env_i, j], st["uy"][env_i, j] = float(rng.uniform(0, 6)), float(rng.uniform(0, 6))
    env.set_state(cfg, *(st[k] for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    P = oracle_params_from_config(cfg, n, m)
    host = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    for t in range(8):
        a = env.random_actions(3, t).cpu().numpy().copy()
        obs, rew4, cov = env.step_device(cfg, None)
        ref = oracle.step_batch(P, case % 2, float(cfg["cooperative"]), None, host, a, nthreads=4)
        assert np.array_equal(cov.cpu().numpy(), ref["covered"]), (case, t)
        assert np.array_equal(env.tracker_counts.cpu().numpy(), ref["tracker_cnt"]), (case, t)
        assert max_scaled_err(obs.double().cpu().numpy(), ref["obs"]) <= TOL_TIGHT, (case, t)
        assert max_scaled_err(rew4.double().cpu().numpy(), ref["rew4"]) <= TOL_TIGHT, (case, t)
    env.close()


@pytest.mark.parametrize("n,m", [(64, 64), (10, 10), (20, 7)])
def test_entities_beyond_the_prefilter_radius(oracle, n, m):
    """The fp32 prefilter is only proven within 32 768 m of the map centre; environments with an entity outside
    bypass it.  Mix near and very far entities and check masks-derived integers and values against the oracle."""
    from marl_uavs_targets_tracking_b200 import default_config
    cfg = default_config("MAAC-G", n, m)
    E = 8
    env = _env(n, m, cfg, E, track_counts=True, seed=4)
    env.reset(cfg)
    st = env.get_state()
    st["ux"][1, 0] = 5.0e4                      # one UAV far away: whole environment 1 takes the bypass
    st["ux"][2, :] += 1.0e5                     # a whole swarm far away (relative geometry intact)
    st["tx"][2, :] += 1.0e5
    st["tx"][3, 1], st["ty"][3, 1] = -4.0e4, 9.0e4   # a far target
    st["ux"][5, :] += 3.0e4                     # inside the radius but large magnitude (prefilter still on)
    st["tx"][5, :] += 3.0e4
    env.set_state(cfg, *(st[k] for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    P = oracle_params_from_config(cfg, n, m)
    host = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    for t in range(5):
        a = env.random_actions(3, t).cpu().numpy().copy()
        obs, rew4, cov = env.step_device(cfg, None)
        ref = oracle.step_batch(P, 1, float(cfg["cooperative"]), None, host, a, nthreads=4)
        assert np.array_equal(cov.cpu().numpy(), ref["covered"])
        assert np.array_equal(env.tracker_counts.cpu().numpy(), ref["tracker_cnt"])
        # positions ~1e5: the observation's self part x/dc is ~200, compare with the scaled rule
        assert max_scaled_err(obs.double().cpu().numpy(), ref["obs"]) <= TOL_TIGHT
        assert max_scaled_err(rew4.double().cpu().numpy(), ref["rew4"]) <= TOL_TIGHT
    env.close()


def test_unusual_actions_and_time_steps(oracle):
    """dt * rate beyond a full turn (general fmod path of the heading wrap) and action indices outside
    {0..na-1} (the reference's formula accepts any integer, uav.py:73-81)."""
    from marl_uavs_targets_tracking_b200 import default_config
    n, m = 12, 9
    cfg = default_config("MAAC-G", n, m, uav__dt=37.0, uav__v_max=3.0)
    env = _env(n, m, cfg, 5, track_counts=True, seed=6)
    env.reset(cfg)
    P = oracle_params_from_config(cfg, n, m)
    host = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    rng = np.random.RandomState(0)
    for t in range(6):
        a = rng.randint(-5, 30, size=(5, n)).astype(np.int32)   # mostly outside 0..11
        obs, rew4, cov = env.step_device(cfg, None, torch.as_tensor(a, device="cuda:0"))
        ref = oracle.step_batch(P, 1, float(cfg["cooperative"]), None, host, a, nthreads=2)
        got = env.get_state()
        for k in ("ux", "uy", "uh"):
            assert max_scaled_err(got[k].cpu().numpy(), host[k]) <= 1e-12, k
        assert np.array_equal(got["ua"].cpu().numpy(), host["ua"])
        assert np.array_equal(cov.cpu().numpy(), ref["covered"])
        assert max_scaled_err(obs.double().cpu().numpy(), ref["obs"]) <= TOL_TIGHT
        assert max_scaled_err(rew4.double().cpu().numpy(), ref["rew4"]) <= TOL_TIGHT
    env.close()


@pytest.mark.parametrize("case", range(24))
def test_random_scenarios_match_the_oracle(oracle, case):
    """Scenario constants drawn at random (map size, speeds, time step, ranges incl. dp > dc, action count, reward
    weights, swarm sizes 1..128 with up to 150 targets): the exact squared thresholds, the prefilter guard bands and the run-time-size kernel
    are exercised away from the shipped YAML values."""
    from marl_uavs_targets_tracking_b200 import PMINetwork, default_config
    rng = np.random.RandomState(1000 + case)
    n, m = int(rng.randint(1, 71)), int(rng.randint(1, 71))
    if case >= 18:  # the two shape-specialised kernel instances, away from the constants they were tuned on
        n, m = ((10, 10), (64, 64))[case % 2]
    elif case >= 12:  # up to UAVSIM_MAX_UAV agents (four 32-partner chunks), more targets than threads
        n, m = int(rng.randint(65, 129)), int(rng.randint(1, 151))
    method = ("MAAC", "MAAC-G", "MAAC-R")[case % 3]
    cfg = default_config(method, n, m)
    side = float(rng.choice([300.0, 2000.0, 9000.0]))
    cfg["environment"].update(x_max=side, y_max=side * float(rng.uniform(0.5, 1.5)), na=int(rng.randint(2, 17)))
    cfg["uav"].update(v_max=float(rng.uniform(1, 60)), dt=float(rng.choice([0.25, 1.0, 2.0])), h_max=float(rng.uniform(2, 12)),
                      dc=float(rng.uniform(0.05, 0.6) * side), dp=float(rng.uniform(0.02, 0.7) * side),
                      alpha=float(rng.uniform(0, 1)), beta=float(rng.uniform(0, 1)), gamma=float(rng.uniform(0, 1)))
    cfg["target"].update(v_max=float(rng.uniform(0.5, 30)))
    cfg["cooperative"] = float(rng.uniform(0.05, 0.9)) if method != "MAAC" else 0.0
    pmi = None
    if method == "MAAC-R":
        torch.manual_seed(case)
        pmi = PMINetwork(hidden_dim=(32, 64, 128, 256)[(case // 3) % 4]).eval()  # every PMI kernel instance
    E, T = 37, 25
    e = cfg["environment"]
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment
    env = BatchedEnvironment(n, m, e["x_max"], e["y_max"], e["na"], n_envs=E, device="cuda:0", track_counts=True, seed=case)
    env.reset(cfg)
    P = oracle_params_from_config(cfg, n, m)
    opmi = oracle_pmi_from_module(pmi) if pmi is not None else None
    st = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    wo = wr = 0.0
    for t in range(T):
        a = env.random_actions(5, t).cpu().numpy().copy()
        obs, rew4, cov = env.step_device(cfg, pmi)
        ref = oracle.step_batch(P, case % 3, float(cfg["cooperative"]), opmi, st, a, nthreads=8)
        assert np.array_equal(cov.cpu().numpy(), ref["covered"]), (case, t)
        assert np.array_equal(env.tracker_counts.cpu().numpy(), ref["tracker_cnt"]), (case, t)
        wo = max(wo, max_scaled_err(obs.double().cpu().numpy(), ref["obs"]))
        wr = max(wr, max_scaled_err(rew4.double().cpu().numpy(), ref["rew4"]))
    print("case", case, n, m, method, "obs %.1e rew %.1e" % (wo, wr))
    assert wo <= TOL_TIGHT and wr <= (TOL_PMI if method == "MAAC-R" else TOL_TIGHT)
    if case % 3 == 1:
        # the mask-recording instance of the kernel gives the same outputs bit for bit, and its masks agree with the
        # counts and blocks the plain instance reports (internal consistency; the masks themselves are pinned by the
        # reference fixtures in test_cuda_matches_reference_golden)
        em = BatchedEnvironment(n, m, e["x_max"], e["y_max"], e["na"], n_envs=E, device="cuda:0", track_counts=True,
                                record_masks=True, seed=case)
        e2 = BatchedEnvironment(n, m, e["x_max"], e["y_max"], e["na"], n_envs=E, device="cuda:0", track_counts=True, seed=case)
        em.reset(cfg)
        e2.reset(cfg)
        for t in range(6):
            em.random_actions(5, t)
            e2.random_actions(5, t)
            o1, r1, c1 = em.step_device(cfg, pmi)
            o2, r2, c2 = e2.step_device(cfg, pmi)
            assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(c1, c2)
            mk = em.masks
            assert torch.equal(mk["cover_mask"].sum(1).int(), em.tracker_counts)          # per-target trackers
            assert torch.equal((mk["cover_mask"].sum(1) > 0).sum(1).int(), c1)            # covered targets
            assert torch.equal(mk["nbr_mask"], mk["nbr_mask"].transpose(1, 2))            # new-new distances are symmetric
            assert torch.equal(mk["dup_mask"], mk["dup_mask"].transpose(1, 2))
            assert not bool((mk["cover_mask"] & ~mk["obs_mask"]).any())                   # d < dp implies d <= dp
            no_obs = mk["obs_mask"].sum(2) == 0
            assert bool((o1[..., 5:9][no_obs] == -1).all())                             # empty list -> -1 block
            no_comm = mk["comm_mask"].sum(2) == 0
            assert bool((o1[..., 0:5][no_comm] == -1).all())
        em.close()
        e2.close()
    env.close()


def test_long_episode_64x64_does_not_stall():
    """A full 200-step episode at 64x64 with many environments (UAVs do reach the origin corner)."""
    from marl_uavs_targets_tracking_b200 import default_config
    cfg = default_config("MAAC-G", 64, 64)
    env = _env(64, 64, cfg, 4096, seed=5)
    env.reset(cfg)
    for t in range(200):
        env.random_actions(8, t)
        env.step_device(cfg, None)
    torch.cuda.synchronize()
    s = env.episode_stats()
    assert s["env_steps"] == 4096 * 200
    env.close()


def test_headline_batch_sampled_against_the_oracle(oracle):
    """BASELINE.json configs[3] at full size (64x64, 65 536 environments): 96 environments spread over the batch are
    replayed in the CPU oracle for a whole 200-step episode -- covered / tracker counts bit-exact every step, state,
    observation and rewards within tolerance -- so the full-size launch geometry (persistent grid, counter-scheduled walk over
    environments, last partial wave) is checked against the reference semantics, not only against itself."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 64
    E, T = 65536, 200
    cfg = default_config("MAAC-G", n, m)
    env = _env(n, m, cfg, E, seed=123, track_counts=True)
    env.reset(cfg)
    ids = np.unique(np.concatenate([np.arange(0, E, 701), [E - 1, E - 2, 2367, 2368, 2369]]))[:96]
    idx = torch.as_tensor(ids, device="cuda:0")
    P = oracle_params_from_config(cfg, n, m)
    st = {k: np.ascontiguousarray(v[idx].cpu().numpy()) for k, v in env.get_state().items()}
    worst_o = worst_r = worst_s = 0.0
    for t in range(T):
        a = env.random_actions(31, t)[idx].cpu().numpy().copy()
        obs, rew4, cov = env.step_device(cfg, None)
        ref = oracle.step_batch(P, 1, float(cfg["cooperative"]), None, st, a, nthreads=8)
        assert np.array_equal(cov[idx].cpu().numpy(), ref["covered"]), t
        assert np.array_equal(env.tracker_counts[idx].cpu().numpy(), ref["tracker_cnt"]), t
        worst_o = max(worst_o, max_scaled_err(obs[idx].double().cpu().numpy(), ref["obs"]))
        worst_r = max(worst_r, max_scaled_err(rew4[:, idx].double().cpu().numpy(), ref["rew4"]))
    gs = env.get_state()
    for k in ("ux", "uy", "uh", "tx", "ty", "th"):
        worst_s = max(worst_s, max_scaled_err(gs[k][idx].cpu().numpy(), st[k]))
    assert np.array_equal(gs["ua"][idx].cpu().numpy(), st["ua"])
    print("full-size sample: obs %.1e rewards %.1e state %.1e" % (worst_o, worst_r, worst_s))
    assert worst_o <= 1e-6 and worst_r <= 1e-6 and worst_s <= 1e-11
    env.close()


def test_reset_and_random_policy_match_philox_reference():
    from marl_uavs_targets_tracking_b200 import default_config
    from philox_ref import actions_reference, reset_reference
    cfg = default_config("MAAC", 10, 7)
    env = _env(10, 7, cfg, 33, env_id_offset=1000, seed=5)
    env.reset(cfg, seed=5)
    ep_seed = (5 * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    ref = reset_reference(ep_seed, 33, 10, 7, 12, 2000, 2000, env_id_offset=1000)
    st = env.get_state()
    for k in ("ux", "uy", "uh", "tx", "ty", "th", "ua"):
        assert np.array_equal(st[k].cpu().numpy(), ref[k]), k
    assert st["uh"].abs().max() <= np.pi and st["tx"].min() >= 0 and st["tx"].max() < 2000
    a = env.random_actions(seed=77, step=12).cpu().numpy()
    assert np.array_equal(a, actions_reference(77, 12, 33, 10, 12, env_id_offset=1000))
    # pre-step observation: -1 blocks + (x/dc, y/dc, a/Na)  (src/agent/uav.py:170-190)
    o = env.get_states().cpu().numpy()
    assert np.all(o[..., :9] == -1)
    np.testing.assert_allclose(o[..., 9], ref["ux"] / 500, rtol=1e-6)
    np.testing.assert_allclose(o[..., 11], ref["ua"] / 12, rtol=1e-6)
    env.close()


def test_sharding_is_invisible_in_the_results():
    """Global env ids key the RNG: 2 shards of 8 == 1 handle of 16, bit for bit."""
    from marl_uavs_targets_tracking_b200 import default_config, shard_envs
    cfg = default_config("MAAC-G", 10, 10)
    full = _env(10, 10, cfg, 16, seed=3)
    full.reset(cfg)
    shards = []
    for r in range(2):
        cnt, off = shard_envs(16, r, 2)
        s = _env(10, 10, cfg, cnt, env_id_offset=off, seed=3)
        s.reset(cfg)
        shards.append(s)
    for t in range(25):
        full.random_actions(11, t); full.step_device(cfg, None)
        for s in shards:
            s.random_actions(11, t); s.step_device(cfg, None)
    for k in ("ux", "uy", "uh", "tx", "ty", "th", "ua"):
        cat = torch.cat([s.get_state()[k] for s in shards])
        assert torch.equal(cat, full.get_state()[k]), k
    assert torch.equal(torch.cat([s._rew4 for s in shards], dim=1), full._rew4)
    assert torch.equal(torch.cat([s._obs for s in shards]), full._obs)
    sf = full.episode_stats()
    ss = [s.episode_stats() for s in shards]
    assert sf["env_steps"] == 16 * 25 == sum(s["env_steps"] for s in ss)
    assert sf["covered_sum"] == sum(s["covered_sum"] for s in ss)
    assert sf["covered_max"] == max(s["covered_max"] for s in ss)
    assert abs(sf["rewards"] - sum(s["rewards"] for s in ss)) < 1e-9
    for e in [full] + shards:
        e.close()


def test_queued_host_buffer_steps_equal_device_steps():
    """uavsim_step_host_async / _wait: step t+1 is queued (other host buffers) before the outputs of step t are read;
    every step's outputs must equal the device-resident run's, for changing chunk counts too (64x64: the fast kernel,
    whose launch-wide counter must be back at zero between the chunk launches)."""
    from marl_uavs_targets_tracking_b200 import default_config
    n = m = 64
    cfg = default_config("MAAC-G", n, m)
    E, T = 3000, 9
    a_env, b_env = _env(n, m, cfg, E, seed=12), _env(n, m, cfg, E, seed=12)
    a_env.reset(cfg); b_env.reset(cfg)
    acts, want = [], []
    for t in range(T):
        acts.append(a_env.random_actions(6, t).cpu().pin_memory())
        o, r, c = a_env.step_device(cfg, None)
        want.append((o.cpu(), r.cpu(), c.cpu()))
    bufs = [(torch.empty((E, n, 12), dtype=torch.float32).pin_memory(), torch.empty((4, E, n), dtype=torch.float32).pin_memory(),
             torch.empty((E,), dtype=torch.int32).pin_memory()) for _ in range(2)]
    chunks = lambda t: 4 if t < 6 else 7  # noqa: E731
    tk = b_env.step_host_async(cfg, None, acts[0], *bufs[0], chunks=chunks(0))
    for t in range(1, T):
        tk2 = b_env.step_host_async(cfg, None, acts[t], *bufs[t & 1], chunks=chunks(t))
        b_env.step_host_wait(tk)
        got = bufs[(t - 1) & 1]
        assert torch.equal(got[0], want[t - 1][0]) and torch.equal(got[1], want[t - 1][1]) and torch.equal(got[2], want[t - 1][2]), t
        tk = tk2
    b_env.step_host_wait(tk)
    got = bufs[(T - 1) & 1]
    assert torch.equal(got[0], want[T - 1][0]) and torch.equal(got[1], want[T - 1][1]) and torch.equal(got[2], want[T - 1][2])
    sa, sb = a_env.get_state(), b_env.get_state()
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert a_env.episode_stats() == b_env.episode_stats()
    a_env.close(); b_env.close()


@pytest.mark.parametrize("method,hidden", [("MAAC-G", 0), ("MAAC-R", 64), ("MAAC-R", 128)])
def test_host_buffer_step_equals_device_step(method, hidden):
    """uavsim_step_host pipelines env ranges over streams; hidden = 64 takes the CUDA-core PMI kernel, 128 the tensor
    kernel (env_begin / env_count of a chunk must land on the same rows as the whole-batch launch)."""
    from marl_uavs_targets_tracking_b200 import PMINetwork, default_config
    cfg = default_config(method, 10, 10)
    torch.manual_seed(0)
    pmi = PMINetwork(hidden_dim=hidden).eval() if method == "MAAC-R" else None
    E = 1000
    a_env, b_env = _env(10, 10, cfg, E, seed=8), _env(10, 10, cfg, E, seed=8)
    a_env.reset(cfg); b_env.reset(cfg)
    h_act = torch.empty((E, 10), dtype=torch.int32).pin_memory()
    h_obs = torch.empty((E, 10, 12), dtype=torch.float32).pin_memory()
    h_rew = torch.empty((4, E, 10), dtype=torch.float32).pin_memory()
    h_cov = torch.empty((E,), dtype=torch.int32).pin_memory()
    for t in range(12):
        acts = a_env.random_actions(4, t)
        h_act.copy_(acts.cpu())
        a_env.step_device(cfg, pmi)
        b_env.step_host(cfg, pmi, h_act, h_obs, h_rew, h_cov, chunks=1 + t % 5)
        assert torch.equal(h_obs, a_env._obs.cpu()) and torch.equal(h_rew, a_env._rew4.cpu())
        assert torch.equal(h_cov, a_env._covered.cpu())
    a_env.close(); b_env.close()


def _fx_counts(rew4):
    """The four reward planes as integer counts of 2^-22 (common.cuh: sf_fx), summed per plane."""
    v = rew4.float().cpu().numpy().reshape(4, -1)
    fx = (v + np.float32(3.0)).astype(np.float32).view(np.int32).astype(np.int64) - 0x40400000
    return fx.sum(axis=1)


def _check_episode_stats_equal_output_sums(n, method, hidden, step_path, pmi_path, rollout):
    from marl_uavs_targets_tracking_b200 import PMINetwork, default_config
    cfg = default_config(method, n, n)
    torch.manual_seed(0)
    pmi = PMINetwork(hidden_dim=hidden).eval() if hidden else None
    E, T = (300, 6) if n == 64 else (777, 20)
    env = _env(n, n, cfg, E, seed=2)
    env.set_step_path(step_path)
    env.set_pmi_path(pmi_path)
    env.reset(cfg)
    fx = np.zeros(4, dtype=np.int64)
    cs, cm = 0, 0
    for t in range(T):
        if rollout:
            _, rew4, cov = env.run_random_policy(cfg, pmi, 1, t, 1)
        else:
            env.random_actions(1, t)
            _, rew4, cov = env.step_device(cfg, pmi)
        fx += _fx_counts(rew4)
        cs += int(cov.sum()); cm = max(cm, int(cov.max()))
    s = env.episode_stats()
    got = [s["rewards"], s["target_tracking_reward"], s["boundary_punishment"], s["duplicate_tracking_punishment"]]
    assert got == [float(c) * 2.0 ** -22 for c in fx]
    assert s["covered_sum"] == cs and s["covered_max"] == cm and s["env_steps"] == E * T
    assert s["pmi_rows_out_of_range"] == 0
    env.reset(cfg)
    assert env.episode_stats()["env_steps"] == 0
    env.close()


def test_episode_stats_equal_output_sums():
    """episode_stats() is exactly what the steps wrote: the four reward sums are the integer sums of the float32 outputs
    as counts of 2^-22 (times 2^-22), covered sum / max and env-steps are equal (10x10, automatic kernel choice)."""
    _check_episode_stats_equal_output_sums(10, "MAAC-G", 0, 0, 0, False)


@pytest.mark.parametrize("n,method,hidden,step_path,pmi_path,rollout", [
    pytest.param(64, "MAAC-G", 0, 1, 0, False, id="64x64-generic"),
    pytest.param(64, "MAAC-G", 0, 2, 0, False, id="64x64-fast"),
    pytest.param(64, "MAAC-G", 0, 3, 0, False, id="64x64-tile"),
    pytest.param(10, "MAAC-G", 0, 1, 0, False, id="10x10-generic"),
    pytest.param(10, "MAAC-G", 0, 4, 0, False, id="10x10-small"),
    pytest.param(10, "MAAC-G", 0, 0, 0, True, id="10x10-rollout"),
    pytest.param(10, "MAAC-R", 32, 0, 0, False, id="10x10-pmi-cuda-cores-h32"),
    pytest.param(10, "MAAC-R", 64, 0, 1, False, id="10x10-pmi-cuda-cores-h64"),
    pytest.param(10, "MAAC-R", 128, 0, 0, False, id="10x10-pmi-tensor-h128"),
])
def test_episode_stats_equal_output_sums_on_every_path(n, method, hidden, step_path, pmi_path, rollout):
    """The same exact equality whichever kernel served the steps: every step kernel, the rollout loop below the FFI and
    both PMI kernels keep their statistics in one fixed-point format."""
    _check_episode_stats_equal_output_sums(n, method, hidden, step_path, pmi_path, rollout)


def test_reference_shaped_api_single_env():
    """n_envs == 1: the call pattern of src/train.py:160-192 (operate_epoch) works unchanged."""
    from marl_uavs_targets_tracking_b200 import Environment, default_config
    cfg = default_config("MAAC-G")
    e = cfg["environment"]
    env = Environment(n_uav=e["n_uav"], m_targets=e["m_targets"], x_max=e["x_max"], y_max=e["y_max"], na=e["na"])
    env.reset(config=cfg)
    rng = np.random.RandomState(0)
    ep_ret, covered_list = 0.0, []
    for i in range(15):
        cfg["step"] = i + 1
        action_list = []
        for uav in env.uav_list:
            state = uav.get_local_state()
            assert isinstance(state, np.ndarray) and state.shape == (12,) and state.dtype == np.float64
            action_list.append(int(rng.randint(0, 12)))
        next_state_list, reward_list, covered = env.step(cfg, None, action_list)
        assert isinstance(next_state_list, list) and len(next_state_list) == 10 and next_state_list[0].shape == (12,)
        assert set(reward_list) == {"rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment"}
        assert all(isinstance(v, list) and len(v) == 10 for v in reward_list.values())
        assert isinstance(covered, int)
        ep_ret += sum(reward_list["rewards"])
        covered_list.append(covered)
        np.testing.assert_array_equal(next_state_list[3], env.uav_list[3].get_local_state())
    assert len(env.position["all_uav_xs"]) == 15 and len(env.position["all_uav_xs"][0]) == 10
    assert env.covered_target_num == covered_list
    assert env.uav_list[0].dp == 200 and isinstance(env.uav_list[0].x, float)
    env.close()


def test_device_side_rollout_loop_equals_stepwise_calls():
    """uavsim_run_random_policy (loop below the FFI) == random_actions + step per step, bit for bit, statistics included."""
    from marl_uavs_targets_tracking_b200 import default_config
    cfg = default_config("MAAC-G", 10, 10)
    a, b = _env(10, 10, cfg, 500, seed=9), _env(10, 10, cfg, 500, seed=9)
    a.reset(cfg)
    b.reset(cfg)
    for t in range(37):
        a.random_actions(11, t)
        oa, ra, ca = a.step_device(cfg, None)
    ob, rb, cb = b.run_random_policy(cfg, None, 11, 0, 37)
    assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(ca, cb)
    sa, sb = a.get_state(), b.get_state()
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert a.episode_stats() == b.episode_stats()
    a.close()
    b.close()


def test_trace_files_have_the_reference_layout(tmp_path):
    """Row f-4: `save_position` / `save_covered_num` write what src/environment.py:229-244 writes -- u_xy<k>.csv is the
    (n_uav, steps, 2) array flattened to rows (UAV-major), header `x,y`; covered_target_num<k>.csv one count per step.
    Replays a reference recording so the numbers are the reference's too."""
    from marl_uavs_targets_tracking_b200 import Environment
    g = load_golden("d10_mean_s42")
    cfg = golden_config(g)
    e = cfg["environment"]
    env = Environment(n_uav=e["n_uav"], m_targets=e["m_targets"], x_max=e["x_max"], y_max=e["y_max"], na=e["na"])
    env.reset(config=cfg)
    env.set_state(cfg, *(torch.as_tensor(np.asarray(g[k + "0"])[None]) for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    T = 30
    for t in range(T):
        env.step(cfg, None, [int(a) for a in g["actions"][t]])
    for d in ("u_xy", "t_xy", "covered_target_num"):
        (tmp_path / d).mkdir()
    env.save_position(str(tmp_path), 7)
    env.save_covered_num(str(tmp_path), 7)
    u = np.loadtxt(tmp_path / "u_xy" / "u_xy7.csv", delimiter=",", skiprows=1)
    tt = np.loadtxt(tmp_path / "t_xy" / "t_xy7.csv", delimiter=",", skiprows=1)
    c = np.loadtxt(tmp_path / "covered_target_num" / "covered_target_num7.csv", delimiter=",", skiprows=1)
    assert open(tmp_path / "u_xy" / "u_xy7.csv").readline().strip() == "x,y"
    assert open(tmp_path / "covered_target_num" / "covered_target_num7.csv").readline().strip() == "covered_target_num"
    n, m = e["n_uav"], e["m_targets"]
    ref_u = np.stack([g["ux"][:T], g["uy"][:T]], axis=-1).transpose(1, 0, 2).reshape(-1, 2)   # (n, T, 2) -> rows
    ref_t = np.stack([g["tx"][:T], g["ty"][:T]], axis=-1).transpose(1, 0, 2).reshape(-1, 2)
    assert u.shape == (n * T, 2) and tt.shape == (m * T, 2)
    np.testing.assert_allclose(u, ref_u, rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(tt, ref_t, rtol=1e-12, atol=1e-9)
    assert np.array_equal(c.astype(int), g["covered"][:T])
    env.close()


@pytest.mark.parametrize("n,m,E,method", [(10, 10, 4096, "MAAC"), (64, 64, 65536, "MAAC-G"), (10, 10, 16384, "MAAC-R")])
def test_full_size_properties(n, m, E, method):
    """BASELINE.json sizes, size-independent properties: the second half of the batch is a copy of the
    first half (same state, same actions) and must produce bit-identical results wherever it lands;
    covered == #targets with a tracker; rewards in [-1,1]; terms in their normalised ranges."""
    from marl_uavs_targets_tracking_b200 import PMINetwork, default_config
    cfg = default_config(method, n, m)
    torch.manual_seed(3)
    pmi = PMINetwork(hidden_dim=128).eval() if method == "MAAC-R" else None
    env = _env(n, m, cfg, E, track_counts=True, seed=17)
    env.reset(cfg)
    half = E // 2
    st = env.get_state()
    for k, v in st.items():
        v[half:] = v[:half]
    env.set_state(cfg, *(st[k] for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    for t in range(10):
        a = env.random_actions(5, t)
        a[half:] = a[:half]
        obs, rew4, cov = env.step_device(cfg, pmi)
        assert torch.equal(obs[:half], obs[half:]) and torch.equal(rew4[:, :half], rew4[:, half:])
        assert torch.equal(cov[:half], cov[half:])
        assert torch.equal(cov, (env.tracker_counts > 0).sum(dim=1).to(torch.int32))
        assert float(rew4[0].min()) >= -1 and float(rew4[0].max()) <= 1
        assert float(rew4[1].min()) >= 0 and float(rew4[1].max()) <= 1
        assert float(rew4[2].min()) >= -1 and float(rew4[2].max()) <= 0
        assert float(rew4[3].min()) >= -1 and float(rew4[3].max()) <= 0
        assert torch.isfinite(obs).all()
    for k, v in env.get_state().items():
        assert torch.equal(v[:half], v[half:]), k
    env.close()


def test_errors_are_loud():
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, UavSimError, default_config
    cfg = default_config("MAAC-R", 10, 10)
    with pytest.raises(UavSimError):
        BatchedEnvironment(129, 10, 2000, 2000, 12, n_envs=2).reset(default_config("MAAC", 129, 10))
    env = _env(10, 10, cfg, 4)
    with pytest.raises(UavSimError):
        env.step_device(cfg, None)  # step before reset
    env.reset(cfg)

    class NotAPmi:
        def state_dict(self):
            return {}
    with pytest.raises(Exception):
        env.step_device(cfg, NotAPmi())
    env.close()
