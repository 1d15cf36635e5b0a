"""Drop-in proof: the reference's OWN driver code runs against the CUDA environment.

`baseline/_ref/src` is an unmodified copy of the reference (made by __graft_entry__.build(); tests skip without it).
`src/train.py:operate_epoch` (lines 142-196) -- the rollout loop of `python main.py` -- is imported as is and given

    env   = marl_uavs_targets_tracking_b200.Environment   (n_envs = 1: the reference's shapes)
    agent = the reference's ActorCritic                    (src/models/actor_critic.py:114-148)
    pmi   = the reference's PMINetwork for MAAC-R          (src/models/PMINet.py:20-72)

for all three methods with the shipped YAML files.  The recorded transitions are then replayed step by step in the
reference's own `Environment` (same initial state, same actions): next states, the four reward lists and the covered
count must agree within the contract (1e-5; integer count exact), so the numbers the learner saw are the reference's.

Without that copy, the same comparison runs against episodes recorded from the reference's own `Environment.step`
(tests/golden/d10_*.npz, made by tests/golden/make_golden.py): the single-environment drop-in replays them through the
reference-shaped API and must reproduce every step.
"""
import random

import numpy as np
import pytest
import torch

from conftest import load_golden
from gpu_util import STATE, golden_config, golden_pmi_module, max_scaled_err

pytestmark = pytest.mark.gpu

TOL = 1e-5
REWARDS = (("rewards", "rewards"), ("target_tracking_reward", "tt"), ("boundary_punishment", "bp"),
           ("duplicate_tracking_punishment", "dup"))


def _reference():
    import baseline
    if not baseline.available():
        pytest.skip("baseline/_ref/src absent (build() copies it from $UAVSIM_REFERENCE_SRC)")
    return baseline, baseline.import_reference()


@pytest.mark.parametrize("method", ["MAAC", "MAAC-G", "MAAC-R"])
def test_reference_operate_epoch_drives_the_cuda_environment(method):
    baseline, ref = _reference()
    from marl_uavs_targets_tracking_b200 import Environment
    cfg = baseline.load_yaml_config(method)
    cfg["devices"] = [torch.device("cuda:0")]
    e, ac = cfg["environment"], cfg["actor_critic"]
    n, m, T = e["n_uav"], e["m_targets"], 25
    random.seed(3); np.random.seed(3); torch.manual_seed(3)

    env = Environment(n_uav=n, m_targets=m, x_max=e["x_max"], y_max=e["y_max"], na=e["na"])   # src/main.py:55-59
    agent = ref.ActorCritic(state_dim=12, hidden_dim=ac["hidden_dim"], action_dim=e["na"], actor_lr=float(ac["actor_lr"]),
                            critic_lr=float(ac["critic_lr"]), gamma=float(ac["gamma"]), device=cfg["devices"][0])
    pmi = None
    if method == "MAAC-R":
        pmi = ref.PMINetwork(hidden_dim=cfg["pmi"]["hidden_dim"], b2_size=cfg["pmi"]["b2_size"])
        with torch.no_grad():  # BatchNorm statistics away from the identity, so folding is exercised
            for bn in (pmi.bn_comm, pmi.bn_obs, pmi.bn_boundary_state, pmi.bn1):
                bn.running_mean.normal_(0, 0.3)
                bn.running_var.uniform_(0.5, 1.5)

    env.reset(cfg)                                                                              # src/train.py:232
    st0 = {k: v.cpu().numpy().copy()[0] for k, v in env.get_state().items()}
    out = ref.train.operate_epoch(cfg, env, agent, pmi, T)                                      # src/train.py:238
    tr, ret, tt_ret, bp_ret, dup_ret, avg_cov, max_cov = out

    # shapes and types the reference's learner consumes (src/train.py:250-262, actor_critic.py:150-179)
    assert len(tr["states"]) == len(tr["actions"]) == len(tr["next_states"]) == len(tr["rewards"]) == T * n
    assert all(isinstance(s, np.ndarray) and s.shape == (12,) and s.dtype == np.float64 for s in tr["states"])
    assert all(isinstance(a, int) for a in tr["actions"])
    assert cfg["step"] == T
    a_loss, c_loss, td = agent.update(tr)                                                       # src/train.py:255
    assert torch.isfinite(a_loss) and torch.isfinite(c_loss) and td.shape[0] == T * n
    assert len(env.covered_target_num) == T and len(env.position["all_uav_xs"]) == T            # traces for main.py

    # replay in the reference's own environment
    renv = ref.environment.Environment(n_uav=n, m_targets=m, x_max=e["x_max"], y_max=e["y_max"], na=e["na"])
    renv.reset(cfg)
    for i, u in enumerate(renv.uav_list):
        u.x, u.y, u.h, u.a = float(st0["ux"][i]), float(st0["uy"][i]), float(st0["uh"][i]), int(st0["ua"][i])
    for j, t in enumerate(renv.target_list):
        t.x, t.y, t.h = float(st0["tx"][j]), float(st0["ty"][j]), float(st0["th"][j])
    acts = np.asarray(tr["actions"]).reshape(T, n)
    sums = np.zeros(4)
    covs = []
    worst = 0.0
    first = np.stack([u.get_local_state() for u in renv.uav_list])
    assert max_scaled_err(np.stack(tr["states"][:n]), first) <= TOL
    for t in range(T):
        ns, rew, cov = renv.step(cfg, pmi, [int(a) for a in acts[t]])
        got_ns = np.stack(tr["next_states"][t * n:(t + 1) * n])
        worst = max(worst, max_scaled_err(got_ns, np.stack(ns)))
        worst = max(worst, max_scaled_err(np.asarray(tr["rewards"][t * n:(t + 1) * n]), np.asarray(rew["rewards"])))
        if t + 1 < T:  # the states the policy saw at the next step are these next states
            assert np.array_equal(np.stack(tr["states"][(t + 1) * n:(t + 2) * n]), got_ns)
        assert env.covered_target_num[t] == cov, (t, "covered")
        covs.append(cov)
        for q, k in enumerate(("rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment")):
            sums[q] += sum(rew[k])
    print(method, "worst %.1e" % worst)
    assert worst <= TOL
    ref_returns = sums / (T * n)
    assert np.allclose([ret, tt_ret, bp_ret, dup_ret], ref_returns, rtol=0, atol=TOL)
    assert avg_cov == pytest.approx(np.mean(covs)) and max_cov == np.max(covs)
    env.close()


@pytest.mark.parametrize("seed", [42, 7])
@pytest.mark.parametrize("method", ["MAAC", "MAAC-G", "MAAC-R"])
def test_reference_shaped_environment_replays_the_reference_recordings(method, seed):
    """The single-environment drop-in, built and configured the way src/main.py does it with the shipped YAML values,
    replays a 200-step episode recorded from the reference's own `Environment.step` (same initial state, same actions,
    for MAAC-R the recorded PMINetwork state_dict).  Next states, the four reward lists, the covered count, the
    `uav_list` views, the position / coverage traces and the returns operate_epoch reports must be the reference's."""
    from marl_uavs_targets_tracking_b200 import Environment, default_config
    g = load_golden("d10_%s_s%d" % ({"MAAC": "self", "MAAC-G": "mean", "MAAC-R": "pmi"}[method], seed))
    cfg = default_config(method)
    rec = golden_config(g)
    assert all(cfg[k] == rec[k] for k in ("cooperative", "environment", "uav", "target"))  # the recorded scenario
    e = cfg["environment"]
    n, T = e["n_uav"], int(g["params_i"][3])
    pmi = golden_pmi_module(g) if method == "MAAC-R" else None

    env = Environment(n_uav=n, m_targets=e["m_targets"], x_max=e["x_max"], y_max=e["y_max"], na=e["na"])
    env.reset(cfg)
    env.set_state(cfg, *(np.asarray(g[k + "0"])[None] for k in STATE))
    assert max_scaled_err(np.stack([u.get_local_state() for u in env.uav_list]), g["obs0"]) <= TOL
    worst, pos = 0.0, 0.0
    sums, ref_sums = np.zeros(4), np.zeros(4)
    for t in range(T):
        ns, rew, cov = env.step(cfg, pmi, [int(a) for a in g["actions"][t]])
        assert isinstance(ns, list) and len(ns) == n and all(s.shape == (12,) and s.dtype == np.float64 for s in ns)
        assert isinstance(cov, int) and cov == int(g["covered"][t]), (t, "covered")
        worst = max(worst, max_scaled_err(np.stack(ns), g["obs"][t]))
        for q, (key, gk) in enumerate(REWARDS):
            assert len(rew[key]) == n
            worst = max(worst, max_scaled_err(np.asarray(rew[key]), g[gk][t]))
            sums[q] += sum(rew[key])
            ref_sums[q] += g[gk][t].sum()
        np.testing.assert_array_equal(np.stack(ns), np.stack([u.get_local_state() for u in env.uav_list]))
        for attr, gk in (("x", "ux"), ("y", "uy"), ("h", "uh")):
            pos = max(pos, max_scaled_err([getattr(u, attr) for u in env.uav_list], g[gk][t]))
        assert [u.a for u in env.uav_list] == [int(a) for a in g["actions"][t]]
    print(method, seed, "worst %.1e, positions %.1e" % (worst, pos))
    assert worst <= TOL and pos <= 1e-9
    assert env.covered_target_num == [int(c) for c in g["covered"]]
    for key, gk in (("all_uav_xs", "ux"), ("all_uav_ys", "uy"), ("all_target_xs", "tx"), ("all_target_ys", "ty")):
        assert max_scaled_err(np.asarray(env.position[key]), g[gk]) <= 1e-9, key
    assert np.allclose(sums / (T * n), ref_sums / (T * n), rtol=0, atol=TOL)
    env.close()
