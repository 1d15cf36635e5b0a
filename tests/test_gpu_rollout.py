"""Row f-1: batched policy rollout + one actor-critic update on the GPU-resident environment."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_batched_rollout_and_update():
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, operate_epoch_batched
    cfg = default_config("MAAC-G", 10, 10)
    E, T = 512, 25
    env = BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=E, device="cuda:0", seed=1)
    env.reset(cfg)
    torch.manual_seed(0)
    agent = BatchedActorCritic(12, 64, 12, 1e-3, 1e-3, 0.95, torch.device("cuda:0"))
    tr, summary = operate_epoch_batched(cfg, env, agent, None, T)
    assert tr["states"].shape == (T * E * 10, 12) and tr["actions"].shape == (T * E * 10,)
    assert tr["actions"].min() >= 0 and tr["actions"].max() < 12
    # transitions chain: next_states of step t are the states of step t+1
    assert torch.equal(tr["next_states"][:E * 10], tr["states"][E * 10:2 * E * 10])
    # the summary equals the mean of the collected rewards (src/train.py:187)
    assert abs(summary["return"] - float(tr["rewards"].double().mean())) < 1e-6
    # the environment's own buffers are bound again and hold the last observation; stepping on works
    assert torch.equal(env.get_states().reshape(-1, 12), tr["next_states"][-E * 10:])
    assert env.get_states().data_ptr() != tr["next_states"].data_ptr()
    env.random_actions(3, 0)
    o_after, _, _ = env.step_device(cfg, None)
    assert o_after.data_ptr() == env.get_states().data_ptr() and not torch.equal(o_after.reshape(-1, 12), tr["next_states"][-E * 10:])
    # states / next_states are overlapping views of one trajectory tensor (no per-step copies)
    assert tr["next_states"].data_ptr() == tr["states"].data_ptr() + E * 10 * 12 * 4
    assert 0 <= summary["average_covered_targets"] <= 10
    before = [p.detach().clone() for p in agent.actor.parameters()]
    a_loss, c_loss, td = agent.update(tr["states"], tr["actions"], tr["rewards"], tr["next_states"])
    assert torch.isfinite(a_loss) and torch.isfinite(c_loss) and td.shape == (T * E * 10,)
    assert any(not torch.equal(b, p) for b, p in zip(before, agent.actor.parameters()))
    env.close()


def test_reference_training_loop_on_the_device():
    """Rows f-1..f-3 together (src/train.py:199-287): rollout -> device PER -> update -> priorities -> train_pmi."""
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, PMINetwork, PrioritizedReplayBuffer, default_config
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, train_batched
    cfg = default_config("MAAC-R", 10, 10)
    cfg.setdefault("pmi", {}).update(batch_size=64)
    E, T = 64, 12
    dev = torch.device("cuda:0")
    env = BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=E, device=dev, seed=2)
    torch.manual_seed(0)
    agent = BatchedActorCritic(12, 64, 12, 1e-3, 1e-3, 0.95, dev)
    pmi = PMINetwork(hidden_dim=128, b2_size=256).to(dev)
    buf = PrioritizedReplayBuffer(10_000, device=dev, seed=5)
    w0 = pmi.fc1.weight.detach().clone()
    hist = train_batched(cfg, env, agent, pmi, 3, T, buffer=buf, sample_size=2048)
    assert len(hist) == 3 and all(k in hist[-1] for k in ("return", "actor_loss", "critic_loss", "avg_pmi_loss"))
    assert buf.size() == 10_000 and buf.pos == (3 * E * 10 * T) % 10_000        # 23 040 transitions through a 10 000 ring
    pri = buf.export()["priorities"]
    assert (pri > 0).all() and pri.unique().numel() > 100                       # |TD| written back
    assert not torch.equal(w0, pmi.fc1.weight.detach())                         # PMI trained
    assert all(abs(h["return"]) <= 1.0 for h in hist)
    env.close()


def test_rollout_paths_agree():
    """keep_transitions on/off and the stock torch policy step drive the same environment dynamics: with the fused
    policy (Philox draws keyed by call number) the two modes visit identical states."""
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, operate_epoch_batched
    cfg = default_config("MAAC-G", 10, 10)
    E, T = 200, 15
    dev = torch.device("cuda:0")
    finals = []
    for keep in (True, False):
        env = BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=E, device=dev, seed=4)
        env.reset(cfg)
        torch.manual_seed(0)
        agent = BatchedActorCritic(12, 64, 12, 1e-3, 1e-3, 0.95, dev, seed=7)
        tr, summary = operate_epoch_batched(cfg, env, agent, None, T, keep_transitions=keep)
        finals.append((env.get_states().clone(), {k: v.clone() for k, v in env.get_state().items()}, summary))
        assert (tr is None) == (not keep)
        env.close()
    assert torch.equal(finals[0][0], finals[1][0])
    assert all(torch.equal(finals[0][1][k], finals[1][1][k]) for k in finals[0][1])
    assert finals[0][2] == finals[1][2]
    # stock torch policy step (multinomial): same structure, valid actions
    env = BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=E, device=dev, seed=4)
    env.reset(cfg)
    agent = BatchedActorCritic(12, 64, 12, 1e-3, 1e-3, 0.95, dev, fused=False)
    tr, _ = operate_epoch_batched(cfg, env, agent, None, T)
    assert tr["actions"].dtype == torch.int32 and 0 <= int(tr["actions"].min()) and int(tr["actions"].max()) < 12
    assert torch.equal(tr["next_states"][:E * 10], tr["states"][E * 10:2 * E * 10])
    env.close()
