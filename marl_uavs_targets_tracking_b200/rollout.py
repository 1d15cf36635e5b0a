"""Batched rollout on the GPU-resident environment (SURVEY.md section 8f, row f-1).

The reference rolls one environment out with a per-agent, batch-of-one policy forward and an `.item()` sync per
action (src/train.py:160-176, src/models/actor_critic.py:138-148).  Here every step is one `[E*n, 12]` actor
forward, one on-device categorical sample and one `uavsim_step` launch; observations, actions and rewards never
leave HBM.  The learner is stock PyTorch with the reference's architecture and one-step TD actor-critic update
(src/models/actor_critic.py:85-179): it is the consumer of the accelerated path, not part of it.
"""
import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi
from .distributed import episode_summary, reduce_episode_stats
from .replay import PrioritizedReplayBuffer


class PolicyNet(nn.Module):
    """12 -> H -> na softmax policy (FnnPolicyNet, src/models/actor_critic.py:85-99)."""

    def __init__(self, n_states, n_hiddens, n_actions):
        super().__init__()
        self.fc1 = nn.Linear(n_states, n_hiddens)
        self.fc2 = nn.Linear(n_hiddens, n_actions)

    def forward(self, x):
        return F.softmax(self.fc2(F.relu(self.fc1(x))), dim=1)


class ValueNet(nn.Module):
    """12 -> H -> 1 critic (FnnValueNet, src/models/actor_critic.py:102-113)."""

    def __init__(self, n_states, n_hiddens):
        super().__init__()
        self.fc1 = nn.Linear(n_states, n_hiddens)
        self.fc2 = nn.Linear(n_hiddens, 1)

    def forward(self, x):
        return self.fc2(F.relu(self.fc1(x))).squeeze(1)


def policy_weights(policy, state_dim, device=None):
    """The UavSimPolicyWeights of a PolicyNet (or a DDP wrapper around one) and the tensors it points into, which the
    caller keeps alive while the struct is in use.  The kernel reads contiguous float32 on `device` (default: where the
    parameters are): parameters of another dtype, layout or device are converted into fresh tensors (a .double() or
    .half() net would otherwise be read as float32 bit patterns); parameters that already are so are used in place."""
    net = policy.module if hasattr(policy, "module") else policy
    w = _cabi.UavSimPolicyWeights()
    w.state_dim, w.hidden, w.n_actions = state_dim, net.fc1.out_features, net.fc2.out_features
    params = [net.fc1.weight, net.fc1.bias, net.fc2.weight, net.fc2.bias]
    params = [p.detach().to(device=device, dtype=torch.float32).contiguous() for p in params]
    w.w1, w.b1, w.w2, w.b2 = (p.data_ptr() for p in params)
    return w, params


def fused_policy_sample(policy, states, seed, counter, want_probs=False, out=None):
    """One launch of libuavsim's fused policy kernel (`uavsim_policy_sample`, csrc/policy.cuh): softmax(fc2(relu(fc1(x))))
    and one categorical draw per row, uniforms from Philox4x32-10 keyed (seed; row, counter).  `policy` is a PolicyNet
    (or a DDP wrapper around one) on the device of `states` [B,12] float32; `out` = a contiguous int32 [B] tensor to write
    the actions into (e.g. the environment's bound action buffer).  Returns (actions int32 [B], probs or None)."""
    x = states if (states.dtype == torch.float32 and states.is_contiguous()) else states.float().contiguous()
    if x.data_ptr() % 16:  # the kernel reads rows with 16-byte loads: a view off a 16-byte boundary is copied
        x = x.clone()
    dev = x.device
    if dev.type != "cuda":
        raise _cabi.UavSimError("fused_policy_sample needs CUDA tensors (no CPU fallback)")
    w, params = policy_weights(policy, x.shape[1], dev)
    B, A = x.shape[0], w.n_actions
    if out is not None:
        assert out.dtype == torch.int32 and out.is_contiguous() and out.numel() == B and out.device == dev
    actions = out if out is not None else torch.empty(B, dtype=torch.int32, device=dev)
    probs = torch.empty(B, A, dtype=torch.float32, device=dev) if want_probs else None
    lib = _cabi.load()
    with torch.cuda.device(dev):
        _cabi.check(lib.uavsim_policy_sample(C.c_void_p(x.data_ptr()), B, C.byref(w), C.c_uint64(seed), C.c_uint64(counter),
                                             C.c_void_p(actions.data_ptr()),
                                             C.c_void_p(probs.data_ptr()) if probs is not None else None,
                                             dev.index or 0, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
                    "uavsim_policy_sample")
    return actions, probs


class BatchedActorCritic:
    """Same constructor and update rule as the reference `ActorCritic` (src/models/actor_critic.py:116-179), but
    `take_actions` works on all agents of all environments at once and `update` takes device tensors."""

    def __init__(self, state_dim, hidden_dim, action_dim, actor_lr, critic_lr, gamma, device, ddp=False, seed=0,
                 fused=True):
        self.actor = PolicyNet(state_dim, hidden_dim, action_dim).to(device)
        self.critic = ValueNet(state_dim, hidden_dim).to(device)
        if ddp:  # gradient all-reduce over NCCL when several ranks train one policy
            from torch.nn.parallel import DistributedDataParallel as DDP
            self.actor = DDP(self.actor, device_ids=[torch.device(device).index])
            self.critic = DDP(self.critic, device_ids=[torch.device(device).index])
        self.actor_optimizer = torch.optim.Adam(self.actor.parameters(), lr=actor_lr)
        self.critic_optimizer = torch.optim.Adam(self.critic.parameters(), lr=critic_lr)
        self.gamma, self.device = gamma, device
        # rollout policy step: the fused kernel draws from Philox (seed; row, call number); fused=False is the stock
        # torch forward + multinomial, which also serves the sizes the kernel does not (csrc/policy.cuh: 12 inputs,
        # 1..512 hidden units, 2..16 actions)
        self.fused = (bool(fused) and torch.device(device).type == "cuda" and state_dim == 12 and 1 <= hidden_dim <= 512
                      and 2 <= action_dim <= 16)
        # Every rank rolls out its own environments: the draws of rank r must differ from rank 0's (the Philox counter
        # is the LOCAL row), so the rank is folded into the seed.
        import torch.distributed as dist
        rank = dist.get_rank() if (dist.is_available() and dist.is_initialized()) else 0
        self.seed, self._calls = (int(seed) + 0x9E3779B97F4A7C15 * rank) & 0xFFFFFFFFFFFFFFFF, 0

    # ---- checkpoints in the reference's layout (src/models/actor_critic.py:181-200): actor/actor_weights_N.pth and
    #      critic/critic_weights_N.pth, each {'model_state_dict', 'optimizer_state_dict'} with the key names of
    #      FnnPolicyNet / FnnValueNet (a DistributedDataParallel wrapper is looked through, so no 'module.' prefix) ----
    @staticmethod
    def _plain(net):
        return net.module if hasattr(net, "module") else net

    def save(self, save_dir, epoch_i):
        import os
        for sub, net, opt in (("actor", self.actor, self.actor_optimizer), ("critic", self.critic, self.critic_optimizer)):
            os.makedirs(os.path.join(save_dir, sub), exist_ok=True)
            torch.save({"model_state_dict": self._plain(net).state_dict(), "optimizer_state_dict": opt.state_dict()},
                       os.path.join(save_dir, sub, "%s_weights_%s.pth" % (sub, epoch_i)))

    def load(self, actor_path, critic_path):
        import os
        for path, net, opt in ((actor_path, self.actor, self.actor_optimizer), (critic_path, self.critic, self.critic_optimizer)):
            if path and os.path.exists(path):
                checkpoint = torch.load(path, map_location=self.device)
                self._plain(net).load_state_dict(checkpoint["model_state_dict"])
                opt.load_state_dict(checkpoint["optimizer_state_dict"])

    @torch.no_grad()
    def take_actions(self, states, out=None):
        """states [B,12] float -> (actions [B] int32, probs [B,na] or None on the fused path)."""
        if self.fused:
            self._calls += 1
            return fused_policy_sample(self.actor, states, self.seed, self._calls, out=out)
        probs = self.actor(states)
        actions = torch.multinomial(probs, 1).squeeze(1)  # Categorical(probs).sample()
        return actions.to(torch.int32), probs

    def update(self, states, actions, rewards, next_states):
        """One-step TD actor-critic update on [B,...] device tensors (src/models/actor_critic.py:150-179)."""
        with torch.no_grad():  # the reference detaches td_target in both losses (actor_critic.py:171-173)
            td_target = rewards + self.gamma * self.critic(next_states)
        v = self.critic(states)  # evaluated once; the reference's two evaluations give the same value
        td_delta = td_target - v
        log_probs = torch.log(self.actor(states).gather(1, actions.long().view(-1, 1)))
        # The reference multiplies log_probs [B,1] by td_delta [B]: that broadcasts to a [B,B] outer product whose mean
        # is mean(-log_probs) * mean(td_delta) (src/models/actor_critic.py:171).  Same value and gradient, O(B) memory.
        actor_loss = torch.mean(-log_probs) * torch.mean(td_delta.detach())
        critic_loss = F.mse_loss(v, td_target)
        self.actor_optimizer.zero_grad()
        self.critic_optimizer.zero_grad()
        actor_loss.backward()
        critic_loss.backward()
        self.actor_optimizer.step()
        self.critic_optimizer.step()
        return actor_loss.detach(), critic_loss.detach(), td_delta.detach()


def operate_epoch_batched(config, env, agent, pmi, num_steps, keep_transitions=True):
    """One episode for all environments of `env` (the batched form of src/train.py:142-196).

    Returns (transitions, summary): transitions = dict of device tensors states [T*E*n,12], actions [T*E*n],
    rewards [T*E*n], next_states [T*E*n,12] (None if keep_transitions is False); summary = the six scalars the
    reference logs per episode, averaged over every environment of every rank.

    With keep_transitions the observations of the whole episode live in ONE [T+1,E,n,12] tensor: step t writes its
    observations into slot t+1, so `states` and `next_states` are overlapping views of it and no observation is copied;
    the actions of step t go to slot t of an [T,E,n] action trajectory.

    With the fused policy (agent.fused) the whole episode is one library call, `env.run_policy` (uavsim_run_policy):
    the per-step interpreter and FFI time is gone, and the result is bit-identical to driving the steps from Python
    (step t draws with counter agent._calls + 1 + t, as take_actions would).  With keep_transitions it records all four
    reward planes of every step, [T,4,E,n] float32: 12 B per agent-step more than the plane-0 buffer of the per-step
    loop (1.6 GB at 65 536 environments x 10 UAVs x 200 steps).  `rewards` is a copy of plane 0 (4 B per agent-step,
    allocated while the four planes still exist); the four planes are freed on return.  The stock torch policy
    (fused=False) is driven step by step from Python."""
    E, n = env.n_envs, env.n_uav
    dev = env.device
    fused = bool(getattr(agent, "fused", False))
    if fused:
        first_counter = agent._calls + 1
        if keep_transitions:
            traj = torch.empty((num_steps + 1, E, n, 12), dtype=torch.float32, device=dev)
            acts = torch.empty((num_steps, E, n), dtype=torch.int32, device=dev)
            rew4 = torch.empty((num_steps, 4, E, n), dtype=torch.float32, device=dev)
            env.run_policy(config, pmi, agent.actor, agent.seed, first_counter, num_steps, obs=traj, actions=acts,
                           rew4=rew4)
            transitions = {"states": traj[:-1].reshape(num_steps * E * n, 12), "actions": acts.reshape(-1),
                           "rewards": rew4[:, 0].reshape(-1), "next_states": traj[1:].reshape(num_steps * E * n, 12)}
        else:
            env.run_policy(config, pmi, agent.actor, agent.seed, first_counter, num_steps)
            transitions = None
        agent._calls += num_steps
        if num_steps > 0:
            config["step"] = num_steps
    elif keep_transitions:
        home_obs, home_act = env._obs, env.actions
        traj = torch.empty((num_steps + 1, E, n, 12), dtype=torch.float32, device=dev)
        acts = torch.empty((num_steps, E, n), dtype=torch.int32, device=dev)
        rews = torch.empty((num_steps, E * n), dtype=torch.float32, device=dev)
        traj[0].copy_(env._obs)
        try:
            for step in range(num_steps):
                config["step"] = step + 1
                env.bind_obs(traj[step + 1])
                env.bind_actions(acts[step])
                a, _ = agent.take_actions(traj[step].view(E * n, 12))
                acts[step].view(-1).copy_(a)
                _, rew4, _ = env.step_device(config, pmi)
                rews[step].copy_(rew4[0].reshape(E * n))
        finally:
            home_obs.copy_(traj[num_steps])
            env.bind_obs(home_obs)
            env.bind_actions(home_act)
        transitions = {"states": traj[:-1].reshape(num_steps * E * n, 12), "actions": acts.reshape(-1),
                       "rewards": rews.reshape(-1), "next_states": traj[1:].reshape(num_steps * E * n, 12)}
    else:
        for step in range(num_steps):
            config["step"] = step + 1
            a, _ = agent.take_actions(env._obs.view(E * n, 12))
            env.step_device(config, pmi, a.view(E, n))
        transitions = None
    stats = reduce_episode_stats(env.episode_stats(), device=env.device)
    return transitions, episode_summary(stats, n)


def train_batched(config, env, agent, pmi, num_episodes, num_steps, buffer=None, sample_size=None, on_episode=None):
    """The reference's training loop (src/train.py:199-287) on device tensors: per episode reset, roll out every
    environment, push the transitions into the device prioritized replay, draw `sample_size` of them by priority,
    one actor-critic update, write |TD error| back as priorities, and for MAAC-R one `train_pmi` pass on the sampled
    states (the environment picks the new PMI weights up on its next step).

    buffer defaults to a PrioritizedReplayBuffer of config['actor_critic']['buffer_size']; sample_size to
    config['actor_critic']['sample_size'] or, if that is not positive, to one episode of one environment
    (n_uav * num_steps, src/train.py:217-220).  Returns the list of per-episode summaries (plus losses)."""
    ac = config.get("actor_critic", {})
    if buffer is None:
        buffer = PrioritizedReplayBuffer(int(ac.get("buffer_size", 1 << 20)), device=env.device, seed=config.get("seed", 0))
    if sample_size is None:
        sample_size = int(ac.get("sample_size", 0))
    if sample_size <= 0:
        sample_size = env.n_uav * num_steps
    history = []
    for ep in range(num_episodes):
        env.reset(config)
        transitions, summary = operate_epoch_batched(config, env, agent, pmi.eval() if pmi is not None else None, num_steps)
        buffer.add(transitions)
        sample, indices, _ = buffer.sample(sample_size)
        actor_loss, critic_loss, td = agent.update(sample["states"], sample["actions"], sample["rewards"],
                                                   sample["next_states"])
        buffer.update_priorities(indices, td.abs())
        summary.update(actor_loss=float(actor_loss), critic_loss=float(critic_loss))
        if pmi is not None:
            summary["avg_pmi_loss"] = pmi.train_pmi(config, sample["states"], env.n_uav)
        history.append(summary)
        if on_episode is not None:
            on_episode(ep, summary)
    return history
