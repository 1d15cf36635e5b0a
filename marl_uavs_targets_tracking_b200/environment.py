"""Batched drop-in for the reference `Environment` (src/environment.py:12-253).

Same constructor, `reset(config)`, `get_states()`, `step(config, pmi, actions)`, `uav_list`,
`target_list`, `position`, `covered_target_num`, `save_position`, `save_covered_num` -- but the state
of `n_envs` independent environments lives in HBM as structure-of-arrays torch tensors and every step
is one launch of the fused sm_100a kernel in libuavsim.so (through the C ABI, include/uavsim.h).

With `n_envs == 1` the return values have the reference's Python shapes (lists of ndarray(12), dict of
lists, int) so src/train.py:operate_epoch and src/main.py run unchanged.  With `n_envs > 1` the same
calls return CUDA tensors: obs [E,n,12] f32, the four reward planes [E,n] f32, covered [E] i32.

There is no CPU implementation: constructing the environment needs a CUDA device and the built library.
"""
import contextlib
import ctypes as C
import os
from math import pi

import numpy as np
import torch

from . import _cabi
from ._cabi import (MODE_MEAN, MODE_PMI, MODE_SELF, UavSimBuffers, UavSimError, UavSimParams, UavSimPmiWeights,
                    UavSimTrajectory)
from .pmi import fold_pmi, pmi_version
from .rollout import policy_weights

_REWARD_KEYS = ("rewards", "target_tracking_reward", "boundary_punishment", "duplicate_tracking_punishment")


def params_from_config(config, n_uav, m_targets, x_max, y_max, na, num_steps=0):
    """The config keys Environment.reset / step read (src/environment.py:97-107, :207-224)."""
    p = UavSimParams()
    p.n_uav, p.m_targets, p.na, p.num_steps = int(n_uav), int(m_targets), int(na), int(num_steps)
    p.x_max, p.y_max = float(x_max), float(y_max)
    u, t = config["uav"], config["target"]
    p.dt, p.uav_v_max, p.uav_h_max = float(u["dt"]), float(u["v_max"]), pi / float(u["h_max"])
    p.dc, p.dp = float(u["dc"]), float(u["dp"])
    p.tgt_v_max, p.tgt_h_max = float(t["v_max"]), pi / float(t["h_max"])
    p.alpha, p.beta, p.gamma = float(u.get("alpha", 0.6)), float(u.get("beta", 0.2)), float(u.get("gamma", 0.2))
    return p


class _UavView:
    """`env.uav_list[i]` for environment 0: the attributes src/train.py:165-166 and
    src/utils/draw_util.py:33,78 read."""

    def __init__(self, env, i):
        self._env, self._i = env, i

    def get_local_state(self):
        return self._env._host0()["obs"][self._i].copy()

    # every attribute reads the per-step host snapshot of environment 0 (one device->host copy per step, not one
    # synchronisation per attribute)
    x = property(lambda s: float(s._env._host0()["ux"][s._i]))
    y = property(lambda s: float(s._env._host0()["uy"][s._i]))
    h = property(lambda s: float(s._env._host0()["uh"][s._i]))
    a = property(lambda s: int(s._env._host0()["ua"][s._i]))
    dp = property(lambda s: s._env._params.dp)
    dc = property(lambda s: s._env._params.dc)
    reward = property(lambda s: float(s._env._host0()["rew"][0, s._i]))


class _TargetView:
    def __init__(self, env, j):
        self._env, self._j = env, j

    x = property(lambda s: float(s._env._host0()["tx"][s._j]))
    y = property(lambda s: float(s._env._host0()["ty"][s._j]))
    h = property(lambda s: float(s._env._host0()["th"][s._j]))


class BatchedEnvironment:
    def __init__(self, n_uav, m_targets, x_max, y_max, na, n_envs=1, device=None, env_id_offset=0, seed=0,
                 num_steps=0, record_masks=False, track_counts=False, trace=None):
        """First five arguments as the reference (src/environment.py:13); the rest are batch options:
        n_envs environments on `device`, global id of env 0 (`env_id_offset`, for rank sharding),
        Philox `seed`, episode length for the done flag, optional integer mask / per-target counts
        outputs, and whether to keep the env-0 position trace (default: only when n_envs == 1)."""
        self.x_max, self.y_max = x_max, y_max
        self.state_dim = (4 + 1) + 4 + (2 + 1)
        self.action_dim = na
        self.n_uav, self.m_targets = int(n_uav), int(m_targets)
        self.n_envs, self.env_id_offset = int(n_envs), int(env_id_offset)
        self.seed, self.num_steps = int(seed), int(num_steps)
        self.record_masks, self.track_counts = bool(record_masks), bool(track_counts)
        self.trace = (self.n_envs == 1) if trace is None else bool(trace)
        self._lib = _cabi.load()  # raises if libuavsim.so is not built
        if not torch.cuda.is_available():
            raise UavSimError("BatchedEnvironment needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._h = None
        self._host = None
        self._params = None
        self._episode = 0
        self._pmi_key = None
        self.uav_list = [_UavView(self, i) for i in range(self.n_uav)]
        self.target_list = [_TargetView(self, j) for j in range(self.m_targets)]
        self.position = {"all_uav_xs": [], "all_uav_ys": [], "all_target_xs": [], "all_target_ys": []}
        self.covered_target_num = []
        self._alloc()

    # ------------------------------------------------------------------ buffers
    def _alloc(self):
        E, n, m, dev = self.n_envs, self.n_uav, self.m_targets, self.device
        f64, i32, f32 = torch.float64, torch.int32, torch.float32
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        self._ux, self._uy, self._uh, self._ua = z((E, n), f64), z((E, n), f64), z((E, n), f64), z((E, n), i32)
        self._tx, self._ty, self._th = z((E, m), f64), z((E, m), f64), z((E, m), f64)
        self._actions = z((E, n), i32)
        self._obs, self._rew4, self._covered = z((E, n, 12), f32), z((4, E, n), f32), z((E,), i32)
        self._tracker = z((E, m), i32) if self.track_counts else None
        self._done = z((E,), i32)
        self._raw, self._nbr_bits = None, None
        self._masks = None
        if self.record_masks:
            u8 = torch.uint8
            self._masks = {"obs_mask": z((E, n, m), u8), "comm_mask": z((E, n, n), u8), "nbr_mask": z((E, n, n), u8),
                           "dup_mask": z((E, n, n), u8), "cover_mask": z((E, n, m), u8)}

    def _ensure_pmi_scratch(self):
        if self._raw is None:
            E, n = self.n_envs, self.n_uav
            self._raw = torch.zeros((E, n), dtype=torch.float64, device=self.device)
            self._nbr_bits = torch.zeros((E, n, 2), dtype=torch.int64, device=self.device)
            self._bind()

    def _bind(self):
        b = UavSimBuffers()
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        b.ux, b.uy, b.uh, b.ua = ptr(self._ux), ptr(self._uy), ptr(self._uh), ptr(self._ua)
        b.tx, b.ty, b.th = ptr(self._tx), ptr(self._ty), ptr(self._th)
        b.actions, b.obs, b.rew4, b.covered = ptr(self._actions), ptr(self._obs), ptr(self._rew4), ptr(self._covered)
        b.tracker_cnt, b.done, b.raw, b.nbr_bits = ptr(self._tracker), ptr(self._done), ptr(self._raw), ptr(self._nbr_bits)
        if self._masks:
            for k, t in self._masks.items():
                setattr(b, k, t.data_ptr())
        _cabi.check(self._lib.uavsim_bind(self._h, C.byref(b)), "uavsim_bind")
        self._bufs = b   # kept: bind_actions only swaps one pointer

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _on_device(self):
        """Context that makes this environment's GPU current.  Entering torch.cuda.device costs several microseconds --
        more than a small step kernel takes to queue -- so it is skipped when the device is current already."""
        if torch.cuda.current_device() == self.device.index:
            return contextlib.nullcontext()
        return torch.cuda.device(self.device)

    def _ensure_handle(self, config):
        p = params_from_config(config, self.n_uav, self.m_targets, self.x_max, self.y_max, self.action_dim,
                               self.num_steps)
        if "environment" in config:
            ce = config["environment"]
            if int(ce.get("n_uav", self.n_uav)) != self.n_uav or int(ce.get("m_targets", self.m_targets)) != self.m_targets:
                raise UavSimError("config n_uav/m_targets differ from the constructor's")
        key = bytes(p)
        if self._h is not None and key == self._params_key:
            return
        if self._h is not None:
            self._lib.uavsim_destroy(self._h)
            self._h = None
        h = C.c_void_p()
        _cabi.check(self._lib.uavsim_create(C.byref(p), self.n_envs, self.env_id_offset, self.device.index, C.byref(h)),
                    "uavsim_create")
        self._h, self._params, self._params_key = h, p, key
        self._pmi_key = None
        self._bind()
        if getattr(self, "_step_path", 0):
            _cabi.check(self._lib.uavsim_set_step_path(self._h, self._step_path), "uavsim_set_step_path")

    # ------------------------------------------------------------------ reference API
    def reset(self, config, seed=None):
        """Environment.reset (src/environment.py:87-107).  Draws come from the counter-based RNG keyed
        (seed, episode, global env id), so every episode and every environment differs but a run is
        reproducible for any number of GPUs."""
        self._ensure_handle(config)
        with self._on_device():
            _cabi.check(self._lib.uavsim_reset(self._h, C.c_uint64(self._episode_seed(seed, self._episode)),
                                               self._stream()), "uavsim_reset")
        self._episode += 1
        self._clear_traces()

    def _episode_seed(self, seed, episode):
        s = self.seed if seed is None else int(seed)
        return (s * 0x9E3779B97F4A7C15 + episode * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF

    def set_state(self, config, ux, uy, uh, ua, tx, ty, th):
        """Replay path: load a recorded reset (e.g. the reference's `random`-module draws) for all envs."""
        self._ensure_handle(config)
        for dst, src in ((self._ux, ux), (self._uy, uy), (self._uh, uh), (self._ua, ua), (self._tx, tx),
                         (self._ty, ty), (self._th, th)):
            dst.copy_(torch.as_tensor(np.asarray(src) if not torch.is_tensor(src) else src).reshape(dst.shape).to(dst.dtype))
        with self._on_device():
            _cabi.check(self._lib.uavsim_begin_episode(self._h, self._stream()), "uavsim_begin_episode")
        self._clear_traces()

    def get_state(self):
        return {"ux": self._ux, "uy": self._uy, "uh": self._uh, "ua": self._ua, "tx": self._tx, "ty": self._ty,
                "th": self._th}

    def _host0(self):
        """Host snapshot of environment 0 (observations, rewards, state, covered count), fetched with ONE packed
        device->host copy and kept until the next step / reset / set_state.  The reference-shaped API (n_envs == 1,
        `uav_list[i].get_local_state()`, traces) reads it instead of synchronising once per value."""
        if self._host is None:
            n, m = self.n_uav, self.m_targets
            parts = [self._obs[0].reshape(-1).double(), self._rew4[:, 0, :].reshape(-1).double(), self._ux[0], self._uy[0],
                     self._uh[0], self._ua[0].double(), self._tx[0], self._ty[0], self._th[0], self._covered[:1].double()]
            flat = torch.cat(parts).cpu().numpy()
            o = 0

            def take(k):
                nonlocal o
                v = flat[o:o + k]
                o += k
                return v
            self._host = {"obs": take(n * 12).reshape(n, 12), "rew": take(4 * n).reshape(4, n), "ux": take(n), "uy": take(n),
                          "uh": take(n), "ua": take(n).astype(np.int64), "tx": take(m), "ty": take(m), "th": take(m),
                          "covered": int(take(1)[0])}
        return self._host

    def _clear_traces(self):
        self._host = None
        self.position = {"all_uav_xs": [], "all_uav_ys": [], "all_target_xs": [], "all_target_ys": []}
        self.covered_target_num = []

    def get_states(self):
        """Environment.get_states (src/environment.py:109-118)."""
        if self.n_envs == 1:
            o = self._host0()["obs"]
            return [o[i].copy() for i in range(self.n_uav)]
        return self._obs

    def _mode(self, config, pmi):
        coop = float(config.get("cooperative", 0) or 0)
        if pmi is None:
            return (MODE_MEAN if coop != 0 else MODE_SELF), coop
        if coop != 0:
            key = pmi_version(pmi)
            if key != self._pmi_key:
                self.set_pmi(pmi)
                self._pmi_key = key
        return MODE_PMI, coop

    def set_pmi(self, pmi):
        """Upload BN-folded PMI weights (uavsim_set_pmi_weights)."""
        f = fold_pmi(pmi)
        w = UavSimPmiWeights()
        w.hidden = f["hidden"]
        w.w0, w.b0, w.w1, w.b1, w.w2 = (f[k].ctypes.data for k in ("w0", "b0", "w1", "b1", "w2"))
        w.b2 = f["b2"]
        self._ensure_pmi_scratch()
        with self._on_device():
            _cabi.check(self._lib.uavsim_set_pmi_weights(self._h, C.byref(w), self._stream()), "uavsim_set_pmi_weights")
        if getattr(self, "_pmi_path", 0):
            _cabi.check(self._lib.uavsim_set_pmi_path(self._h, self._pmi_path), "uavsim_set_pmi_path")

    def set_pmi_path(self, path):
        """0 = automatic, 1 = fp32 CUDA cores, 2 = tcgen05 tensor cores (split fp16 operands; hidden 64 or 128)."""
        self._pmi_path = int(path)
        if self._h is not None:
            _cabi.check(self._lib.uavsim_set_pmi_path(self._h, self._pmi_path), "uavsim_set_pmi_path")

    def set_step_path(self, path):
        """0 = automatic, 1 = generic step kernel, 2 = per-UAV fast 64 x 64 kernel, 3 = all-pairs tile 64 x 64 kernel
        (uavsim_set_step_path)."""
        self._step_path = int(path)
        if self._h is not None:
            _cabi.check(self._lib.uavsim_set_step_path(self._h, self._step_path), "uavsim_set_step_path")

    def _sync_weights(self, config):
        u = config.get("uav", {})
        a, b, g = float(u.get("alpha", self._params.alpha)), float(u.get("beta", self._params.beta)), float(u.get("gamma", self._params.gamma))
        if (a, b, g) != (self._params.alpha, self._params.beta, self._params.gamma):
            self._params.alpha, self._params.beta, self._params.gamma = a, b, g
            _cabi.check(self._lib.uavsim_set_reward_weights(self._h, a, b, g), "uavsim_set_reward_weights")

    def step_device(self, config, pmi, actions=None):
        """One step for all environments, everything stays on the GPU.  `actions`: int tensor [E,n] on
        the device (or None to keep what is in the bound action buffer, e.g. after random_actions)."""
        if self._h is None:
            raise UavSimError("step before reset")
        self._sync_weights(config)
        mode, coop = self._mode(config, pmi)
        if actions is not None:
            self._actions.copy_(actions.reshape(self._actions.shape), non_blocking=True)
        with self._on_device():
            _cabi.check(self._lib.uavsim_step(self._h, mode, coop, self._stream()), "uavsim_step")
        self._host = None
        return self._obs, self._rew4, self._covered

    def run_random_policy(self, config, pmi, seed, first_step, nsteps):
        """`nsteps` random-policy steps queued from C without returning to Python in between
        (uavsim_run_random_policy): actions of step k are Philox(seed; agent, env, first_step + k), exactly what
        `random_actions(seed, first_step + k)` followed by `step_device` gives.  Returns the last step's outputs."""
        if self._h is None:
            raise UavSimError("step before reset")
        self._sync_weights(config)
        mode, coop = self._mode(config, pmi)
        with self._on_device():
            _cabi.check(self._lib.uavsim_run_random_policy(self._h, mode, coop, C.c_uint64(seed), int(first_step),
                                                           int(nsteps), self._stream()), "uavsim_run_random_policy")
        self._host = None
        return self._obs, self._rew4, self._covered

    def run_policy(self, config, pmi, policy, seed, first_counter, nsteps, obs=None, actions=None, rew4=None,
                   covered=None):
        """`nsteps` steps of a learned policy queued from C without returning to Python in between
        (uavsim_run_policy).  `policy` is a PolicyNet (or a DDP wrapper around one) on this device; step k draws its
        actions with the fused policy kernel, counter `first_counter + k`, exactly what `fused_policy_sample(policy,
        states, seed, first_counter + k, out=actions)` followed by `step_device` gives -- bit for bit, in every output.

        Optional trajectory tensors (contiguous, on this device), T = nsteps: obs float32 [T+1,E,n,12] (slot 0 <- the
        current observation, slot k+1 <- step k), actions int32 [T,E,n], rew4 float32 [T,4,E,n], covered int32 [T,E].
        A field left None goes to the bound buffer.  Afterwards the bound buffers hold the last step's values, as after
        stepping one step at a time.  Returns the bound (obs, rew4, covered)."""
        if self._h is None:
            raise UavSimError("step before reset")
        E, n, T = self.n_envs, self.n_uav, int(nsteps)
        traj = UavSimTrajectory()
        for name, t, dtype, shape in (("obs", obs, torch.float32, (T + 1, E, n, 12)),
                                      ("actions", actions, torch.int32, (T, E, n)),
                                      ("rew4", rew4, torch.float32, (T, 4, E, n)),
                                      ("covered", covered, torch.int32, (T, E))):
            if t is None:
                continue
            if t.dtype != dtype or tuple(t.shape) != shape or not t.is_contiguous() or t.device != self.device:
                raise ValueError("run_policy: %s must be a contiguous %s tensor of shape %s on %s (got %s %s on %s)"
                                 % (name, dtype, shape, self.device, t.dtype, tuple(t.shape), t.device))
            setattr(traj, name, t.data_ptr())
        w, params = policy_weights(policy, self.state_dim, self.device)  # (params: kept alive over the call)
        self._sync_weights(config)
        mode, coop = self._mode(config, pmi)
        with self._on_device():
            _cabi.check(self._lib.uavsim_run_policy(self._h, mode, coop, C.byref(w), C.c_uint64(seed),
                                                    C.c_uint64(first_counter), T, C.byref(traj), self._stream()),
                        "uavsim_run_policy")
        self._host = None
        return self._obs, self._rew4, self._covered

    def evaluate_policy(self, config, pmi, policy, n_episodes, nsteps, greedy=False, seed=None, first_counter=1,
                        policy_seed=0):
        """`n_episodes` evaluation episodes of `nsteps` steps in one library call (uavsim_evaluate_policy), equal bit for
        bit to

            for k in range(n_episodes):
                env.reset(config, seed)
                env.run_policy(config, pmi, policy, policy_seed, first_counter + k * nsteps, nsteps)

        in the state, the bound buffers and episode_stats() (the last episode's); with greedy, every step takes the most
        probable action (`fused_policy_greedy`) instead of a draw.  Episode k's reset seed is derived from `seed`
        (default: the constructor's) exactly as reset() derives it, and the episode count advances by n_episodes.

        Returns float64 [n_episodes, E, 6] on the device: per episode and environment the sums over UAVs and steps of the
        four reward planes (rewards, target_tracking_reward, boundary_punishment, duplicate_tracking_punishment, as the
        episode statistics hold them), the covered-target sum and the covered-target maximum.  Summed over environments
        (maximum for the last field) an episode's rows equal its episode_stats() exactly."""
        K, T = int(n_episodes), int(nsteps)
        self._ensure_handle(config)
        seeds = (C.c_uint64 * max(K, 1))(*[self._episode_seed(seed, self._episode + k) for k in range(max(K, 0))])
        out = torch.empty((max(K, 0), self.n_envs, 6), dtype=torch.float64, device=self.device)
        w, params = policy_weights(policy, self.state_dim, self.device)  # (params: kept alive over the call)
        self._sync_weights(config)
        mode, coop = self._mode(config, pmi)
        with self._on_device():
            _cabi.check(self._lib.uavsim_evaluate_policy(self._h, mode, coop, C.byref(w), int(bool(greedy)),
                                                         C.c_uint64(policy_seed), C.c_uint64(first_counter),
                                                         seeds if K > 0 else None, K, T,
                                                         C.c_void_p(out.data_ptr()) if K > 0 else None, self._stream()),
                        "uavsim_evaluate_policy")
        self._episode += K
        self._clear_traces()
        return out

    def step_host(self, config, pmi, h_actions, h_obs=None, h_rew4=None, h_covered=None, chunks=4):
        """uavsim_step_host: host (ideally pinned) int32 actions [E,n] in, host obs/rew4/covered out."""
        if self._h is None:
            raise UavSimError("step before reset")
        self._sync_weights(config)
        mode, coop = self._mode(config, pmi)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        with self._on_device():
            _cabi.check(self._lib.uavsim_step_host(self._h, mode, coop, ptr(h_actions), ptr(h_obs), ptr(h_rew4),
                                                   ptr(h_covered), int(chunks), self._stream()), "uavsim_step_host")
        self._host = None

    def step_host_async(self, config, pmi, h_actions, h_obs=None, h_rew4=None, h_covered=None, chunks=4):
        """uavsim_step_host_async: the same step queued without waiting; returns a ticket for step_host_wait.  Queue
        step t+1 (other host output buffers) before waiting for step t and the download of step t overlaps the upload
        and the kernels of step t+1.  Wait for the last ticket before any other call on this environment."""
        if self._h is None:
            raise UavSimError("step before reset")
        self._sync_weights(config)
        mode, coop = self._mode(config, pmi)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        ticket = C.c_int64(-1)
        with self._on_device():
            _cabi.check(self._lib.uavsim_step_host_async(self._h, mode, coop, ptr(h_actions), ptr(h_obs), ptr(h_rew4),
                                                         ptr(h_covered), int(chunks), self._stream(), C.byref(ticket)),
                        "uavsim_step_host_async")
        self._host = None
        return int(ticket.value)

    def step_host_wait(self, ticket):
        """Blocks until the outputs of the step with this ticket are in its host buffers."""
        with self._on_device():
            _cabi.check(self._lib.uavsim_step_host_wait(self._h, int(ticket)), "uavsim_step_host_wait")

    @property
    def actions(self):
        """The bound int32 [E,n] action buffer the next step_device(config, pmi) call reads."""
        return self._actions

    def bind_obs(self, obs):
        """Point the kernel at another resident float32 [E,n,12] observation buffer (no copy): the next step writes its
        observations there and `get_states()` returns it.  A rollout binds slot t+1 of a [T+1,E,n,12] trajectory
        tensor before step t, so states and next_states of every transition are views of one tensor and nothing is
        copied per step.  The caller keeps the tensor alive while it is bound."""
        assert obs.dtype == torch.float32 and obs.is_contiguous() and obs.numel() == self.n_envs * self.n_uav * 12
        assert obs.device == self._obs.device
        self._obs = obs.view(self.n_envs, self.n_uav, 12)
        self._host = None
        self._bind()

    def bind_actions(self, actions):
        """Point the kernel at another resident int32 [E,n] action tensor (no copy)."""
        assert actions.dtype == torch.int32 and actions.is_contiguous() and actions.numel() == self.n_envs * self.n_uav
        self._actions = actions
        b = getattr(self, "_bufs", None)
        if b is None or self._h is None:
            self._bind()
            return
        # one pointer changes: filling the whole struct again (15 data_ptr() calls) cost ~8 us per step, as much as a
        # small step kernel takes to run
        b.actions = actions.data_ptr()
        _cabi.check(self._lib.uavsim_bind(self._h, C.byref(b)), "uavsim_bind")

    def random_actions(self, seed, step):
        with self._on_device():
            _cabi.check(self._lib.uavsim_random_actions(self._h, C.c_uint64(seed), int(step), self._stream()),
                        "uavsim_random_actions")
        return self._actions

    def step(self, config, pmi, actions):
        """Environment.step (src/environment.py:120-164)."""
        if self.n_envs == 1:
            a = torch.as_tensor(np.asarray(actions, dtype=np.int32).reshape(1, self.n_uav), device=self.device)
        elif torch.is_tensor(actions):
            a = actions.to(device=self.device, dtype=torch.int32)
        else:
            a = torch.as_tensor(np.asarray(actions, dtype=np.int32), device=self.device)
        obs, rew4, covered = self.step_device(config, pmi, a)
        if self.trace:
            h0 = self._host0()
            self.position["all_uav_xs"].append(h0["ux"].tolist())
            self.position["all_uav_ys"].append(h0["uy"].tolist())
            self.position["all_target_xs"].append(h0["tx"].tolist())
            self.position["all_target_ys"].append(h0["ty"].tolist())
        if self.n_envs == 1:
            h0 = self._host0()
            r = h0["rew"]
            reward = {k: [r[q, i] for i in range(self.n_uav)] for q, k in enumerate(_REWARD_KEYS)}
            cov = h0["covered"]
            self.covered_target_num.append(cov)
            return self.get_states(), reward, cov
        if self.trace:
            self.covered_target_num.append(self._host0()["covered"])
        return obs, {k: rew4[q] for q, k in enumerate(_REWARD_KEYS)}, covered

    # ------------------------------------------------------------------ extra outputs
    @property
    def done(self):
        return self._done

    @property
    def tracker_counts(self):
        return self._tracker

    @property
    def masks(self):
        return self._masks

    def episode_stats(self):
        """Sums accumulated on the device since the last reset (what src/train.py:181-192 accumulates):
        dict with the four reward sums, covered sum / max, the number of env-steps and `pmi_rows_out_of_range`: pair rows
        the tensor-core PMI kernel saw with inputs beyond the range its fp16 activations hold (0 when it is exact)."""
        out = (C.c_double * 8)()
        with self._on_device():
            _cabi.check(self._lib.uavsim_episode_stats(self._h, out, self._stream()), "uavsim_episode_stats")
        v = list(out)
        return {"rewards": v[0], "target_tracking_reward": v[1], "boundary_punishment": v[2],
                "duplicate_tracking_punishment": v[3], "covered_sum": v[4], "covered_max": v[5], "env_steps": v[6],
                "pmi_rows_out_of_range": v[7]}

    def launch_count(self):
        return int(self._lib.uavsim_launch_count(self._h)) if self._h is not None else 0

    # ------------------------------------------------------------------ traces (src/environment.py:166-244)
    def get_uav_and_target_position(self):
        p = self.position
        return p["all_uav_xs"], p["all_uav_ys"], p["all_target_xs"], p["all_target_ys"]

    def save_position(self, save_dir, epoch_i):
        u_xy = np.array([self.position["all_uav_xs"], self.position["all_uav_ys"]]).transpose()
        t_xy = np.array([self.position["all_target_xs"], self.position["all_target_ys"]]).transpose()
        np.savetxt(os.path.join(save_dir, "u_xy", "u_xy" + str(epoch_i) + ".csv"), u_xy.reshape(-1, 2),
                   delimiter=",", header="x,y", comments="")
        np.savetxt(os.path.join(save_dir, "t_xy", "t_xy" + str(epoch_i) + ".csv"), t_xy.reshape(-1, 2),
                   delimiter=",", header="x,y", comments="")

    def save_covered_num(self, save_dir, epoch_i):
        arr = np.array(self.covered_target_num).reshape(-1, 1)
        np.savetxt(os.path.join(save_dir, "covered_target_num", "covered_target_num" + str(epoch_i) + ".csv"), arr,
                   delimiter=",", header="covered_target_num", comments="")

    def close(self):
        if getattr(self, "_h", None) is not None:
            self._lib.uavsim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# drop-in name: `from marl_uavs_targets_tracking_b200.environment import Environment`
Environment = BatchedEnvironment
