"""Device-resident prioritized replay (SURVEY.md section 8f, row f-2).

`PrioritizedReplayBuffer` keeps the reference's constructor and method names (src/train.py:73-139) but stores the
transitions in HBM and takes / returns CUDA tensors; every call is a handful of kernel launches of libuavsim.so
(`csrc/replay.cuh`) instead of a python loop with an O(capacity) `priorities.max()` per inserted transition.
There is no CPU fallback.
"""
import ctypes as C

import torch

from . import _cabi


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class PrioritizedReplayBuffer:
    """Same behaviour as the reference class; differences a caller sees:

    * `add` takes a dict of device tensors (states [B,D] f32, actions [B] int, rewards [B] f32, next_states [B,D] f32)
      -- what `rollout.operate_epoch_batched` returns -- instead of python lists;
    * `sample` returns device tensors and draws its uniforms from Philox4x32-10 (seed given at construction, one
      counter per call) instead of numpy's global generator; `uniforms=` overrides them (tests);
    * rewards are stored as float32 (the device environment emits float32 rewards).
    """

    def __init__(self, capacity, alpha=0.6, state_dim=12, device="cuda:0", seed=0):
        self.capacity, self.alpha, self.state_dim = int(capacity), float(alpha), int(state_dim)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _cabi.UavSimError("PrioritizedReplayBuffer needs a CUDA device (no CPU fallback)")
        self._lib = _cabi.load()
        self._h = C.c_void_p()
        _cabi.check(self._lib.uavsim_replay_create(self.capacity, self.state_dim, self.alpha, self.device.index or 0,
                                                   C.byref(self._h)), "uavsim_replay_create")
        # every rank keeps its own ring: its draws must not repeat rank 0's
        import torch.distributed as dist
        rank = dist.get_rank() if (dist.is_available() and dist.is_initialized()) else 0
        self.seed, self._draws = (int(seed) + 0xD1B54A32D192ED03 * rank) & 0xFFFFFFFFFFFFFFFF, 0

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.uavsim_replay_destroy(h)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def add(self, transition_dict):
        s = transition_dict["states"].to(self.device, torch.float32).reshape(-1, self.state_dim).contiguous()
        s2 = transition_dict["next_states"].to(self.device, torch.float32).reshape(-1, self.state_dim).contiguous()
        a = transition_dict["actions"].to(self.device, torch.int32).reshape(-1).contiguous()
        r = transition_dict["rewards"].to(self.device, torch.float32).reshape(-1).contiguous()
        n = s.shape[0]
        if not (s2.shape[0] == a.shape[0] == r.shape[0] == n):
            raise ValueError("transition_dict entries disagree on the number of transitions")
        _cabi.check(self._lib.uavsim_replay_add(self._h, _ptr(s), _ptr(a), _ptr(r), _ptr(s2), n, self._stream()),
                    "uavsim_replay_add")

    def sample(self, batch_size, beta=0.4, uniforms=None):
        n = min(int(batch_size), self.size())
        if n == 0:  # train.py:101-102
            return dict(states=[], actions=[], rewards=[], next_states=[]), None, None
        dev, D = self.device, self.state_dim
        out = {"states": torch.empty(n, D, dtype=torch.float32, device=dev),
               "actions": torch.empty(n, dtype=torch.int32, device=dev),
               "rewards": torch.empty(n, dtype=torch.float32, device=dev),
               "next_states": torch.empty(n, D, dtype=torch.float32, device=dev)}
        indices = torch.empty(n, dtype=torch.int64, device=dev)
        weights = torch.empty(n, dtype=torch.float32, device=dev)
        if uniforms is not None:
            uniforms = uniforms.to(dev, torch.float64).contiguous()
            if uniforms.numel() < n:
                raise ValueError("need %d uniforms, got %d" % (n, uniforms.numel()))
        n_out = C.c_int64(0)
        _cabi.check(self._lib.uavsim_replay_sample(self._h, n, float(beta), _ptr(uniforms), self.seed, self._draws,
                                                   _ptr(out["states"]), _ptr(out["actions"]), _ptr(out["rewards"]),
                                                   _ptr(out["next_states"]), _ptr(indices), _ptr(weights),
                                                   C.byref(n_out), self._stream()), "uavsim_replay_sample")
        self._draws += 1
        assert n_out.value == n
        return out, indices, weights

    def update_priorities(self, batch_indices, batch_priorities):
        idx = torch.as_tensor(batch_indices).to(self.device, torch.int64).reshape(-1).contiguous()
        pri = torch.as_tensor(batch_priorities).to(self.device, torch.float32).reshape(-1).contiguous()
        if idx.numel() != pri.numel():
            raise ValueError("indices and priorities differ in length")
        if idx.numel():
            # one host synchronisation for both checks, before anything is written.  A NaN, infinite or negative
            # priority would give the next sample NaN or negative probabilities (the reference's numpy.random.choice
            # raises there); -0.0 is a zero priority.
            lo, hi, bad = torch.stack([idx.min(), idx.max(), (~torch.isfinite(pri) | (pri < 0)).any().long()]).tolist()
            if lo < 0 or hi >= self.capacity:
                raise IndexError("replay index out of range")
            if bad:
                raise ValueError("priorities must be finite and non-negative")
        _cabi.check(self._lib.uavsim_replay_update_priorities(self._h, _ptr(idx), _ptr(pri), idx.numel(), self._stream()),
                    "uavsim_replay_update_priorities")

    def size(self):
        return int(self._lib.uavsim_replay_size(self._h))

    @property
    def pos(self):
        return int(self._lib.uavsim_replay_pos(self._h))

    @property
    def launches(self):
        return int(self._lib.uavsim_replay_launch_count(self._h))

    def export(self):
        """Host copy of the ring: dict(states, actions, rewards, next_states [size,...], priorities [capacity],
        probabilities [size] of the last sample call) -- checkpointing and tests."""
        n, D = self.size(), self.state_dim
        out = {"states": torch.empty(n, D, dtype=torch.float32), "actions": torch.empty(n, dtype=torch.int32),
               "rewards": torch.empty(n, dtype=torch.float32), "next_states": torch.empty(n, D, dtype=torch.float32),
               "priorities": torch.empty(self.capacity, dtype=torch.float32),
               "probabilities": torch.empty(n, dtype=torch.float32)}
        _cabi.check(self._lib.uavsim_replay_export(self._h, _ptr(out["states"]), _ptr(out["actions"]), _ptr(out["rewards"]),
                                                   _ptr(out["next_states"]), _ptr(out["priorities"]),
                                                   _ptr(out["probabilities"]), self._stream()), "uavsim_replay_export")
        return out
