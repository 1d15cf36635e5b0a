"""ctypes binding of libuavsim.so (the C ABI declared in include/uavsim.h).

There is no CPU path: if the library has not been built this module raises, and every
compute entry point returns an error code (raised as UavSimError) when no CUDA device is
present.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UAVSIM_LIB") or os.path.join(_HERE, "csrc", "libuavsim.so")  # UAVSIM_LIB: tuning builds

MODE_SELF, MODE_MEAN, MODE_PMI = 0, 1, 2
OBS_DIM = 12
MAX_UAV = 128


class UavSimError(RuntimeError):
    pass


class UavSimParams(C.Structure):
    _fields_ = [("n_uav", C.c_int32), ("m_targets", C.c_int32), ("na", C.c_int32), ("num_steps", C.c_int32)] + [
        (k, C.c_double) for k in ("x_max", "y_max", "dt", "uav_v_max", "uav_h_max", "dc", "dp", "tgt_v_max",
                                  "tgt_h_max", "alpha", "beta", "gamma")]


_BUF_FIELDS = ("ux", "uy", "uh", "ua", "tx", "ty", "th", "actions", "obs", "rew4", "covered", "tracker_cnt", "done",
               "raw", "nbr_bits", "obs_mask", "comm_mask", "nbr_mask", "dup_mask", "cover_mask")


class UavSimBuffers(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in _BUF_FIELDS]


class UavSimPolicyWeights(C.Structure):
    _fields_ = [("state_dim", C.c_int32), ("hidden", C.c_int32), ("n_actions", C.c_int32), ("_pad", C.c_int32),
                ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p)]


class UavSimTrajectory(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("obs", "actions", "rew4", "covered")]


class UavSimPmiWeights(C.Structure):
    _fields_ = [("hidden", C.c_int32), ("_pad", C.c_int32), ("w0", C.c_void_p), ("b0", C.c_void_p),
                ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_float), ("_pad2", C.c_float)]


# every symbol include/uavsim.h declares: name -> (restype, argtypes)
_H = C.c_void_p
SYMBOLS = {
    "uavsim_abi_version": (C.c_int, []),
    "uavsim_last_error": (C.c_char_p, []),
    "uavsim_create": (C.c_int, [C.POINTER(UavSimParams), C.c_int64, C.c_int64, C.c_int, C.POINTER(_H)]),
    "uavsim_destroy": (C.c_int, [_H]),
    "uavsim_bind": (C.c_int, [_H, C.POINTER(UavSimBuffers)]),
    "uavsim_reset": (C.c_int, [_H, C.c_uint64, C.c_void_p]),
    "uavsim_begin_episode": (C.c_int, [_H, C.c_void_p]),
    "uavsim_random_actions": (C.c_int, [_H, C.c_uint64, C.c_int64, C.c_void_p]),
    "uavsim_step": (C.c_int, [_H, C.c_int, C.c_double, C.c_void_p]),
    "uavsim_run_random_policy": (C.c_int, [_H, C.c_int, C.c_double, C.c_uint64, C.c_int64, C.c_int64, C.c_void_p]),
    "uavsim_step_host": (C.c_int, [_H, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_void_p]),
    "uavsim_step_host_async": (C.c_int, [_H, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_void_p, C.POINTER(C.c_int64)]),
    "uavsim_step_host_wait": (C.c_int, [_H, C.c_int64]),
    "uavsim_set_reward_weights": (C.c_int, [_H, C.c_double, C.c_double, C.c_double]),
    "uavsim_set_pmi_weights": (C.c_int, [_H, C.POINTER(UavSimPmiWeights), C.c_void_p]),
    "uavsim_set_pmi_path": (C.c_int, [_H, C.c_int]),
    "uavsim_set_step_path": (C.c_int, [_H, C.c_int]),
    "uavsim_episode_stats": (C.c_int, [_H, C.POINTER(C.c_double), C.c_void_p]),
    "uavsim_launch_count": (C.c_int64, [_H]),
    "uavsim_step_count": (C.c_int64, [_H]),
    "uavsim_policy_sample": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(UavSimPolicyWeights), C.c_uint64, C.c_uint64,
                                       C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "uavsim_run_policy": (C.c_int, [_H, C.c_int, C.c_double, C.POINTER(UavSimPolicyWeights), C.c_uint64, C.c_uint64,
                                    C.c_int64, C.POINTER(UavSimTrajectory), C.c_void_p]),
    # prioritized replay (src/train.py:73-139)
    "uavsim_replay_create": (C.c_int, [C.c_int64, C.c_int, C.c_double, C.c_int, C.POINTER(_H)]),
    "uavsim_replay_destroy": (C.c_int, [_H]),
    "uavsim_replay_add": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "uavsim_replay_sample": (C.c_int, [_H, C.c_int64, C.c_double, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.POINTER(C.c_int64), C.c_void_p]),
    "uavsim_replay_update_priorities": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "uavsim_replay_size": (C.c_int64, [_H]),
    "uavsim_replay_pos": (C.c_int64, [_H]),
    "uavsim_replay_launch_count": (C.c_int64, [_H]),
    "uavsim_replay_export": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
}

_lib = None


def load():
    """Load libuavsim.so; raises UavSimError if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UavSimError(
            "libuavsim.so is missing (%s): build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C marl_uavs_targets_tracking_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    if lib.uavsim_abi_version() != 1:
        raise UavSimError("libuavsim.so ABI version %d, expected 1" % lib.uavsim_abi_version())
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().uavsim_last_error()
        raise UavSimError("%s failed (code %d): %s" % (what or "libuavsim call", rc, (msg or b"").decode()))
