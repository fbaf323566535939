"""ctypes binding of include/footsies_b200.h (libfootsies_b200.so, built in-tree by build.py).

There is no CPU fallback anywhere in this package: if the library is missing it is an error, and
fg_create fails loudly when no CUDA device is present.
"""
import ctypes as C
import os

from . import build as _build

FG_STATE_PLANES = 4
FG_STAT_COUNT = 16
STAT_NAMES = ["episodes", "p1_wins", "p2_wins", "double_ko", "episode_frames", "p1_specials",
              "p1_specials_neutral", "guard_breaks", "hits", "blocks", "env_frames", "resets"]


class FgConfig(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("num_envs", C.c_int32), ("device", C.c_int32),
                ("p1_bot", C.c_int32), ("p2_bot", C.c_int32), ("dense_reward", C.c_int32),
                ("frame_skip", C.c_int32), ("autoreset", C.c_int32), ("stale_intro_input", C.c_int32),
                ("skip_unactionable", C.c_int32), ("first_env_index", C.c_int64)]


class FgBuffers(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("reserved0", C.c_int32),
                ("state", C.c_void_p * FG_STATE_PLANES), ("stats", C.c_void_p),
                ("actions_p1", C.c_void_p), ("actions_p2", C.c_void_p), ("obs", C.c_void_p),
                ("reward", C.c_void_p), ("terminated", C.c_void_p), ("info_frame", C.c_void_p),
                ("info_misc", C.c_void_p), ("step_mask", C.c_void_p)]


class FgHostOutputs(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("reserved0", C.c_int32), ("position", C.c_void_p),
                ("obs_u8", C.c_void_p), ("reward", C.c_void_p), ("terminated", C.c_void_p),
                ("info_frame", C.c_void_p), ("info_misc", C.c_void_p)]


class FgRolloutBuffers(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("hidden", C.c_int32), ("horizon", C.c_int32), ("reserved0", C.c_int32),
                ("scale", C.c_void_p), ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("w3", C.c_void_p), ("b3", C.c_void_p), ("seed", C.c_uint64), ("counter_base", C.c_void_p),
                ("obs", C.c_void_p), ("actions", C.c_void_p), ("logp", C.c_void_p), ("rewards", C.c_void_p),
                ("dones", C.c_void_p),
                ("p2_scale", C.c_void_p), ("p2_w1", C.c_void_p), ("p2_b1", C.c_void_p), ("p2_w2", C.c_void_p),
                ("p2_b2", C.c_void_p), ("p2_w3", C.c_void_p), ("p2_b3", C.c_void_p), ("p2_seed", C.c_uint64),
                ("actions_p2", C.c_void_p), ("logp_p2", C.c_void_p), ("p2_mirror", C.c_int32), ("reserved1", C.c_int32)]


FG_POOL_MAX = 16
FG_POOL_BLOCK = 128


class FgMlpWeights(C.Structure):
    _fields_ = [("scale", C.c_void_p), ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("w3", C.c_void_p), ("b3", C.c_void_p)]


class FgOpponentPool(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("count", C.c_int32), ("member", FgMlpWeights * FG_POOL_MAX),
                ("end", C.c_int64 * FG_POOL_MAX), ("stats", C.c_void_p)]


class FgDelayRing(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("depth", C.c_int32), ("pos", C.c_int32), ("reserved0", C.c_int32),
                ("ring_obs", C.c_void_p), ("ring_frame", C.c_void_p), ("ring_misc", C.c_void_p),
                ("out_obs", C.c_void_p), ("out_frame", C.c_void_p), ("out_misc", C.c_void_p)]


class FgFighterState(C.Structure):
    _fields_ = [("pos_x", C.c_float), ("velocity_x", C.c_float), ("action_id", C.c_int32),
                ("action_frame", C.c_int32), ("hitstun", C.c_int32), ("guard", C.c_int32), ("vital", C.c_int32),
                ("hit_count", C.c_int32), ("buffer_id", C.c_int32), ("reserve_id", C.c_int32),
                ("is_input_backward", C.c_int32), ("is_reserve_prox", C.c_int32), ("shake", C.c_int32),
                ("has_won", C.c_int32), ("input0", C.c_int32), ("hist_left", C.c_uint32),
                ("hist_right", C.c_uint32), ("attack_run", C.c_int32)]


class FgEnvState(C.Structure):
    _fields_ = [("f", FgFighterState * 2), ("frame", C.c_int32), ("recorded_input", C.c_int32 * 2),
                ("done", C.c_int32), ("cum_reward_index", C.c_int32), ("actor_input", C.c_int32 * 2),
                ("rng_state", C.c_uint32 * 4), ("bot_queue", C.c_uint32 * 2), ("p1_bot_memory", C.c_int32)]


# numpy view of FgEnvState (same memory layout)
def env_state_dtype():
    import numpy as np
    fighter = np.dtype([(n, {C.c_float: "<f4", C.c_int32: "<i4", C.c_uint32: "<u4"}[t]) for n, t in FgFighterState._fields_])
    dt = np.dtype([("f", fighter, (2,)), ("frame", "<i4"), ("recorded_input", "<i4", (2,)), ("done", "<i4"),
                   ("cum_reward_index", "<i4"), ("actor_input", "<i4", (2,)), ("rng_state", "<u4", (4,)),
                   ("bot_queue", "<u4", (2,)), ("p1_bot_memory", "<i4")])
    assert dt.itemsize == C.sizeof(FgEnvState), (dt.itemsize, C.sizeof(FgEnvState))
    return dt


class FootsiesLibraryError(RuntimeError):
    pass


FG_PACKED_REWARD_TABLE_SIZE = 128


class HostBlock:
    """Pinned host memory from fg_host_alloc (placed on the GPU's NUMA node), viewed as torch tensors.  The memory lives as
    long as any tensor taken from it: torch.frombuffer keeps the ctypes buffer object alive, and the buffer's finaliser is
    what returns the block to fg_host_free."""

    def __init__(self, device_index: int, nbytes: int):
        import weakref

        import torch
        lib = load()
        self.nbytes = int(nbytes)
        ptr = lib.fg_host_alloc(int(device_index), self.nbytes)
        if not ptr:
            raise FootsiesLibraryError("fg_host_alloc failed: " + lib.fg_last_error().decode("utf-8", "replace"))
        self.ptr = ptr
        raw = (C.c_uint8 * max(self.nbytes, 1)).from_address(ptr)
        weakref.finalize(raw, lib.fg_host_free, ptr).atexit = False     # at interpreter exit the process goes away anyway
        self.bytes = torch.frombuffer(raw, dtype=torch.uint8, count=self.nbytes)
        self._offset = 0

    def take(self, shape, dtype):
        """Next tensor of the block (64-byte aligned)."""
        import torch
        n = int(torch.Size(shape).numel()) * torch.empty((), dtype=dtype).element_size()
        off = (self._offset + 63) // 64 * 64
        if off + n > self.nbytes:
            raise ValueError("host block exhausted")
        self._offset = off + n
        return self.bytes[off:off + n].view(dtype).reshape(shape)


_lib = None

# every symbol include/footsies_b200.h declares
EXPORTS = ["fg_abi_version", "fg_last_error", "fg_algorithmic_bytes_per_env_step", "fg_create", "fg_destroy",
           "fg_bind", "fg_seed", "fg_reset", "fg_step", "fg_step_host", "fg_reset_host", "fg_step_host_compact",
           "fg_reset_host_compact", "fg_packed_reward_table", "fg_step_host_packed", "fg_reset_host_packed", "fg_host_alloc",
           "fg_host_free", "fg_delay_ring_step", "fg_get_state",
           "fg_set_state", "fg_read_stats", "fg_launch_count", "fg_policy_mlp_sample", "fg_policy_mlp_sample_p2", "fg_policy_last_error",
           "fg_rollout_mlp", "fg_rollout_mlp_pool", "fg_rollout_mlp_pool_bot", "fg_rollout_mlp_delayed", "fg_value_mlp", "fg_gae"]


def load(build_if_missing=True):
    """Load the CUDA library; never substitutes anything else for it."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if os.environ.get("FOOTSIES_B200_LIB"):
        pass                      # developer experiment: an explicitly named variant build is loaded as it is
    elif _build.is_stale(path):
        # missing, or built from other sources than the ones in the tree (content digest): never run a stale kernel silently
        if not build_if_missing:
            raise FootsiesLibraryError(f"{path} is missing or stale: run `python -m footsies_gym_b200.build`")
        _build.build()            # lock + atomic rename: safe when every rank of a torchrun job gets here at once
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.fg_abi_version.restype = i32
    L.fg_last_error.restype = C.c_char_p
    L.fg_algorithmic_bytes_per_env_step.restype = i32
    L.fg_algorithmic_bytes_per_env_step.argtypes = [C.POINTER(FgConfig)]
    L.fg_create.restype = i32
    L.fg_create.argtypes = [C.POINTER(FgConfig), C.POINTER(vp)]
    L.fg_destroy.restype = None
    L.fg_destroy.argtypes = [vp]
    L.fg_bind.restype = i32
    L.fg_bind.argtypes = [vp, C.POINTER(FgBuffers)]
    L.fg_seed.restype = i32
    L.fg_seed.argtypes = [vp, i64, vp, vp]
    L.fg_reset.restype = i32
    L.fg_reset.argtypes = [vp, vp, vp]
    L.fg_step.restype = i32
    L.fg_step.argtypes = [vp, vp]
    L.fg_step_host.restype = i32
    L.fg_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.fg_reset_host.restype = i32
    L.fg_reset_host.argtypes = [vp, vp, vp, vp, vp, vp]
    L.fg_step_host_compact.restype = i32
    L.fg_step_host_compact.argtypes = [vp, vp, vp, C.POINTER(FgHostOutputs), vp]
    L.fg_reset_host_compact.restype = i32
    L.fg_reset_host_compact.argtypes = [vp, vp, C.POINTER(FgHostOutputs), vp]
    L.fg_packed_reward_table.restype = i32
    L.fg_packed_reward_table.argtypes = [vp, vp, vp]
    L.fg_step_host_packed.restype = i32
    L.fg_step_host_packed.argtypes = [vp, vp, vp, vp, vp]
    L.fg_reset_host_packed.restype = i32
    L.fg_reset_host_packed.argtypes = [vp, vp, vp, vp]
    L.fg_host_alloc.restype = vp
    L.fg_host_alloc.argtypes = [i32, C.c_uint64]
    L.fg_host_free.restype = None
    L.fg_host_free.argtypes = [vp]
    L.fg_delay_ring_step.restype = i32
    L.fg_delay_ring_step.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.fg_get_state.restype = i32
    L.fg_get_state.argtypes = [vp, i32, i32, vp]
    L.fg_set_state.restype = i32
    L.fg_set_state.argtypes = [vp, i32, i32, vp]
    L.fg_read_stats.restype = i32
    L.fg_read_stats.argtypes = [vp, vp, vp]
    L.fg_launch_count.restype = i64
    L.fg_launch_count.argtypes = [vp]
    L.fg_policy_mlp_sample.restype = i32
    L.fg_policy_mlp_sample.argtypes = [vp] * 8 + [i32, i32, C.c_uint64, C.c_uint64, vp, vp, vp, vp, i64, vp]
    L.fg_policy_mlp_sample_p2.restype = i32
    L.fg_policy_mlp_sample_p2.argtypes = [vp] * 8 + [i32, i32, C.c_uint64, C.c_uint64, vp, vp, vp, i32, i64, vp]
    L.fg_policy_last_error.restype = C.c_char_p
    L.fg_rollout_mlp.restype = i32
    L.fg_rollout_mlp.argtypes = [vp, C.POINTER(FgRolloutBuffers), vp]
    L.fg_rollout_mlp_pool.restype = i32
    L.fg_rollout_mlp_pool.argtypes = [vp, C.POINTER(FgRolloutBuffers), C.POINTER(FgOpponentPool), vp]
    L.fg_rollout_mlp_pool_bot.restype = i32
    L.fg_rollout_mlp_pool_bot.argtypes = [vp, C.POINTER(FgRolloutBuffers), C.POINTER(FgOpponentPool), i32, vp]
    L.fg_rollout_mlp_delayed.restype = i32
    L.fg_rollout_mlp_delayed.argtypes = [vp, C.POINTER(FgRolloutBuffers), C.POINTER(FgOpponentPool), i32,
                                         C.POINTER(FgDelayRing), vp]
    L.fg_value_mlp.restype = i32
    L.fg_value_mlp.argtypes = [vp] * 8 + [i32, i64, vp, vp]
    L.fg_gae.restype = i32
    L.fg_gae.argtypes = [vp, vp, vp, i32, i32, C.c_float, C.c_float, vp, vp, vp]
    if L.fg_abi_version() != 2:
        raise FootsiesLibraryError("libfootsies_b200.so ABI version mismatch")
    _lib = L
    return L


def check(rc):
    if rc != 0:
        msg = load().fg_last_error().decode("utf-8", "replace")
        raise FootsiesLibraryError(f"libfootsies_b200 error {rc}: {msg}")
