"""ctypes binding of libvn_b200.so - the C ABI declared in include/vn_b200.h.

There is no CPU fallback: if the library cannot be loaded every entry point raises.  PyTorch only
supplies device memory (``tensor.data_ptr()``) and the current stream.
"""
import ctypes as C
import os

from . import build as _build

VN_MAX_PLANES = 6
VN_N_STATS = 9

RULE_COLLISION_SKIPS_GOAL = 0x01
RULE_NEG_STEP_REWARD = 0x02
RULE_COLLISION_OVERRIDES = 0x04
RULE_TERM_PREV_OBS = 0x08
RULE_TWO_LEVEL = 0x10
RULE_NOOP_ACTION = 0x20
RULE_AUTO_RESET = 0x40

GATHER_AUTO, GATHER_LDG, GATHER_BULK, GATHER_FUSED, GATHER_PERSISTENT = 0, 1, 2, 3, 4
STEP_ACTIONS_READY = 0x01
STEP_SKIP_UNCHANGED = 0x02
STEP_NO_OVERLAP = 0x04
MODE_SPLIT, MODE_FUSED, MODE_PERSISTENT = 0, 1, 2
ABI_VERSION = 6
DTYPE_F16, DTYPE_BF16 = 1, 2
STAT_NAMES = ("episodes", "return_sum", "length_sum", "successes", "collisions", "steps", "truncations", "resets",
              "rows_skipped")

_P = C.c_void_p


class Store(C.Structure):
    _fields_ = [("base", _P), ("state_pitch", C.c_int64), ("n_states", C.c_int32), ("n_planes", C.c_int32),
                ("plane_off", C.c_int32 * VN_MAX_PLANES), ("plane_bytes", C.c_int32 * VN_MAX_PLANES)]


class Tables(C.Structure):
    _fields_ = [("adj", _P), ("task_goal", _P), ("task_cand_off", _P), ("task_prefix", _P), ("cand_state", _P),
                ("n_states", C.c_int32), ("n_tasks", C.c_int32)]


class Envs(C.Structure):
    _fields_ = [("n_envs", C.c_int32), ("env_id_base", C.c_int32), ("state", _P), ("goal", _P), ("task", _P),
                ("elapsed", _P), ("epoch", _P), ("ep_return", _P), ("ep_length", _P), ("task_lo", _P),
                ("task_cnt", _P)]


class Rules(C.Structure):
    _fields_ = [("reward_goal", C.c_float), ("reward_step", C.c_float), ("reward_collision", C.c_float),
                ("max_episode_steps", C.c_int32), ("goal_compare", C.c_int32), ("flags", C.c_int32),
                ("n_actions", C.c_int32), ("reserved", C.c_int32), ("seed", C.c_uint64)]


class Inject(C.Structure):
    _fields_ = [("task", _P), ("start", _P), ("stride", C.c_int32), ("reserved", C.c_int32)]


class FloatLeaf(C.Structure):
    _fields_ = [("plane", C.c_int32), ("source", C.c_int32), ("channels", C.c_int32), ("reserved", C.c_int32),
                ("out", _P)]


class StepOut(C.Structure):
    _fields_ = [("obs", _P * VN_MAX_PLANES), ("goal_obs", _P * VN_MAX_PLANES), ("reward", _P), ("done", _P),
                ("truncated", _P), ("win", _P), ("did_reset", _P), ("last_action_reward", _P),
                ("episode_return", _P), ("episode_length", _P), ("info_state", _P), ("obs_state", _P), ("stats", _P),
                ("gather_desc", _P), ("parity", C.c_int32), ("flags", C.c_int32), ("sched", _P), ("host_pack", _P),
                ("host_seq", _P), ("seq", C.c_uint32), ("reserved", C.c_uint32),
                ("rec_action", _P), ("rec_reward", _P), ("rec_done", _P), ("rec_state", _P), ("rec_goal", _P),
                ("float_leaves", _P), ("n_float_leaves", C.c_int32), ("float_h", C.c_int32), ("float_w", C.c_int32),
                ("reserved2", C.c_int32)]


class Replay(C.Structure):
    _fields_ = [("before", _P), ("after", _P), ("goal", _P), ("goal_before", _P), ("action", _P), ("reward", _P),
                ("done", _P),
                ("n", C.c_int32), ("cap", C.c_int32), ("head", C.c_int32), ("count", C.c_int32)]


class HostCall(C.Structure):
    _fields_ = [("store", _P), ("tables", _P), ("envs", _P), ("rules", _P), ("inject", _P), ("host_actions", _P),
                ("dev_actions_copy", _P), ("out", _P), ("seq_words", C.c_int32), ("gather_variant", C.c_int32),
                ("timeout_us", C.c_int64)]


class U8Frames(C.Structure):
    _fields_ = [("base", _P), ("pitch", C.c_int64), ("idx", _P), ("idx_stride_n", C.c_int64),
                ("idx_stride_t", C.c_int64), ("n", C.c_int32), ("idx_t", C.c_int32), ("h", C.c_int32),
                ("w", C.c_int32), ("c", C.c_int32), ("reserved", C.c_int32)]


class VnError(RuntimeError):
    pass


_lib = None

#: every symbol include/vn_b200.h declares
EXPORTS = ("vn_abi_version", "vn_abi_struct_size", "vn_last_error", "vn_launch_count", "vn_fill_store", "vn_env_reset", "vn_env_step", "vn_env_step_scalar",
           "vn_env_gather", "vn_env_step_host", "vn_env_step_host_sync", "vn_env_step_host_call", "vn_env_step_mode", "vn_debug_gather_trace", "vn_env_host_seq_words", "vn_host_wait_seq", "vn_event_create", "vn_event_destroy", "vn_event_wait", "vn_gather_plane",
           "vn_gather_plane_f32_chw", "vn_gather_plane_f32_chw_rows", "vn_gather_leaves_f32_chw", "vn_nstep_returns", "vn_nstep_returns_scan", "vn_discounted_backup", "vn_pixel_control",
           "vn_transition_rows", "vn_gather_rows", "vn_pixel_control_list", "vn_pixel_control_returns", "vn_pixel_control_returns_from_states", "vn_replay_sample",
           "vn_aux_target", "vn_rp_labels", "vn_conv_u8_forward", "vn_conv_u8_wgrad_scratch_bytes", "vn_conv_u8_backward",
           "vn_conv_u8_forward_lp", "vn_conv_u8_backward_lp", "vn_conv_u8_planes_forward", "vn_conv_u8_planes_forward_lp",
           "vn_conv_u8_planes_backward", "vn_conv_u8_planes_backward_lp")


def library_path():
    return _build.LIB


def load(build_if_missing=True):
    """Loads (building first if the .so is absent or stale and nvcc is present) and types the library."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing and _build.needs_build():
        try:
            _build.build()
        except Exception as e:   # keep a stale-but-present library usable on boxes without nvcc - but say so
            if not os.path.exists(path):
                raise VnError("libvn_b200.so is missing and could not be built: %s" % e)
            import warnings
            warnings.warn("libvn_b200.so is OLDER than its sources and the rebuild failed (%s): running the stale "
                          "library (the ABI version and struct sizes are still checked below)" % e, RuntimeWarning)
    if not os.path.exists(path):
        raise VnError("libvn_b200.so not found at %s - run `python __graft_entry__.py` (build()) first" % path)
    lib = C.CDLL(path)
    i32, i64, u64, f32 = C.c_int32, C.c_int64, C.c_uint64, C.c_float
    S, T, E, R, I, O = (C.POINTER(x) for x in (Store, Tables, Envs, Rules, Inject, StepOut))
    sig = {
        "vn_abi_version": (i32, []),
        "vn_abi_struct_size": (i32, [i32]),
        "vn_last_error": (C.c_char_p, []),
        "vn_launch_count": (i64, []),
        "vn_fill_store": (i32, [S, i32, i32, u64, i32, i32, C.POINTER(i32), _P]),
        "vn_env_reset": (i32, [S, T, E, R, I, _P, O, i32, _P]),
        "vn_env_step": (i32, [S, T, E, R, I, _P, O, i32, _P]),
        "vn_env_step_scalar": (i32, [T, E, R, I, _P, O, _P]),
        "vn_env_gather": (i32, [S, E, O, i32, _P]),
        "vn_env_step_host": (i32, [S, T, E, R, I, _P, _P, O, _P, i32, _P]),
        "vn_env_step_host_sync": (i32, [S, T, E, R, I, _P, _P, O, _P, _P, _P, i32, i32, _P, i64]),
        "vn_env_step_host_call": (i32, [_P, _P, _P, _P]),
        "vn_debug_gather_trace": (i32, [_P]),
        "vn_env_host_seq_words": (i32, [S, E, O, i32]),
        "vn_env_step_mode": (i32, [S, E, O, i32]),
        "vn_host_wait_seq": (i32, [_P, i32, C.c_uint32, _P, i64]),
        "vn_event_create": (i32, [C.POINTER(_P)]),
        "vn_event_destroy": (i32, [_P]),
        "vn_event_wait": (i32, [_P]),
        "vn_gather_plane": (i32, [S, i32, _P, i32, _P, i32, _P]),
        "vn_gather_plane_f32_chw": (i32, [S, i32, _P, i32, i32, i32, i32, _P, _P]),
        "vn_gather_plane_f32_chw_rows": (i32, [S, i32, _P, i32, i32, i32, i32, i32, _P, _P]),
        "vn_gather_leaves_f32_chw": (i32, [S, C.POINTER(FloatLeaf), i32, _P, i32, i32, i32, _P]),
        "vn_nstep_returns": (i32, [_P, _P, _P, f32, i32, i32, i64, i64, _P, i64, i64, _P]),
        "vn_nstep_returns_scan": (i32, [_P, _P, _P, f32, i32, i32, i64, i64, _P, i64, i64, _P]),
        "vn_discounted_backup": (i32, [_P, _P, i64, i64, _P, f32, i32, i32, i32, _P, _P]),
        "vn_pixel_control": (i32, [S, i32, _P, i32, i32, i64, i64, i32, i32, i32, i32, i32, i32, _P, _P]),
        "vn_transition_rows": (i32, [_P, _P, i32, i32, i64, i64, _P, i64, i64, _P, _P, _P]),
        "vn_gather_rows": (i32, [_P, i64, _P, i64, i32, i64, i64, _P, _P]),
        "vn_pixel_control_list": (i32, [S, i32, _P, i32, i32, i64, i64, i32, i32, i32, i32, i32, i32, _P, _P, i32, i32,
                                        _P, _P]),
        "vn_pixel_control_returns": (i32, [_P, i32, _P, i64, i64, _P, _P, i64, i64, _P, f32, i32, i32, _P, _P, _P]),
        "vn_pixel_control_returns_from_states": (i32, [S, i32, _P, _P, _P, i64, i64, _P, i64, i64, _P, f32, i32, i32, i32,
                                                       i32, i32, i32, i32, i32, _P, _P, _P, _P, i32, _P, _P, _P]),
        "vn_replay_sample": (i32, [C.POINTER(Replay), i32, i32, u64, C.c_uint32, i32, _P, _P, _P, _P, _P, _P, _P, _P]),
        "vn_aux_target": (i32, [S, i32, _P, i32, i32, i32, i32, i32, i32, i32, _P, _P]),
        "vn_rp_labels": (i32, [_P, i32, i32, i64, i64, _P, _P, _P, _P, _P, _P]),
        "vn_conv_u8_forward": (i32, [C.POINTER(U8Frames), _P, _P, i32, i32, i32, _P, _P]),
        "vn_conv_u8_wgrad_scratch_bytes": (i64, [i32, i32, i32, i32]),
        "vn_conv_u8_backward": (i32, [C.POINTER(U8Frames), _P, i32, i32, i32, _P, _P, _P, i64, _P]),
        "vn_conv_u8_forward_lp": (i32, [C.POINTER(U8Frames), _P, _P, i32, i32, i32, i32, _P, _P]),
        "vn_conv_u8_backward_lp": (i32, [C.POINTER(U8Frames), _P, i32, i32, i32, i32, _P, _P, _P, i64, _P]),
        "vn_conv_u8_planes_forward": (i32, [C.POINTER(U8Frames), i32, _P, _P, i32, i32, i32, _P, _P]),
        "vn_conv_u8_planes_forward_lp": (i32, [C.POINTER(U8Frames), i32, _P, _P, i32, i32, i32, i32, _P, _P]),
        "vn_conv_u8_planes_backward": (i32, [C.POINTER(U8Frames), i32, _P, i32, i32, i32, _P, _P, _P, i64, _P]),
        "vn_conv_u8_planes_backward_lp": (i32, [C.POINTER(U8Frames), i32, _P, i32, i32, i32, i32, _P, _P, _P, i64, _P]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.vn_abi_version() != ABI_VERSION:
        raise VnError("libvn_b200.so ABI version %d, expected %d - rebuild with `python __graft_entry__.py`"
                      % (lib.vn_abi_version(), ABI_VERSION))
    for which, mirror in enumerate((Store, Tables, Envs, Rules, Inject, StepOut, Replay, FloatLeaf, HostCall,
                                     U8Frames)):
        if lib.vn_abi_struct_size(which) != C.sizeof(mirror):
            raise VnError("libvn_b200.so is stale: sizeof(%s) is %d in the library, %d in lib.py - rebuild with "
                          "`python __graft_entry__.py`" % (mirror.__name__, lib.vn_abi_struct_size(which), C.sizeof(mirror)))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise VnError("libvn_b200 error %d: %s" % (rc, load().vn_last_error().decode()))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def current_stream():
    import torch
    return torch.cuda.current_stream().cuda_stream
