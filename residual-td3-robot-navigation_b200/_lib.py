"""ctypes binding of csrc/librtd3.so (the C ABI declared in include/rtd3.h).

There is no fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int32, c_int64, c_uint32, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "librtd3.so")


class Rtd3Error(RuntimeError):
    pass


class MtBankStruct(Structure):
    _fields_ = [("mt", c_void_p), ("pos", c_void_p), ("has_gauss", c_void_p), ("gauss", c_void_p), ("n", c_int64)]


class TickStateStruct(Structure):
    """`rtd3_tick_state` of include/rtd3.h (same field order)."""
    _fields_ = ([("n", c_int64)]
                + [(k, c_void_p) for k in ("x", "y", "goal", "region", "state64")]
                + [("env_bank", MtBankStruct)]
                + [(k, c_void_p) for k in ("num_episodes", "demo_flag", "plan_index", "path_length", "goal_reached", "stuck_flag", "noise_scale",
                                           "hist", "hist_count", "hist_head", "type", "update", "any_update",
                                           "base", "ax", "ay", "prev_x", "prev_y", "reward", "reward64", "done",
                                           "demo", "demo_list_start", "demo_list")]
                + [("num_demo", c_int64)]
                + [(k, c_void_p) for k in ("rp_s", "rp_a", "rp_r", "rp_s2", "rp_notdone")]
                + [("capacity", c_int64), ("rp_total", c_void_p), ("steps_bought", c_void_p), ("resets_bought", c_void_p),
                   ("philox_seed", c_uint64), ("tick_counter", c_void_p)]
                + [(k, c_void_p) for k in ("mode", "demos_bought", "test_ticks", "test_best", "test_success", "penalty")]
                + [("tick_seconds", c_double), ("test_timeout_ticks", c_int64)]
                + [(k, c_void_p) for k in ("env_demo_pts", "env_demo_cells", "env_demo_count")] + [("env_demo_cap", c_int64)])


class CemWorkspaceStruct(Structure):
    """`rtd3_cem_workspace` of include/rtd3.h."""
    _fields_ = [(k, c_void_p) for k in ("actions", "x", "y", "start_x", "start_y", "start64", "rewards", "elite", "best", "mean", "std",
                                        "best_actions", "traj")]


TICK_NOISE_NONE, TICK_NOISE_GIVEN, TICK_NOISE_PHILOX = 0, 1, 2
TICK_TYPE_STEP, TICK_TYPE_DEMO, TICK_TYPE_RESET, TICK_TYPE_SWITCH, TICK_TYPE_SKIP, TICK_TYPE_TEST, TICK_TYPE_IDLE = range(7)
COMM_ID_BYTES = 128


class P2pStateStruct(Structure):
    """`rtd3_p2p_state` of include/rtd3.h."""
    _fields_ = [("peer_recv", c_void_p), ("peer_flags", c_void_p), ("rank", c_int32), ("world", c_int32), ("seq_counter", c_void_p),
                ("sum", c_void_p), ("slot_floats", c_int64), ("block_counter", c_void_p)]


class Td3UpdateArgs(Structure):
    """`rtd3_td3_update_args` of include/rtd3.h (same field order)."""
    _fields_ = ([(k, c_void_p) for k in ("params", "params_t", "params_uv", "grads", "adam_m", "adam_v", "scratch", "steps", "beta_pows",
                                         "rp_s", "rp_a", "rp_r", "rp_s2", "rp_notdone", "idx")]
                + [("batch", c_int32), ("epochs", c_int32), ("policy_update_delay", c_int32)]
                + [("noise", c_void_p), ("noise_seed", c_uint64), ("noise_counter", c_void_p)]
                + [(k, c_float) for k in ("gamma", "policy_noise", "noise_clip", "max_action")]
                + [("lr_actor", c_double), ("lr_critic", c_double), ("tau", c_float)]
                + [("critic_losses", c_void_p), ("actor_losses", c_void_p), ("world", c_int32), ("tf32", c_int32), ("comm", c_void_p),
                   ("p2p", POINTER(P2pStateStruct))])

_P = c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "rtd3_version": (c_int32, []),
    "rtd3_last_error": (c_char_p, []),
    "rtd3_launch_count": (c_int64, []),
    "rtd3_launch_count_reset": (None, []),
    "rtd3_launch_count_add": (None, [c_int64]),
    "rtd3_env_create": (c_int32, [POINTER(c_void_p), c_int32]),
    "rtd3_env_destroy": (c_int32, [_P]),
    "rtd3_env_set_map": (c_int32, [_P, _P, _P, _P]),
    "rtd3_env_set_maps": (c_int32, [_P, _P, _P, c_int32, _P]),
    "rtd3_env_set_map_index": (c_int32, [_P, _P, c_int64, _P]),
    "rtd3_perlin_maps": (c_int32, [_P, c_int32, _P, _P, _P]),
    "rtd3_perlin_set_raw_fields": (None, [c_int32]),
    "rtd3_env_map_config": (c_int32, [_P, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int32), POINTER(c_int64)]),
    "rtd3_env_step": (c_int32, [_P, _P, _P, _P, _P, c_int64, c_int32, _P]),
    "rtd3_env_dynamics": (c_int32, [_P, _P, _P, _P, _P, _P, _P, c_int64, _P]),
    "rtd3_env_rollout": (c_int32, [_P, _P, _P, _P, _P, c_int64, c_int64, _P]),
    "rtd3_env_force_plain_rollout": (None, [c_int32]),
    "rtd3_env_set_launch_overlap": (None, [c_int32]),
    "rtd3_env_rollout_host": (c_int32, [_P, _P, _P, _P, _P, c_int64, c_int64, c_int32, c_int32, _P]),
    "rtd3_mt_seed": (c_int32, [POINTER(MtBankStruct), _P, _P]),
    "rtd3_mt_draw_u32": (c_int32, [POINTER(MtBankStruct), _P, c_int64, _P]),
    "rtd3_mt_draw_gauss": (c_int32, [POINTER(MtBankStruct), _P, c_int64, _P]),
    "rtd3_mt_draw_gauss_where": (c_int32, [POINTER(MtBankStruct), _P, c_int64, _P, c_int32, _P]),
    "rtd3_env_init_goal_region": (c_int32, [POINTER(MtBankStruct), _P, _P, _P]),
    "rtd3_env_reset": (c_int32, [POINTER(MtBankStruct), _P, _P, c_int32, _P, _P, _P, _P]),
    "rtd3_replay_push": (c_int32, [_P, _P, _P, _P, _P, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, _P]),
    "rtd3_replay_gather": (c_int32, [_P, _P, _P, _P, _P, _P, c_int32, _P, _P, _P, _P, _P, _P]),
    "rtd3_sample_indices_mt19937": (c_int32, [POINTER(MtBankStruct), c_int64, c_int32, c_int32, c_int32, _P, _P, _P]),
    "rtd3_sample_indices_philox": (c_int32, [c_uint64, c_uint64, c_int64, c_int32, c_int32, _P, _P]),
    "rtd3_td3_create": (c_int32, [POINTER(c_void_p), c_int32, c_int32, c_int32]),
    "rtd3_td3_destroy": (c_int32, [_P]),
    "rtd3_td3_param_count": (c_int64, [_P, c_int32]),
    "rtd3_td3_param_offset": (c_int64, [_P, c_int32]),
    "rtd3_td3_arena_floats": (c_int64, [_P]),
    "rtd3_td3_scratch_floats": (c_int64, [_P, c_int32]),
    "rtd3_td3_sync_transposed": (c_int32, [_P, _P, _P, _P]),
    "rtd3_td3_critic_step": (c_int32, [_P] * 12 + [c_int32, c_float, c_float, c_float, c_float] + [_P] * 6),
    "rtd3_td3_actor_step": (c_int32, [_P] * 7 + [c_int32, _P, _P, _P, _P]),
    "rtd3_td3_adam_polyak": (c_int32, [_P] * 8 + [c_int32, c_double, c_double, c_float, c_int32, c_float, _P]),
    "rtd3_mlp_forward": (c_int32, [_P, c_int32, _P, _P, _P, _P, c_int64, _P]),
    "rtd3_tc_sync_weights": (c_int32, [c_int32, c_int32, _P, _P, _P]),
    "rtd3_mlp_forward_tf32": (c_int32, [c_int32, c_int32, c_int32, c_int64, _P, _P, _P, _P, c_int64, _P]),
    "rtd3_tc_sync_weights_f16": (c_int32, [c_int32, c_int32, _P, _P, _P]),
    "rtd3_mlp_forward_f16": (c_int32, [c_int32, c_int32, c_int32, _P, _P, _P, _P, c_int64, _P]),
    "rtd3_td3_tf32_supported": (c_int32, [_P]),
    "rtd3_td3_critic_step_tf32": (c_int32, [_P] * 11 + [c_int32, c_float, c_float, c_float, c_float] + [_P] * 6),
    "rtd3_td3_actor_step_tf32": (c_int32, [_P] * 6 + [c_int32, _P, _P, _P, _P]),
    "rtd3_debug_lt_prof": (c_int32, [c_int32, _P]),
    "rtd3_trainer_tally": (c_int32, [_P, _P, _P, c_int64, _P]),
    "rtd3_p2p_allreduce": (c_int32, [_P, _P, c_int32, c_int32, _P, _P, _P, c_int64, c_int64, _P, _P]),
    "rtd3_comm_nccl_version": (c_int32, []),
    "rtd3_comm_unique_id": (c_int32, [_P]),
    "rtd3_comm_create": (c_int32, [POINTER(c_void_p), _P, c_int32, c_int32, c_int32]),
    "rtd3_comm_destroy": (c_int32, [_P]),
    "rtd3_comm_world": (c_int32, [_P]),
    "rtd3_comm_rank": (c_int32, [_P]),
    "rtd3_allreduce_grads": (c_int32, [_P, _P, c_int64, _P]),
    "rtd3_td3_update": (c_int32, [_P, POINTER(Td3UpdateArgs), _P]),
    "rtd3_td3_coop_supported": (c_int32, [_P, c_int32]),
    "rtd3_td3_coop_scratch_floats": (c_int64, [_P, c_int32]),
    "rtd3_td3_update_coop": (c_int32, [_P, POINTER(Td3UpdateArgs), _P, _P]),
    "rtd3_debug_coop_prof": (c_int32, [_P]),
    "rtd3_td3_cluster_supported": (c_int32, [_P, c_int32]),
    "rtd3_td3_cluster_occupancy": (c_int32, [_P, c_int32]),
    "rtd3_debug_cluster_prof": (c_int32, [_P, _P]),
    "rtd3_debug_cluster_mode": (c_int32, [c_int32]),
    "rtd3_debug_p2p_prof": (c_int32, [_P]),
    "rtd3_td3_target_noise": (c_int32, [c_uint64, c_uint64, _P, c_int64, _P]),
    "rtd3_tick_pre": (c_int32, [POINTER(TickStateStruct), _P]),
    "rtd3_tick_post": (c_int32, [_P, POINTER(TickStateStruct), _P, _P, c_int32, _P]),
    "rtd3_tick_run_f16": (c_int32, [_P, POINTER(TickStateStruct), c_int32, c_int32, _P, _P, c_int32, c_int64, c_uint64, _P]),
    "rtd3_eval_step": (c_int32, [_P] * 10 + [c_int32, c_int64, c_int64, _P]),
    "rtd3_eval_run_f16": (c_int32, [_P, c_int32, c_int32] + [_P] * 9 + [c_int32, c_int64, c_int64, _P, _P]),
    "rtd3_eval_starts": (c_int32, [POINTER(MtBankStruct), _P, _P, c_int64, _P, _P, _P, _P]),
    "rtd3_eval_step_episodes": (c_int32, [_P, _P, c_int64] + [_P] * 7 + [c_int32, c_int64, c_int64, _P]),
    "rtd3_eval_run_f16_episodes": (c_int32, [_P, c_int32, c_int32] + [_P] * 4 + [c_int64] + [_P] * 6 + [c_int32, c_int64, c_int64, _P, _P]),
    "rtd3_robot_baseline": (c_int32, [_P, _P, _P, _P, c_int64, _P]),
    "rtd3_robot_compose_action": (c_int32, [_P] * 10 + [c_int64, _P]),
    "rtd3_demo_lists": (c_int32, [_P, c_int64, _P, _P, _P, _P]),
    "rtd3_robot_transition": (c_int32, [_P] * 18 + [c_int64] + [_P] * 8 + [c_int64] * 2 + [_P, _P] + [_P, _P, _P, c_int64] + [c_int64, _P]),
    "rtd3_env_get_demonstration": (c_int32, [_P, POINTER(MtBankStruct), _P, _P, POINTER(CemWorkspaceStruct)] + [c_int32] * 7 + [_P, _P, _P]),
    "rtd3_robot_process_demonstration": (c_int32, [POINTER(MtBankStruct), _P, _P, _P, _P, c_int32, _P, _P, _P, _P, c_int64, c_int32, c_int32,
                                                   c_double, _P, _P, _P, _P, _P, c_int64, _P, _P]),
    "rtd3_robot_next_action_type": (c_int32, [_P] * 10 + [c_int64, _P]),
}

_lib = None


def exported_symbols():
    """Every symbol include/rtd3.h declares (kept in sync by tests/test_abi.py)."""
    return sorted(_SIGNATURES)


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                "librtd3.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`make -C residual-td3-robot-navigation_b200/csrc`. There is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the .so is stale: fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code, what=""):
    if code != 0:
        msg = lib().rtd3_last_error().decode("utf-8", "replace")
        raise Rtd3Error("librtd3 call failed (%d) %s: %s" % (code, what, msg))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return c_void_p(0)
    return c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, dtype, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("%s must be a CUDA tensor (there is no CPU path)" % name)
    if t.dtype != dtype:
        raise TypeError("%s must have dtype %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


class capture:
    """`torch.cuda.graph(graph)` with Python's cyclic garbage collector held off for the duration of the capture.  A collection
    that happens to run inside the capture can finalise objects of an earlier experiment (environments, learners: reference cycles
    keep them alive until the collector finds them) whose destructors call cudaFree - a prohibited call while a stream is
    capturing, which invalidates the capture (seen as 'operation failed due to a previous error during capture' at the next
    launch; whether it happened depended on how much garbage earlier code had produced)."""

    def __init__(self, graph):
        # thread_local: only THIS thread's unsafe CUDA calls invalidate the capture.  The default ("global") also forbids them to
        # every other thread of the process for the duration - e.g. the service threads of an NCCL communicator, which then fail.
        self._ctx = torch.cuda.graph(graph, capture_error_mode="thread_local")

    def __enter__(self):
        import gc
        gc.collect()
        self._was_enabled = gc.isenabled()
        gc.disable()
        try:
            return self._ctx.__enter__()
        except BaseException:
            if self._was_enabled:
                gc.enable()
            raise

    def __exit__(self, *exc):
        import gc
        try:
            return self._ctx.__exit__(*exc)
        finally:
            if self._was_enabled:
                gc.enable()


def launch_count():
    return int(lib().rtd3_launch_count())


def launch_count_reset():
    lib().rtd3_launch_count_reset()
