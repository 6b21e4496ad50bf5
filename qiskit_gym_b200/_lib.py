"""Loader of the C-ABI engine library (libqg_engine.so, built in-tree by csrc/Makefile).

The product path has no CPU fallback: a missing library is an ImportError, and any call that needs
the GPU returns QG_ERR_CUDA when no device is usable, which surfaces as a RuntimeError.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# QG_ENGINE_LIB: load another build of the same library (kernel A/B runs, tools/); the default is the in-tree build
LIB_PATH = os.environ.get("QG_ENGINE_LIB") or os.path.join(_HERE, "libqg_engine.so")
CSRC = os.path.join(_HERE, "csrc")

# every symbol include/qg_engine.h declares
SYMBOLS = [
    "qg_version", "qg_last_error", "qg_config_default", "qg_gate_kind_from_name", "qg_config_validate",
    "qg_config_obs_shape", "qg_config_state_len", "qg_twists_create", "qg_twists_destroy", "qg_twists_count",
    "qg_twists_obs_len", "qg_twists_act_len", "qg_twists_copy", "qg_workspace_bytes", "qg_create", "qg_destroy",
    "qg_batch", "qg_num_actions", "qg_obs_size", "qg_obs_shape", "qg_set_difficulty", "qg_get_difficulty",
    "qg_set_state", "qg_reset", "qg_snapshot", "qg_restore", "qg_step", "qg_replay", "qg_replay_host", "qg_step_host", "qg_observe", "qg_masks", "qg_read_status",
    "qg_read_metrics", "qg_read_errors", "qg_get_state_host", "qg_solution_host", "qg_search_begin",
    "qg_search_step", "qg_search_best", "qg_read_returns", "qg_reset_select", "qg_collect_step", "qg_gae", "qg_twist_gather",
    "qg_obs_words", "qg_step_bits", "qg_replay_bits", "qg_observe_bits", "qg_search_step_bits",
    "qg_policy_create", "qg_policy_create_value", "qg_policy_destroy", "qg_policy_num_actions", "qg_policy_has_value", "qg_policy_forward_bits",
    "qg_policy_forward_bits_value",
    "qg_step_slots", "qg_copy_records", "qg_mcts_begin", "qg_mcts_select", "qg_mcts_backup", "qg_mcts_root_weights", "qg_mcts_reroot", "qg_mcts_begin_keep",
    "qg_search_run",
    "qg_solutions", "qg_solutions_host", "qg_replay_host_packed", "qg_replay_host_packed_async", "qg_replay_packed", "qg_host_alloc", "qg_host_free", "qg_bind_thread_to_device",
    "qg_dlpack_obs", "qg_search_finish", "qg_nccl_unique_id", "qg_nccl_comm_create", "qg_nccl_comm_destroy",
    "qg_policy_tc_create", "qg_policy_tc_destroy", "qg_policy_tc_num_actions", "qg_policy_tc_forward_bits", "qg_policy_tc_set_mode",
    "qg_reset_select_dev", "qg_collect_step_dev", "qg_collect_step_twisted_dev", "qg_twist_bits", "qg_policy_tc_load_weights_dev",
    "qg_policy_tc_enable_training", "qg_policy_tc_generation", "qg_policy_tc_backward", "qg_set_state_grouped", "qg_search_best_grouped",
    "qg_search_observe_twisted", "qg_search_step_twisted", "qg_search_run_twisted",
    "qg_mcts_observe_twisted", "qg_mcts_begin_twisted", "qg_mcts_begin_keep_twisted", "qg_mcts_backup_twisted",
]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compiles the CUDA extension for sm_100a with nvcc (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if os.path.isfile(os.path.join(CSRC, f))] + [os.path.join(_HERE, "..", "include", "qg_engine.h")]
    stale = force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if stale:
        cmd = ["make", "-C", CSRC, f"-j{min(os.cpu_count() or 1, 8)}"] + (["-B"] if force else [])
        subprocess.check_call(cmd, stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA engine first (python -c 'import __graft_entry__ as g; g.build()' "
            "or make -C qiskit_gym_b200/csrc). There is no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    cfgp = C.POINTER(_abi.QgConfig)
    L.qg_version.restype = C.c_char_p
    L.qg_last_error.restype = C.c_char_p
    L.qg_config_default.argtypes = [cfgp, i32]
    L.qg_config_default.restype = None
    L.qg_gate_kind_from_name.argtypes = [C.c_char_p, i32]
    L.qg_config_validate.argtypes = [cfgp]
    L.qg_config_obs_shape.argtypes = [cfgp, C.POINTER(i32)]
    L.qg_config_state_len.argtypes = [cfgp]
    L.qg_config_state_len.restype = i64
    L.qg_twists_create.argtypes = [cfgp, C.POINTER(vp)]
    L.qg_twists_destroy.argtypes = [vp]
    L.qg_twists_destroy.restype = None
    for n in ("qg_twists_count", "qg_twists_obs_len", "qg_twists_act_len"):
        getattr(L, n).argtypes = [vp]
        getattr(L, n).restype = i64
    L.qg_twists_copy.argtypes = [vp, vp, vp]
    L.qg_workspace_bytes.argtypes = [cfgp, i64]
    L.qg_workspace_bytes.restype = i64
    L.qg_create.argtypes = [cfgp, i32, i64, vp, C.POINTER(vp)]
    L.qg_destroy.argtypes = [vp]
    L.qg_destroy.restype = None
    L.qg_batch.argtypes = [vp]
    L.qg_batch.restype = i64
    L.qg_num_actions.argtypes = [vp]
    L.qg_obs_size.argtypes = [vp]
    L.qg_obs_shape.argtypes = [vp, C.POINTER(i32)]
    L.qg_set_difficulty.argtypes = [vp, i32]
    L.qg_get_difficulty.argtypes = [vp]
    L.qg_set_state.argtypes = [vp, vp, i64, i64, i64, i32, vp]
    L.qg_reset.argtypes = [vp, u64, i64, vp]
    L.qg_snapshot.argtypes = [vp, vp]
    L.qg_restore.argtypes = [vp, vp]
    L.qg_step.argtypes = [vp] + [vp] * 8 + [vp]
    L.qg_replay.argtypes = [vp, i32, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    L.qg_replay_host.argtypes = [vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    L.qg_step_host.argtypes = [vp] + [vp] * 7 + [vp]
    L.qg_observe.argtypes = [vp, vp, vp, vp]
    L.qg_masks.argtypes = [vp, vp, vp]
    L.qg_read_status.argtypes = [vp, vp, vp, vp, vp, vp]
    L.qg_read_metrics.argtypes = [vp, vp, vp]
    L.qg_read_errors.argtypes = [vp, vp, vp]
    L.qg_get_state_host.argtypes = [vp, i64, vp, i64, C.POINTER(i64), vp]
    L.qg_solution_host.argtypes = [vp, i64, vp, i32, C.POINTER(i32), vp]
    L.qg_search_begin.argtypes = [vp, u64, i64, vp]
    L.qg_search_step.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp]
    L.qg_search_best.argtypes = [vp, C.POINTER(i64), C.POINTER(i64), vp]
    L.qg_read_returns.argtypes = [vp, vp, vp]
    L.qg_reset_select.argtypes = [vp, u64, i64, vp, vp]
    L.qg_collect_step.argtypes = [vp, u64, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.qg_gae.argtypes = [vp, vp, vp, vp, i32, i64, C.c_float, C.c_float, vp, vp, vp]
    L.qg_twist_gather.argtypes = [vp, vp, vp, vp, i64, i32, vp]
    L.qg_obs_words.argtypes = [vp]
    L.qg_step_bits.argtypes = [vp] + [vp] * 8 + [vp]
    L.qg_replay_bits.argtypes = [vp, i32, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    L.qg_observe_bits.argtypes = [vp, vp, vp, vp]
    L.qg_search_step_bits.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.qg_policy_create.argtypes = [i32, i32, i32, vp, vp, vp, C.POINTER(vp)]
    L.qg_policy_destroy.argtypes = [vp]
    L.qg_policy_destroy.restype = None
    L.qg_policy_num_actions.argtypes = [vp]
    L.qg_policy_forward_bits.argtypes = [vp, vp, i64, vp, vp, vp]
    L.qg_policy_create_value.argtypes = [i32, i32, i32, vp, vp, vp, vp, C.c_float, C.POINTER(vp)]
    L.qg_policy_has_value.argtypes = [vp]
    L.qg_policy_forward_bits_value.argtypes = [vp, vp, i64, vp, vp, vp, vp]
    L.qg_step_slots.argtypes = [vp, i64] + [vp] * 9 + [vp]
    L.qg_copy_records.argtypes = [vp, vp, vp, i64, vp]
    treep = C.POINTER(_abi.QgMctsTree)
    L.qg_mcts_begin.argtypes = [treep, vp, vp, vp]
    L.qg_mcts_select.argtypes = [treep, C.c_float, vp, vp, vp, vp]
    L.qg_mcts_backup.argtypes = [treep, vp, vp, vp, vp, vp]
    L.qg_mcts_root_weights.argtypes = [treep, vp, vp]
    L.qg_mcts_reroot.argtypes = [treep, vp, vp, vp, i32, vp, vp]
    L.qg_mcts_begin_keep.argtypes = [treep, vp, vp, vp, vp]
    L.qg_mcts_observe_twisted.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]
    L.qg_mcts_begin_twisted.argtypes = [treep, vp, vp, vp, i32, vp, vp]
    L.qg_mcts_begin_keep_twisted.argtypes = [treep, vp, vp, vp, vp, i32, vp, vp]
    L.qg_mcts_backup_twisted.argtypes = [treep, vp, vp, vp, vp, vp, i32, vp, vp, vp]
    L.qg_search_run.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp]
    L.qg_solutions.argtypes = [vp, i64, i64, vp, i32, vp, vp]
    L.qg_solutions_host.argtypes = [vp, i64, i64, vp, i32, vp, vp]
    L.qg_replay_host_packed.argtypes = [vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    L.qg_replay_host_packed_async.argtypes = [vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    L.qg_replay_packed.argtypes = [vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    L.qg_host_alloc.argtypes = [i32, C.c_size_t, C.POINTER(vp), C.POINTER(i32)]
    L.qg_host_free.argtypes = [vp]
    L.qg_bind_thread_to_device.argtypes = [i32]
    L.qg_dlpack_obs.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(vp)]
    L.qg_search_finish.argtypes = [vp, vp, C.POINTER(i64), C.POINTER(i32), C.POINTER(i64), C.POINTER(i32), vp, i32, C.POINTER(i32), vp]
    L.qg_nccl_unique_id.argtypes = [vp]
    L.qg_nccl_comm_create.argtypes = [vp, i32, i32, i32, C.POINTER(vp)]
    L.qg_nccl_comm_destroy.argtypes = [vp]
    L.qg_policy_tc_create.argtypes = [i32, i32, i32, vp, vp, vp, vp, C.c_float, i64, C.POINTER(vp)]
    L.qg_policy_tc_destroy.argtypes = [vp]
    L.qg_policy_tc_destroy.restype = None
    L.qg_policy_tc_num_actions.argtypes = [vp]
    L.qg_policy_tc_forward_bits.argtypes = [vp, vp, i64, vp, vp, vp, vp]
    L.qg_policy_tc_set_mode.argtypes = [vp, i32]
    L.qg_reset_select_dev.argtypes = [vp, vp, i64, vp, vp]
    L.qg_collect_step_dev.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.qg_collect_step_twisted_dev.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    L.qg_twist_bits.argtypes = [vp, vp, i64, i32, i32, i32, vp, i32, vp, vp, i64, i32, vp, vp]
    L.qg_policy_tc_load_weights_dev.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp]
    L.qg_policy_tc_enable_training.argtypes = [vp]
    L.qg_policy_tc_generation.argtypes = [vp]
    L.qg_policy_tc_generation.restype = i64
    L.qg_policy_tc_backward.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp, vp, vp]
    L.qg_set_state_grouped.argtypes = [vp, vp, i64, i64, i64, vp]
    L.qg_search_best_grouped.argtypes = [vp, i64, i64, vp, vp, i32, vp, vp]
    L.qg_search_observe_twisted.argtypes = [vp, vp, vp, i32, vp, vp]
    L.qg_search_step_twisted.argtypes = [vp, vp, i32, vp, vp, vp, i32, vp, vp, vp, vp]
    L.qg_search_run_twisted.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, vp, i32, vp, vp]
    _lib = L
    return L


def check(rc: int) -> int:
    """Maps a negative status to the exception the reference's Python surface would raise."""
    if rc >= 0:
        return rc
    msg = lib().qg_last_error().decode()
    if rc == _abi.QG_ERR_CUDA:
        raise RuntimeError(f"CUDA engine error: {msg}")
    if rc == _abi.QG_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise ValueError(msg)
