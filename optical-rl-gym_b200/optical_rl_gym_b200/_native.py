"""ctypes binding of liborlg.so (include/orlg.h).  No torch types cross this boundary:
only raw device pointers (tensor.data_ptr()) and the raw cudaStream_t handle."""
import ctypes as C
import os

import numpy as np

from . import build as _build

KIND = {"RWA-v0": 0, "RMSA-v0": 1, "DeepRMSA-v0": 2, "RMCSA-v0": 3}
TRAFFIC_TRACE, TRAFFIC_PHILOX = 0, 1
OBS_F32, OBS_F64 = 0, 1
HEURISTICS = {"shortest_path_first_fit": 0, "sp_ff": 0, "sp": 0,
              "shortest_available_path_first_fit": 1, "sap_ff": 1, "sap": 1,
              "shortest_available_path_best_modulation_first_core_first_fit": 1,
              "least_loaded_path_first_fit": 2, "llp_ff": 2,
              "shortest_available_path_last_fit": 3, "sap_lf": 3}
ERR_TRACE_EXHAUSTED, ERR_HEAP_OVERFLOW, ERR_NO_SUCH_PATH, ERR_LOCKSTEP, ERR_STATS_ORDER, ERR_TRACE_RANGE = 1, 2, 4, 8, 16, 32
MAX_BIT_RATE = 1023       # bit rates (Gb/s) are tabulated up to here (orlg_api.cu)


class Config(C.Structure):
    _fields_ = [("kind", C.c_int32), ("num_envs", C.c_int32), ("env_id_base", C.c_int64),
                ("num_slots", C.c_int32), ("num_cores", C.c_int32), ("j", C.c_int32),
                ("episode_length", C.c_int32), ("allow_rejection", C.c_int32),
                ("bit_rate_lo", C.c_int32), ("bit_rate_hi", C.c_int32), ("traffic", C.c_int32),
                ("obs_dtype", C.c_int32), ("auto_reset", C.c_int32), ("heap_capacity", C.c_int32),
                ("seed", C.c_uint64), ("channel_width", C.c_double), ("mean_holding", C.c_double),
                ("mean_iat", C.c_double), ("worst_xt", C.c_double)]


class KernelInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("wide", "fast", "hot", "rollout_kernel", "rollout_lanes", "link_template",
                                         "last_rollout_persistent")]


class PolicyDraw(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("counter_dev", C.c_void_p), ("counter", C.c_uint32), ("deterministic", C.c_int32),
                ("row_id_base", C.c_int64)]


class InfoOut(C.Structure):
    """orlg_info_out: device pointers of the per-step info outputs of a rollout (None = not written)."""
    _fields_ = [(n, C.c_void_p) for n in ("counters_dev", "stats_dev", "bit_rate_blocking_dev", "action_probability_dev")]


class Tables(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("num_nodes", "num_links", "k_paths", "num_paths", "num_mods", "num_bit_rates")] + [
        (n, C.c_void_p) for n in ("pair_first", "pair_count", "path_hops", "path_se", "path_mod", "path_link_ptr",
                                  "path_links", "path_length", "mod_se", "mod_osnr", "mod_xt", "node_prob",
                                  "bit_rates", "bit_rate_prob", "link_order")]


REQUEST_DTYPE = np.dtype([("arrival", np.float64), ("holding", np.float64), ("src", np.int32), ("dst", np.int32),
                          ("bit_rate", np.int32), ("reserved", np.int32)])

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Loads (building if stale and nvcc is present) the CUDA library.  There is no CPU fallback:
    a missing library is a hard error."""
    global _lib
    if _lib is not None:
        return _lib
    try:
        path = _build.build()
    except Exception as exc:  # noqa: BLE001
        path = _build.LIB
        if not os.path.exists(path):
            raise NativeError("liborlg.so is missing and could not be built (%s); run __graft_entry__.build()" % exc)
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.orlg_last_error.restype = C.c_char_p
    L.orlg_create.argtypes = [C.POINTER(Config), C.POINTER(Tables), i32, C.POINTER(vp)]
    L.orlg_destroy.argtypes = [vp]
    for name in ("orlg_action_dim", "orlg_obs_dim", "orlg_mask_words", "orlg_heap_capacity"):
        getattr(L, name).argtypes = [vp]
    L.orlg_state_bytes.argtypes = [vp]
    L.orlg_state_bytes.restype = i64
    L.orlg_kernel_info.argtypes = [vp, C.POINTER(KernelInfo)]
    L.orlg_set_trace.argtypes = [vp, vp, i64]
    L.orlg_seed.argtypes = [vp, C.c_uint64]
    L.orlg_reset.argtypes = [vp, i32, vp, vp]
    L.orlg_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.orlg_observation.argtypes = [vp, vp, vp]
    L.orlg_observation_int.argtypes = [vp, vp, vp]
    L.orlg_heuristic.argtypes = [vp, i32, vp, vp]
    L.orlg_random_actions.argtypes = [vp, vp, vp]
    L.orlg_get_counters.argtypes = [vp, vp, vp]
    L.orlg_get_requests.argtypes = [vp, vp, vp, vp]
    L.orlg_export_state.argtypes = [vp, vp, vp, vp, vp, vp]
    L.orlg_error_flags.argtypes = [vp, vp, vp]
    L.orlg_reduce_counters.argtypes = [vp, vp, vp]
    L.orlg_enable_stats.argtypes = [vp, vp]
    L.orlg_enable_link_stats.argtypes = [vp, i32]
    L.orlg_link_stats.argtypes = [vp, vp, vp, vp]
    L.orlg_num_bit_rates.argtypes = [vp]
    L.orlg_bit_rate_blocking.argtypes = [vp, vp, vp]
    L.orlg_matrix_obs_dim.argtypes = [vp]
    L.orlg_matrix_observation.argtypes = [vp, vp, vp]
    L.orlg_path_only_first_fit.argtypes = [vp, vp, vp, vp]
    L.orlg_action_hist_dim.argtypes = [vp]
    L.orlg_action_probability.argtypes = [vp, vp, vp]
    L.orlg_rollout.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    L.orlg_rollout_info.argtypes = [vp, i32, i32, vp, vp, vp, vp, C.POINTER(InfoOut), vp]
    L.orlg_state_save_bytes.argtypes = [vp]
    L.orlg_state_save_bytes.restype = i64
    L.orlg_state_save.argtypes = [vp, vp, vp]
    L.orlg_state_load.argtypes = [vp, vp, vp]
    L.orlg_policy_create.argtypes = [i32, i32, i32, i32, i32, vp, vp, C.POINTER(vp)]
    L.orlg_policy_act.argtypes = [vp, vp, i32, vp, vp, vp]
    L.orlg_policy_destroy.argtypes = [vp]
    L.orlg_policy_sample.argtypes = [vp, vp, i32, C.POINTER(PolicyDraw), vp, vp, vp, vp]
    L.orlg_rollout_policy.argtypes = [vp, i32, vp, vp, C.c_uint64, i32, vp, vp, vp, vp, vp, vp, vp]
    L.orlg_rollout_policy_info.argtypes = [vp, i32, vp, vp, C.c_uint64, i32, vp, vp, vp, vp, vp, vp, C.POINTER(InfoOut), vp]
    L.orlg_action_mask_dim.argtypes = [vp]
    L.orlg_action_masks.argtypes = [vp, vp, vp]
    L.orlg_policy_sample_masked.argtypes = [vp, vp, i32, C.POINTER(PolicyDraw), vp, vp, vp, vp, vp]
    L.orlg_rollout_policy_masked.argtypes = [vp, i32, vp, vp, C.c_uint64, i32, vp, vp, vp, vp, vp, vp, vp, C.POINTER(InfoOut), vp]
    L.orlg_policy_create_wide.argtypes = [i32, i32, i32, i32, i32, vp, vp, C.POINTER(vp)]
    L.orlg_policy_tile_groups.argtypes = [vp]
    L.orlg_policy_create_matrix.argtypes = [i32, i32, i32, i32, i32, i32, i32, vp, vp, C.POINTER(vp)]
    L.orlg_matrix_obs_words.argtypes = [vp]
    L.orlg_matrix_observation_packed.argtypes = [vp, vp, vp]
    L.orlg_request_index.argtypes = [vp]
    L.orlg_request_index.restype = i64
    L.orlg_rollout_packed.argtypes = [vp, i32, i32, vp, vp, vp]
    L.orlg_expand_packed.argtypes = [vp, i64, i32, i32, vp, vp, vp, vp, i32]
    L.orlg_rollout_host.argtypes = [vp, i32, i32, vp, vp, vp, vp, i32, i32, vp]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise NativeError("liborlg: %s (code %d)" % (lib().orlg_last_error().decode(), rc))


EXPORTED = ["orlg_create", "orlg_destroy", "orlg_last_error", "orlg_version", "orlg_action_dim", "orlg_obs_dim",
            "orlg_mask_words", "orlg_heap_capacity", "orlg_state_bytes", "orlg_kernel_info", "orlg_seed", "orlg_set_trace", "orlg_reset", "orlg_step",
            "orlg_observation", "orlg_observation_int", "orlg_heuristic", "orlg_random_actions", "orlg_get_counters",
            "orlg_get_requests", "orlg_export_state", "orlg_error_flags", "orlg_reduce_counters", "orlg_enable_stats",
            "orlg_num_bit_rates", "orlg_bit_rate_blocking", "orlg_matrix_obs_dim", "orlg_matrix_observation",
            "orlg_path_only_first_fit", "orlg_rollout", "orlg_state_save_bytes", "orlg_state_save", "orlg_state_load", "orlg_policy_create", "orlg_policy_act", "orlg_policy_destroy", "orlg_rollout_packed", "orlg_expand_packed", "orlg_rollout_host", "orlg_action_hist_dim", "orlg_action_probability",
            "orlg_enable_link_stats", "orlg_link_stats", "orlg_policy_sample", "orlg_rollout_policy", "orlg_request_index",
            "orlg_rollout_info", "orlg_rollout_policy_info", "orlg_action_mask_dim", "orlg_action_masks",
            "orlg_policy_sample_masked", "orlg_rollout_policy_masked", "orlg_policy_create_wide", "orlg_policy_tile_groups",
            "orlg_policy_create_matrix", "orlg_matrix_obs_words", "orlg_matrix_observation_packed"]
