"""ctypes binding of libnfsp_b200.so (the C ABI declared in include/nfsp_b200.h).

There is no fallback: if the shared library is missing or a call fails, this raises.
PyTorch is used only to own device memory and streams; every pointer crossing this boundary is a
raw device address.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libnfsp_b200.so")

RULES_LEGACY, RULES_NFSP = 0, 1
OBS_DIM, ACTIONS, HIDDEN, NET_PARAMS = 30, 3, 64, 2179
EXPORT_FIELDS, LEGACY_EXPORT_FIELDS, STATS_FIELDS = 24, 14, 16

# every symbol include/nfsp_b200.h declares (tests/test_boundary.py checks the two lists agree)
SYMBOLS = [
    "nfsp_version", "nfsp_last_error", "nfsp_device_info",
    "nfsp_env_create", "nfsp_env_destroy", "nfsp_env_num_games", "nfsp_env_rules", "nfsp_env_step_counter",
    "nfsp_env_set_step_counter", "nfsp_env_state_ptr", "nfsp_env_kernel_error", "nfsp_env_save_state", "nfsp_env_load_state",
    "nfsp_env_reset", "nfsp_env_set_hands", "nfsp_env_step", "nfsp_env_do_action", "nfsp_fsm_image", "nfsp_legacy_fsm_image", "nfsp_rollout_image", "nfsp_env_observe", "nfsp_env_export",
    "nfsp_legacy_reset", "nfsp_legacy_set_hands", "nfsp_legacy_step", "nfsp_legacy_get_new_state",
    "nfsp_legacy_rollout", "nfsp_legacy_export",
    "nfsp_expand_obs",
    "nfsp_act_set_weights", "nfsp_act_set_weights_from_host", "nfsp_act_forward", "nfsp_act_forward_tc", "nfsp_rollout", "nfsp_rollout_with_weights", "nfsp_rollout_runs", "nfsp_rollout_tune", "nfsp_rollout_profile",
    "nfsp_ring_insert", "nfsp_reservoir_insert", "nfsp_insert_multi", "nfsp_ring_insert_multi", "nfsp_reservoir_insert_multi", "nfsp_sample_indices", "nfsp_sample_minibatches", "nfsp_gather_rl", "nfsp_gather_sl",
    "nfsp_learner_grads", "nfsp_learner_fit", "nfsp_learner_fit_runs", "nfsp_learner_fit_peers", "nfsp_sgd_apply",
    "nfsp_peer_buffer_create", "nfsp_peer_buffer_open", "nfsp_peer_buffer_close", "nfsp_peer_buffer_destroy",
]


class RolloutIO(C.Structure):
    _fields_ = [("d_rl", C.c_void_p * 2), ("d_sl", C.c_void_p * 2), ("cap_rl", C.c_int64), ("cap_sl", C.c_int64),
                ("n_segments", C.c_int32), ("d_counts", C.c_void_p), ("d_stats", C.c_void_p), ("d_trace", C.c_void_p), ("d_vec", C.c_void_p),
                ("d_forced_vec", C.c_void_p), ("variant", C.c_int32), ("reserve_sms", C.c_int32),
                ("d_ring", C.c_void_p * 2), ("d_ring_total", C.c_void_p * 2), ("ring_cap", C.c_int64),
                ("epsilon_per_player", C.c_int32), ("epsilon_p1", C.c_double)]


class InsertReq(C.Structure):
    _fields_ = [("d_mem", C.c_void_p), ("cap", C.c_int64), ("d_total", C.c_void_p), ("d_scratch", C.c_void_p),
                ("d_recs", C.c_void_p), ("d_counts", C.c_void_p), ("n_segments", C.c_int32), ("seg_cap", C.c_int64),
                ("seed", C.c_uint64), ("mode", C.c_int32), ("reservoir", C.c_int32)]


INSERT_SCRATCH_WORDS, RESERVOIR_SLOT_BYTES = 4, 32  # NFSP_INSERT_SCRATCH_WORDS, NFSP_RESERVOIR_SLOT_BYTES


MAX_PEERS, PEER_BUF_FLOATS = 8, 279552  # NFSP_MAX_PEERS, NFSP_PEER_BUF_FLOATS


class Peers(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("d_buf", C.c_void_p * MAX_PEERS), ("epoch0", C.c_uint32),
                ("d_err", C.c_void_p), ("d_mc", C.c_void_p)]


MAX_RUNS, MAX_SAMPLE_REQS = 32, 128  # NFSP_MAX_RUNS, NFSP_MAX_SAMPLE_REQS (= 4 * NFSP_MAX_RUNS)
FIT_ROWS_MAX_MINIBATCH, FIT_ROWS_MAX_STEP = 256, 64  # NFSP_FIT_ROWS_MAX_MINIBATCH, NFSP_FIT_ROWS_MAX_STEP (row-parallel fit)


class SampleReq(C.Structure):
    _fields_ = [("d_mem", C.c_void_p), ("d_total", C.c_void_p), ("cap", C.c_int64), ("seed", C.c_uint64),
                ("call_idx", C.c_uint64), ("is_ring", C.c_int32), ("d_out", C.c_void_p), ("d_rec_out", C.c_void_p)]


class LearnerIO(C.Structure):
    _fields_ = [("d_weights", C.c_void_p), ("d_target_weights", C.c_void_p), ("d_rl", C.c_void_p * 2),
                ("d_rl_idx", C.c_void_p * 2), ("d_sl", C.c_void_p * 2), ("d_sl_idx", C.c_void_p * 2),
                ("row0", C.c_int32), ("rows", C.c_int32), ("gamma", C.c_float), ("net_mask", C.c_int32),
                ("terminal_bootstraps", C.c_int32), ("others_to_target", C.c_int32), ("d_grad", C.c_void_p), ("d_stats", C.c_void_p)]


class NfspError(RuntimeError):
    pass


_lib = None


def lib():
    """Loads libnfsp_b200.so once.  Raises if it has not been built (python __graft_entry__.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NfspError("libnfsp_b200.so is not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'`; "
                        "there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i8p = C.c_void_p, C.c_void_p
    L.nfsp_version.restype = C.c_int
    L.nfsp_last_error.restype = C.c_char_p
    L.nfsp_device_info.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p,
                                   C.c_int]
    L.nfsp_env_create.argtypes = [C.c_int, C.c_int64, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(vp)]
    L.nfsp_env_destroy.argtypes = [vp]
    L.nfsp_env_num_games.argtypes = [vp]
    L.nfsp_env_num_games.restype = C.c_int64
    L.nfsp_env_rules.argtypes = [vp]
    L.nfsp_env_step_counter.argtypes = [vp]
    L.nfsp_env_step_counter.restype = C.c_uint64
    L.nfsp_env_set_step_counter.argtypes = [vp, C.c_uint64]
    L.nfsp_env_state_ptr.argtypes = [vp]
    L.nfsp_env_state_ptr.restype = vp
    L.nfsp_env_kernel_error.argtypes = [vp, C.POINTER(C.c_uint32)]
    L.nfsp_rollout_tune.argtypes = [vp, C.c_int, C.c_int]
    L.nfsp_rollout_profile.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.nfsp_env_save_state.argtypes = [vp, vp, vp]
    L.nfsp_env_load_state.argtypes = [vp, vp, vp]
    L.nfsp_env_reset.argtypes = [vp, i8p, C.c_double, vp]
    L.nfsp_env_set_hands.argtypes = [vp, i8p, i8p, i8p, vp]
    L.nfsp_env_step.argtypes = [vp, i8p, i8p, C.c_int, C.c_int, C.c_double, vp, vp]
    L.nfsp_env_do_action.argtypes = [vp, i8p, i8p, i8p, vp]
    L.nfsp_fsm_image.argtypes = [vp, C.c_int]
    L.nfsp_legacy_fsm_image.argtypes = [vp, C.c_int, vp]
    L.nfsp_rollout_image.argtypes = [vp, C.c_int]
    L.nfsp_env_observe.argtypes = [vp, i8p, C.c_int, vp, vp, vp, vp, vp, vp]
    L.nfsp_env_export.argtypes = [vp, vp, vp]
    L.nfsp_legacy_reset.argtypes = [vp, vp]
    L.nfsp_legacy_set_hands.argtypes = [vp, i8p, vp]
    L.nfsp_legacy_step.argtypes = [vp, i8p, i8p, C.c_int, vp]
    L.nfsp_legacy_get_new_state.argtypes = [vp, i8p, C.c_int, vp, vp]
    L.nfsp_legacy_rollout.argtypes = [vp, i8p, C.c_int, vp, vp]
    L.nfsp_legacy_export.argtypes = [vp, vp, vp]
    L.nfsp_expand_obs.argtypes = [vp, C.c_int64, vp, vp]
    L.nfsp_act_set_weights.argtypes = [vp, vp, vp]
    L.nfsp_act_set_weights_from_host.argtypes = [vp, vp, vp, vp]
    L.nfsp_act_forward.argtypes = [vp, vp, i8p, C.c_int64, vp, vp]
    L.nfsp_act_forward_tc.argtypes = [vp, vp, i8p, C.c_int64, vp, vp]
    L.nfsp_rollout.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.POINTER(RolloutIO), vp]
    L.nfsp_rollout_with_weights.argtypes = [vp, vp, vp, C.c_int, C.c_double, C.c_double, C.POINTER(RolloutIO), vp]
    L.nfsp_rollout_runs.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                    C.POINTER(RolloutIO), C.POINTER(vp), vp]
    L.nfsp_ring_insert.argtypes = [vp, C.c_int64, vp, vp, vp, C.c_int, C.c_int64, vp, vp]
    L.nfsp_reservoir_insert.argtypes = [vp, C.c_int64, vp, vp, vp, C.c_int, C.c_int64, C.c_uint64, C.c_int, vp, vp]
    L.nfsp_insert_multi.argtypes = [C.POINTER(InsertReq), C.c_int, vp]
    L.nfsp_ring_insert_multi.argtypes = [C.POINTER(InsertReq), C.c_int, vp]
    L.nfsp_reservoir_insert_multi.argtypes = [C.POINTER(InsertReq), C.c_int, vp]
    L.nfsp_sample_indices.argtypes = [C.c_uint64, C.c_uint64, vp, C.c_int64, C.c_int, C.c_int, vp, vp, vp]
    L.nfsp_sample_minibatches.argtypes = [C.POINTER(SampleReq), C.c_int, C.c_int, vp, vp, vp]
    L.nfsp_gather_rl.argtypes = [vp, vp, C.c_int, vp, vp, vp, vp, vp, vp]
    L.nfsp_gather_sl.argtypes = [vp, vp, C.c_int, vp, vp, vp]
    L.nfsp_learner_grads.argtypes = [C.POINTER(LearnerIO), vp]
    L.nfsp_learner_fit.argtypes = [C.POINTER(LearnerIO), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), vp, vp]
    L.nfsp_learner_fit_runs.argtypes = [C.POINTER(LearnerIO), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                        C.POINTER(vp), vp]
    L.nfsp_learner_fit_peers.argtypes = [C.POINTER(LearnerIO), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), vp,
                                         C.POINTER(Peers), vp]
    L.nfsp_sgd_apply.argtypes = [vp, vp, C.POINTER(C.c_float * 4), C.c_float, vp]
    L.nfsp_peer_buffer_create.argtypes = [C.c_int, C.POINTER(vp), C.c_char_p]
    L.nfsp_peer_buffer_open.argtypes = [C.c_int, C.c_char_p, C.POINTER(vp)]
    L.nfsp_peer_buffer_close.argtypes = [C.c_int, vp]
    L.nfsp_peer_buffer_destroy.argtypes = [C.c_int, vp]
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise NfspError("libnfsp_b200 error %d: %s" % (rc, lib().nfsp_last_error().decode("utf-8", "replace")))
