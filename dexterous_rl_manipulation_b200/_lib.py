"""ctypes binding of include/dexsim.h (libdexsim_b200.so).

There is no fallback: if the shared library is missing or fails to load, importing the
product raises.  Nothing here touches ``oracle/``.
"""
import ctypes as C
import os

import numpy as _np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DEXSIM_LIB_PATH") or os.path.join(HERE, "libdexsim_b200.so")   # env override: kernel experiments only

ABI_VERSION = 5
NJ, NF, OBS = 15, 5, 45
NCOUNTERS = 18
MAX_GROUPS = 256
ROW_JP, ROW_JV, ROW_OP, ROW_QUAT, ROW_OV, ROW_CONTACT = 0, 15, 30, 33, 37, 40
POLICY_EXTERNAL, POLICY_RANDOM, POLICY_HEURISTIC, POLICY_LEARNER = 0, 1, 2, 3
LABEL_NONE = 255
CNT_EPISODES, CNT_SUCCESSES, CNT_SUM_STEPS, CNT_SUM_FINAL_CONTACTS = 0, 1, 2, 3
CNT_LABEL_METRICS, CNT_LABEL_TAXONOMY, CNT_VAR_TIES, CNT_SUM_STEPS_SQ = 4, 10, 16, 17
RNG_STREAM_DYN, RNG_STREAM_OBS = 2, 3
EPISODE_RECORD_DTYPE = _np.dtype([("env_gid", "u4"), ("episode", "u4"), ("steps", "i4"), ("success", "u1"),
                                  ("final_contacts", "u1"), ("label_metrics", "u1"), ("label_taxonomy", "u1"),
                                  ("episode_reward", "f8"), ("t_end", "u4"), ("var_tie", "u4")])
HOST_SKIP_QUAT, HOST_ASYNC, HOST_PACKED_CONTACTS, HOST_EXPAND_CONTACTS, HOST_STATIC_ROWS = 1, 2, 4, 8, 16
HOST_ZERO_COPY = 32
SCHED_WORDS = 64
STEP_REVERSE_TILES = 1
STEP_HOST_ALL_ROWS = 2
ROLLOUT_NO_DYN_NOISE = 1
ACT_RELU, ACT_TANH = 0, 1
MLP_MAX_WIDTH = 64

# value strings of FailureType (evaluation/metrics.py:15-22) / FailureMode
# (evaluation/failure_taxonomy.py:14-26) in enum declaration order = device label codes
LABELS_METRICS = ("slippage", "unstable_contacts", "misaligned_grasp", "timeout", "object_dropped",
                  "insufficient_contacts")
LABELS_TAXONOMY = ("slippage", "unstable_grasp", "misalignment", "timeout", "object_dropped",
                   "insufficient_contacts")


class DexsimState(C.Structure):
    _fields_ = [("n", C.c_int64), ("ld", C.c_int64), ("obs", C.c_void_p), ("op64", C.c_void_p),
                ("thr", C.c_void_p), ("damp", C.c_void_p), ("step_count", C.c_void_p), ("cmask", C.c_void_p),
                ("size", C.c_void_p), ("mass", C.c_void_p), ("friction", C.c_void_p), ("episode", C.c_void_p),
                ("ep_return", C.c_void_p), ("ep_stats", C.c_void_p)]


class DexsimParams(C.Structure):
    _fields_ = [("w_distance", C.c_double), ("w_contact", C.c_double), ("w_closure", C.c_double),
                ("w_stability", C.c_double), ("reward_type", C.c_int32), ("max_episode_steps", C.c_int32),
                ("success_threshold", C.c_int32), ("auto_reset", C.c_int32), ("respawn", C.c_int32),
                ("success_is_terminated", C.c_int32), ("loop_max_steps", C.c_int32), ("num_groups", C.c_int32),
                ("seed", C.c_uint64), ("env_gid0", C.c_int64)]


class DexsimGroup(C.Structure):
    _fields_ = [("size", C.c_double), ("mass", C.c_double), ("friction", C.c_double),
                ("size_lo", C.c_double), ("size_hi", C.c_double), ("size_ranged", C.c_int32), ("pad0_", C.c_int32),
                ("mass_lo", C.c_double), ("mass_hi", C.c_double), ("mass_ranged", C.c_int32), ("pad1_", C.c_int32),
                ("fric_lo", C.c_double), ("fric_hi", C.c_double), ("fric_ranged", C.c_int32), ("pad2_", C.c_int32),
                ("spawn_lo", C.c_double * 3), ("spawn_hi", C.c_double * 3),
                ("sigma_obs", C.c_float), ("sigma_dyn", C.c_float)]


class DexsimStepIO(C.Structure):
    _fields_ = [("action", C.c_void_p), ("action_layout", C.c_int32), ("flags", C.c_int32),
                ("dyn_noise", C.c_void_p), ("obs_noise", C.c_void_p), ("noisy_obs", C.c_void_p),
                ("reward", C.c_void_p), ("reward_comps", C.c_void_p), ("terminated", C.c_void_p),
                ("truncated", C.c_void_p), ("num_contacts", C.c_void_p), ("finished", C.c_void_p),
                ("counters", C.c_void_p), ("ret_sums", C.c_void_p), ("reward64", C.c_void_p),
                ("sigma_dyn", C.c_float), ("sigma_obs", C.c_float), ("sched", C.c_void_p), ("host_static_rows", C.c_void_p),
                ("host_cmask", C.c_void_p)]


class DexsimEpisodeRecord(C.Structure):
    _fields_ = [("env_gid", C.c_uint32), ("episode", C.c_uint32), ("steps", C.c_int32), ("success", C.c_uint8),
                ("final_contacts", C.c_uint8), ("label_metrics", C.c_uint8), ("label_taxonomy", C.c_uint8),
                ("episode_reward", C.c_double), ("t_end", C.c_uint32), ("var_tie", C.c_uint32)]


class DexsimRolloutIO(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("dyn_noise", C.c_void_p), ("counters", C.c_void_p), ("ret_sums", C.c_void_p),
                ("ep_log", C.c_void_p), ("ep_log_count", C.c_void_p), ("ep_log_capacity", C.c_int64),
                ("hist", C.c_void_p), ("hist_steps", C.c_int64), ("step_base", C.c_int64),
                ("one_episode", C.c_int32), ("flags", C.c_int32),
                ("learner_mean", C.c_void_p), ("learner_best", C.c_void_p), ("learner_act_noise", C.c_void_p),
                ("learner_upd_noise", C.c_void_p), ("learner_exploration", C.c_float), ("learner_lr", C.c_float),
                ("learner_clip", C.c_float), ("pad2_", C.c_int32)]


class DexsimTrajectory(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("action", C.c_void_p), ("reward", C.c_void_p), ("terminated", C.c_void_p),
                ("truncated", C.c_void_p), ("finished", C.c_void_p), ("capacity", C.c_int64)]


class DexsimMlpPolicy(C.Structure):
    _fields_ = [("params", C.c_void_p), ("num_hidden", C.c_int32), ("hidden", C.c_int32 * 2), ("activation", C.c_int32),
                ("action_std", C.c_void_p)]


class DexsimPolicyRecord(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("raw_action", C.c_void_p), ("log_prob", C.c_void_p)]


class DexsimEpisodeSummary(C.Structure):
    _fields_ = [("success", C.c_int32), ("episode_steps", C.c_int32), ("num_contacts", C.c_int32),
                ("final_contacts", C.c_int32), ("hist_len", C.c_int32), ("max_count", C.c_int32),
                ("sum_counts", C.c_int32), ("sum_sq_counts", C.c_int32), ("first5_sum", C.c_int32),
                ("last5_sum", C.c_int32)]


EXPORTS = (
    "dexsim_version", "dexsim_error_string", "dexsim_sizeof_state", "dexsim_sizeof_params",
    "dexsim_sizeof_group", "dexsim_sizeof_step_io", "dexsim_sizeof_rollout_io", "dexsim_sizeof_episode_record",
    "dexsim_device_info", "dexsim_set_step_impl", "dexsim_set_step_tile", "dexsim_set_rollout_impl", "dexsim_reset_predrawn",
    "dexsim_reset_philox", "dexsim_step", "dexsim_rollout", "dexsim_rollout_record", "dexsim_rollout_record_final",
    "dexsim_sizeof_trajectory", "dexsim_sizeof_mlp_policy", "dexsim_rollout_mlp", "dexsim_mlp_policy_mean",
    "dexsim_sizeof_policy_record", "dexsim_rollout_mlp_record", "dexsim_gae",
    "dexsim_fill_policy_actions", "dexsim_fill_mlp_actions",
    "dexsim_fill_normal", "dexsim_classify_summary", "dexsim_step_host", "dexsim_pack_env", "dexsim_pack_env_tagged", "dexsim_step_single",
    "dexsim_step_final", "dexsim_step_host_final", "dexsim_step_next_reset",
    "dexsim_expand_contact_rows",
    "dexsim_host_zero_copy_steps",
)

_lib = None


class DexsimError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        msg = lib().dexsim_error_string(code).decode()
        super().__init__(f"{where} failed with code {code}: {msg}")


def lib():
    """Load libdexsim_b200.so (once).  Raises if it is missing -- there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m dexterous_rl_manipulation_b200.build` "
            "(nvcc, sm_100a).  The simulator has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.dexsim_version.restype = C.c_int
    L.dexsim_error_string.restype = C.c_char_p
    L.dexsim_error_string.argtypes = [C.c_int]
    for name in ("dexsim_sizeof_state", "dexsim_sizeof_params", "dexsim_sizeof_group", "dexsim_sizeof_step_io",
                 "dexsim_sizeof_rollout_io", "dexsim_sizeof_episode_record", "dexsim_sizeof_trajectory",
                 "dexsim_sizeof_mlp_policy", "dexsim_sizeof_policy_record"):
        getattr(L, name).restype = C.c_int
    L.dexsim_device_info.argtypes = [C.POINTER(C.c_int)] * 3
    L.dexsim_set_step_impl.argtypes = [C.c_int]
    L.dexsim_set_step_tile.argtypes = [C.c_int]
    L.dexsim_set_rollout_impl.argtypes = [C.c_int]
    L.dexsim_reset_predrawn.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, vp, vp, vp, vp, vp]
    L.dexsim_reset_philox.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, vp, i32, vp]
    L.dexsim_step.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, C.POINTER(DexsimStepIO), vp]
    L.dexsim_step_final.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, C.POINTER(DexsimStepIO), vp, vp]
    L.dexsim_step_next_reset.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, C.POINTER(DexsimStepIO), vp]
    L.dexsim_rollout.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, i32, i32,
                                 C.POINTER(DexsimRolloutIO), vp]
    L.dexsim_rollout_record.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, i32, i32,
                                        C.POINTER(DexsimRolloutIO), C.POINTER(DexsimTrajectory), vp]
    L.dexsim_rollout_record_final.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, i32, i32,
                                              C.POINTER(DexsimRolloutIO), C.POINTER(DexsimTrajectory), vp, vp]
    L.dexsim_rollout_mlp.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, i32, C.POINTER(DexsimRolloutIO),
                                     C.POINTER(DexsimMlpPolicy), C.POINTER(DexsimTrajectory), vp, vp]
    L.dexsim_rollout_mlp_record.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, i32,
                                            C.POINTER(DexsimRolloutIO), C.POINTER(DexsimMlpPolicy),
                                            C.POINTER(DexsimTrajectory), vp, C.POINTER(DexsimPolicyRecord), vp]
    L.dexsim_gae.argtypes = [C.POINTER(DexsimTrajectory), i64, i64, i32, vp, vp, C.c_float, C.c_float, vp, vp, vp]
    L.dexsim_mlp_policy_mean.argtypes = [C.POINTER(DexsimMlpPolicy), vp, i64, i64, vp, vp]
    L.dexsim_fill_policy_actions.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), i32, vp, vp]
    L.dexsim_fill_mlp_actions.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp,
                                          C.POINTER(DexsimMlpPolicy), vp, vp]
    L.dexsim_fill_normal.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), i32, i32, C.c_float, vp, vp]
    L.dexsim_pack_env.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimStepIO), i64, i32, vp, vp]
    L.dexsim_pack_env_tagged.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimStepIO), i64, i32, vp, C.c_double, vp]
    L.dexsim_step_single.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, C.POINTER(DexsimStepIO), vp,
                                     C.c_double, vp]
    L.dexsim_classify_summary.argtypes = [C.POINTER(DexsimEpisodeSummary), vp, i32, i32, C.POINTER(i32),
                                          C.POINTER(i32), C.POINTER(i32)]
    L.dexsim_step_host.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, C.POINTER(DexsimStepIO),
                                   vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
    L.dexsim_step_host_final.argtypes = [C.POINTER(DexsimState), C.POINTER(DexsimParams), vp, vp, C.POINTER(DexsimStepIO),
                                         vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
    L.dexsim_expand_contact_rows.argtypes = [vp, vp, i64, i64]
    L.dexsim_host_zero_copy_steps.argtypes = []
    L.dexsim_host_zero_copy_steps.restype = C.c_int64
    for name in EXPORTS:
        fn = getattr(L, name)          # raises AttributeError if a declared symbol is not exported
        if name not in ("dexsim_error_string", "dexsim_host_zero_copy_steps"):
            fn.restype = C.c_int
    if L.dexsim_version() != ABI_VERSION:
        raise ImportError(f"libdexsim_b200.so ABI {L.dexsim_version()} != binding ABI {ABI_VERSION}")
    assert L.dexsim_sizeof_state() == C.sizeof(DexsimState)
    assert L.dexsim_sizeof_params() == C.sizeof(DexsimParams)
    assert L.dexsim_sizeof_group() == C.sizeof(DexsimGroup)
    assert L.dexsim_sizeof_step_io() == C.sizeof(DexsimStepIO)
    assert L.dexsim_sizeof_rollout_io() == C.sizeof(DexsimRolloutIO)
    assert L.dexsim_sizeof_episode_record() == C.sizeof(DexsimEpisodeRecord) == 32
    assert L.dexsim_sizeof_trajectory() == C.sizeof(DexsimTrajectory)
    assert L.dexsim_sizeof_mlp_policy() == C.sizeof(DexsimMlpPolicy)
    assert L.dexsim_sizeof_policy_record() == C.sizeof(DexsimPolicyRecord)
    _ = i64
    _lib = L
    return L


def set_step_impl(impl):
    """'auto' | 'register' | 'tma' -- which step kernel dexsim_step launches (tests / profiling)."""
    code = {"auto": 0, "register": 1, "tma": 2}[impl]
    check(lib().dexsim_set_step_impl(code), "dexsim_set_step_impl")


def set_step_tile(tile):
    """'auto' | 'narrow' | 'wide' -- tile width of the pipelined step kernel (tests / profiling)."""
    check(lib().dexsim_set_step_tile({"auto": 0, "narrow": 1, "wide": 2}[tile]), "dexsim_set_step_tile")


def set_rollout_impl(impl):
    """'auto' | 'thread' | 'split' -- which fused-rollout kernel dexsim_rollout launches (tests / profiling)."""
    check(lib().dexsim_set_rollout_impl({"auto": 0, "thread": 1, "split": 2}[impl]), "dexsim_set_rollout_impl")


def check(code, where):
    if code != 0:
        raise DexsimError(code, where)


def classify_summary(success, episode_steps, num_contacts, final_contacts, hist_len, max_count, sum_counts,
                     sum_sq_counts, first5_sum, last5_sum, max_steps=200, success_threshold=3, counts=None):
    """Host entry point: both failure labels from an episode summary.
    Returns (metrics.py label code, taxonomy label code, var_tie); LABEL_NONE (255) = success.
    ``counts``: the per-step contact counts (len == hist_len).  With them an exact variance tie is decided by
    NumPy's own np.var arithmetic (var_tie == 2, labels bit-exact); without them var_tie == 1 marks the label
    as resolved in exact arithmetic only."""
    s = DexsimEpisodeSummary(int(bool(success)), int(episode_steps), int(num_contacts), int(final_contacts),
                             int(hist_len), int(max_count), int(sum_counts), int(sum_sq_counts), int(first5_sum),
                             int(last5_sum))
    a, b, t = C.c_int32(), C.c_int32(), C.c_int32()
    ptr = None
    if counts is not None:
        buf = _np.ascontiguousarray(counts, dtype=_np.uint8)
        if buf.shape != (int(hist_len),):
            raise ValueError("counts must hold hist_len entries")
        ptr = buf.ctypes.data
    check(lib().dexsim_classify_summary(C.byref(s), ptr, int(max_steps), int(success_threshold), C.byref(a), C.byref(b),
                                        C.byref(t)), "dexsim_classify_summary")
    return a.value, b.value, t.value


def classify_counts(success, episode_steps, num_contacts, final_contacts, counts, max_steps=200, success_threshold=3):
    """Both failure labels of one episode from its per-step contact counts -- what
    EvaluationMetrics.classify_failure (evaluation/metrics.py:39-96) and FailureClassifier.classify
    (evaluation/failure_taxonomy.py:156-239) return for ``contact_history = count-encoded rows``.
    Returns (metrics label code, taxonomy label code); bit-exact including variance ties."""
    c = _np.ascontiguousarray(counts, dtype=_np.uint8)
    n = int(c.shape[0])
    w = c.astype(_np.int64)
    la, lb, _ = classify_summary(success, episode_steps, num_contacts, final_contacts, n, int(w.max()) if n else 0,
                                 int(w.sum()), int((w * w).sum()), int(w[:5].sum()), int(w[-5:].sum()) if n else 0,
                                 max_steps, success_threshold, counts=c)
    return la, lb
