"""ctypes binding of libssb (include/ssb.h).  There is NO fallback: if the CUDA library has not been
built (`python -c "import __graft_entry__ as g; g.build()"`), importing the env fails loudly."""
from __future__ import annotations

import ctypes as C
import os.path as osp

import numpy as np

PKG_DIR = osp.dirname(osp.abspath(__file__))
LIB_PATH = osp.join(PKG_DIR, "_lib", "libssb.so")
ABI_VERSION = 9


class SsbConfig(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32),
        ("num_executors", C.c_int32),
        ("job_arrival_cap", C.c_int32),
        ("max_jobs", C.c_int32),
        ("tape_capacity", C.c_int32),
        ("log_capacity", C.c_int32),
        ("moving_delay", C.c_double),
        ("warmup_delay", C.c_double),
        ("job_arrival_rate", C.c_double),
        ("beta", C.c_double),
        ("flags", C.c_int32),
        ("history_capacity", C.c_int32),
    ]


FLAG_DECIMA_OBS = 1
ENV_CAPACITY = 10  # SSB_ENV_CAPACITY (include/ssb.h)
FLAG_DECIMA_POLICY = 2
DECIMA_NUM_PARAMS = 20802


class SsbPolicyViews(C.Structure):
    _fields_ = [
        ("stage_logits", C.c_void_p),
        ("exec_logits", C.c_void_p),
        ("action", C.c_void_p),
        ("lgprob", C.c_void_p),
        ("node_stride", C.c_int32),
        ("exec_stride", C.c_int32),
        ("entropy", C.c_void_p),
    ]


class SsbDecimaViews(C.Structure):
    _fields_ = [
        ("features", C.c_void_p),
        ("stage_mask", C.c_void_p),
        ("commit_caps", C.c_void_p),
        ("edge_bits", C.c_void_p),
        ("depth", C.c_void_p),
        ("node_stride", C.c_int32),
        ("edge_stride", C.c_int32),
        ("job_stride", C.c_int32),
        ("pad", C.c_int32),
        ("frontier_mask", C.c_void_p),
    ]


class SsbPackedObs(C.Structure):
    _fields_ = [
        ("offsets", C.c_void_p),
        ("nodes", C.c_void_p),
        ("edge_links", C.c_void_p),
        ("dag_ptr", C.c_void_p),
        ("exec_supplies", C.c_void_p),
        ("node_capacity", C.c_int64),
        ("edge_capacity", C.c_int64),
        ("job_capacity", C.c_int64),
    ]


class SsbBank(C.Structure):
    _fields_ = [
        ("num_templates", C.c_int32),
        ("num_template_stages", C.c_int32),
        ("num_template_edges", C.c_int32),
        ("num_values", C.c_int64),
        ("num_stages", C.c_void_p),
        ("stage_base", C.c_void_p),
        ("edge_base", C.c_void_p),
        ("edges", C.c_void_p),
        ("num_tasks", C.c_void_p),
        ("rough_duration", C.c_void_p),
        ("parent_mask", C.c_void_p),
        ("child_mask", C.c_void_p),
        ("present", C.c_void_p),
        ("dur_off", C.c_void_p),
        ("dur_cnt", C.c_void_p),
        ("dur_values", C.c_void_p),
    ]


class SsbViews(C.Structure):
    _fields_ = [
        ("hdr", C.c_void_p),
        ("nodes", C.c_void_p),
        ("edge_links", C.c_void_p),
        ("dag_ptr", C.c_void_p),
        ("exec_supplies", C.c_void_p),
        ("node_stride", C.c_int32),
        ("edge_stride", C.c_int32),
        ("job_stride", C.c_int32),
        ("pad", C.c_int32),
    ]


# numpy mirrors of ssb_obs_hdr / ssb_stats
OBS_HDR_DTYPE = np.dtype(
    [
        ("reward", "<f8"),
        ("wall_time", "<f8"),
        ("num_nodes", "<i4"),
        ("num_edges", "<i4"),
        ("num_active_jobs", "<i4"),
        ("num_committable_execs", "<i4"),
        ("source_job_idx", "<i4"),
        ("num_schedulable", "<i4"),
        ("error", "<i4"),
        ("terminated", "u1"),
        ("truncated", "u1"),
        ("pending", "u1"),
        ("was_reset", "u1"),
    ]
)
assert OBS_HDR_DTYPE.itemsize == 48
# ssb_transition (include/ssb.h): one stored step of a fused rollout
TRANSITION_DTYPE = np.dtype([("wall_time", "<f8"), ("reward", "<f8"), ("stage_idx", "<i4"), ("num_exec", "<i4"),
                             ("flags", "<i4"), ("lgprob", "<f4")])
assert TRANSITION_DTYPE.itemsize == 32
STATS_FIELDS = ("decisions", "events", "sched_scans", "sum_nodes", "sum_edges", "sum_jobs",
                "observations", "episodes")
STATS_DTYPE = np.dtype([(f, "<u8") for f in STATS_FIELDS])

EXPORTS = [
    "ssb_abi_version", "ssb_last_cuda_error", "ssb_workspace_bytes", "ssb_create", "ssb_destroy",
    "ssb_load_trace", "ssb_clear_trace", "ssb_reset", "ssb_step", "ssb_reset_host", "ssb_step_host", "ssb_step_fair_host", "ssb_set_autoreset", "ssb_set_mean_time_limit",
    "ssb_rollout_fair", "ssb_rollout_fair_traj", "ssb_rollout_fair_async", "ssb_discounted_returns", "ssb_differential_returns", "ssb_group_baselines", "ssb_ppo_loss", "ssb_adam_step", "ssb_fair_actions", "ssb_random_actions", "ssb_rollout_random", "ssb_rollout_random_async", "ssb_get_views", "ssb_get_stats", "ssb_collect_stats", "ssb_reset_stats",
    "ssb_get_jobs", "ssb_get_log", "ssb_get_history", "ssb_decima_obs", "ssb_get_decima_views",
    "ssb_set_decima_weights", "ssb_decima_policy", "ssb_rollout_decima", "ssb_rollout_decima_async", "ssb_set_policy_streams", "ssb_decima_attach_rollout_store", "ssb_decima_snapshot_bytes",
    "ssb_decima_snapshot", "ssb_decima_snapshot_gather", "ssb_decima_snapshot_load", "ssb_decima_snapshot_unload", "ssb_decima_evaluate", "ssb_decima_head_adjoint", "ssb_decima_head_backward", "ssb_decima_backward_bytes", "ssb_decima_attach_backward_scratch", "ssb_decima_backward", "ssb_get_policy_views", "ssb_decima_work", "ssb_decima_mlp_rows", "ssb_packed_obs_bytes", "ssb_get_obs_host", "ssb_get_debug_counters",
]

_lib = None


def lib():
    """Loads libssb.so (built in-tree by __graft_entry__.build()); raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    import os

    path = os.environ.get("SSB_LIB", LIB_PATH)  # SSB_LIB: A/B-test another build of the same library
    if not osp.exists(path):
        raise ImportError(
            f"{path} not found: the CUDA library has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback."
        )
    L = C.CDLL(path)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.ssb_abi_version.restype = C.c_int
    L.ssb_last_cuda_error.restype = C.c_char_p
    L.ssb_workspace_bytes.argtypes = [C.POINTER(SsbConfig), C.POINTER(SsbBank), C.POINTER(C.c_size_t)]
    L.ssb_create.argtypes = [C.POINTER(SsbConfig), C.POINTER(SsbBank), C.c_int, vp, C.c_size_t,
                             C.POINTER(vp)]
    L.ssb_destroy.argtypes = [vp]
    L.ssb_load_trace.argtypes = [vp, i32, i32, vp, vp, vp, i64]
    L.ssb_clear_trace.argtypes = [vp, i32]
    L.ssb_reset.argtypes = [vp, vp, vp, vp, vp]
    L.ssb_step.argtypes = [vp, vp, vp, vp, i32, vp]
    L.ssb_reset_host.argtypes = [vp, vp, vp, vp, vp]
    L.ssb_step_host.argtypes = [vp, vp, vp, vp, i32, vp]
    L.ssb_set_autoreset.argtypes = [vp, i32, u64]
    L.ssb_set_mean_time_limit.argtypes = [vp, C.c_double]
    L.ssb_step_fair_host.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, vp]
    L.ssb_rollout_decima.argtypes = [vp, i32, i32, vp, vp]
    L.ssb_rollout_decima_async.argtypes = [vp, i32, C.c_double, u64, vp, vp, vp, vp]
    L.ssb_set_policy_streams.argtypes = [vp, vp]
    L.ssb_decima_attach_rollout_store.argtypes = [vp, vp, i32, vp, vp]
    L.ssb_decima_snapshot_bytes.argtypes = [vp, C.POINTER(C.c_size_t)]
    L.ssb_decima_snapshot.argtypes = [vp, vp, vp]
    L.ssb_decima_snapshot_gather.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.ssb_decima_evaluate.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.ssb_rollout_fair.argtypes = [vp, i32, i32, i32, u64, vp]
    L.ssb_rollout_fair_traj.argtypes = [vp, i32, i32, i32, u64, vp, vp]
    L.ssb_rollout_fair_async.argtypes = [vp, i32, C.c_double, i32, u64, vp, vp, vp, vp]
    L.ssb_discounted_returns.argtypes = [vp, vp, vp, i32, i32, C.c_double, vp, vp]
    L.ssb_group_baselines.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    L.ssb_ppo_loss.argtypes = [vp, vp, vp, vp, vp, vp, i32, C.c_float, C.c_float, vp, vp, vp, vp, vp]
    L.ssb_decima_head_adjoint.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ssb_decima_head_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(i32), vp]
    L.ssb_decima_backward_bytes.argtypes = [vp, C.POINTER(C.c_size_t)]
    L.ssb_decima_attach_backward_scratch.argtypes = [vp, vp]
    L.ssb_decima_backward.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp]
    L.ssb_decima_snapshot_load.argtypes = [vp, vp, vp]
    L.ssb_decima_snapshot_unload.argtypes = [vp, vp]
    L.ssb_adam_step.argtypes = [vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp, vp, vp]
    L.ssb_differential_returns.argtypes = [vp, vp, vp, i32, i32, vp, i32, C.POINTER(i32), vp, vp, vp, vp]
    L.ssb_fair_actions.argtypes = [vp, i32, vp, vp, vp]
    L.ssb_random_actions.argtypes = [vp, vp, vp, vp, vp]
    L.ssb_rollout_random.argtypes = [vp, i32, i32, u64, vp, vp]
    L.ssb_rollout_random_async.argtypes = [vp, i32, C.c_double, u64, vp, vp, vp, vp]
    L.ssb_get_views.argtypes = [vp, C.POINTER(SsbViews)]
    L.ssb_decima_obs.argtypes = [vp, vp]
    L.ssb_get_decima_views.argtypes = [vp, C.POINTER(SsbDecimaViews)]
    L.ssb_set_decima_weights.argtypes = [vp, vp, i32]
    L.ssb_decima_policy.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ssb_get_policy_views.argtypes = [vp, C.POINTER(SsbPolicyViews)]
    L.ssb_decima_work.argtypes = [vp, vp]
    L.ssb_decima_mlp_rows.argtypes = [vp, i32, vp, i32, vp, vp]
    L.ssb_packed_obs_bytes.argtypes = [vp, C.POINTER(C.c_size_t)]
    L.ssb_get_obs_host.argtypes = [vp, C.POINTER(SsbPackedObs), vp, C.c_size_t]
    L.ssb_get_stats.argtypes = [vp, C.POINTER(vp)]
    L.ssb_reset_stats.argtypes = [vp, vp]
    L.ssb_collect_stats.argtypes = [vp, vp, vp]
    L.ssb_get_debug_counters.argtypes = [vp, C.POINTER(vp)]
    L.ssb_get_jobs.argtypes = [vp, i32, C.POINTER(i32), vp, vp, vp, vp, i32]
    L.ssb_get_log.argtypes = [vp, i32, i64, i64, C.POINTER(i64)] + [vp] * 7
    L.ssb_get_history.argtypes = [vp, i32, C.POINTER(i64), vp, vp, vp, i64]
    if L.ssb_abi_version() != ABI_VERSION:
        raise ImportError("libssb ABI version mismatch; rebuild")
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().ssb_last_cuda_error().decode() if rc == -2 else ""
        raise RuntimeError(f"{what} failed: status {rc} {msg}")


def make_bank_struct(bank):
    """Returns (SsbBank, keepalive list of contiguous numpy arrays)."""
    keep = [np.ascontiguousarray(a) for a in (
        bank.num_stages.astype(np.int32), bank.stage_base.astype(np.int32),
        bank.edge_base.astype(np.int32), bank.edges.astype(np.int32),
        bank.num_tasks.astype(np.int32), bank.rough_duration.astype(np.float64),
        bank.parent_mask.astype(np.uint64), bank.child_mask.astype(np.uint64),
        bank.present.astype(np.uint8), bank.dur_off.astype(np.uint32),
        bank.dur_cnt.astype(np.uint32), bank.dur_values.astype(np.float64))]
    s = SsbBank(bank.num_templates, int(bank.stage_base[-1]), int(bank.edge_base[-1]),
                int(bank.dur_values.shape[0]), *[a.ctypes.data for a in keep])
    return s, keep
