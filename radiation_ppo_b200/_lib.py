"""ctypes binding of the C-ABI CUDA library (include/radsearch_b200.h).  There is no CPU fallback: if the library is
missing or the symbols do not resolve, importing the package's compute entry points raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# RADSEARCH_B200_LIB: another build of the same library (e.g. one made with different -D tuning macros, see build.py)
LIB_PATH = os.environ.get("RADSEARCH_B200_LIB") or os.path.join(HERE, "_C", "libradsearch_b200.so")

OBS_DIM, MAX_K, MAX_A = 11, 8, 8
F_AUTO_RESET, F_EPOCH_END, F_RESET_LIST, F_NEW_OBSTACLES, F_FAST_POISSON = 1, 2, 4, 8, 16
F_PREFETCH, F_REFILL_LIST, F_DEVICE_CTR, F_PARITY1, F_BUMP_CTR, F_ZERO_REFILL = 32, 64, 128, 256, 512, 1024
I_OOB, I_BLOCKED, I_COLLISION, I_LOS_BLOCKED, I_MOVED = 1, 2, 4, 8, 16
E_TERMINAL, E_TIMEOUT, E_RESET = 1, 2, 4
ST_REJECT_CAP, ST_LAMBDA_INF, ST_UNIFORMS_OUT, ST_CORRECT_MISS, ST_WALL_ASSERT, ST_COORD_RANGE = 1, 2, 4, 8, 16, 32
ST_REFILL_OVERFLOW = 64

EXPORTS = [
    "rs_step", "rs_reset", "rs_prepare", "rs_bump_ctr", "rs_load_scenarios", "rs_query_shortest_path", "rs_gae", "rs_adv_stats", "rs_adv_normalize", "rs_last_error",
    "rs_version", "rs_sizeof_config", "rs_sizeof_state", "rs_maps_update", "rs_maps_reset", "rs_sizeof_maps_config",
    "rs_sizeof_maps_state", "rs_pack_rollout", "rs_episode_table", "rs_rollout_pre", "rs_rollout_post",
    "rs_rollout_pre_team", "rs_rollout_post_team", "rs_maps_replay", "rs_eval_step", "rs_policy_param_count",
    "rs_policy_act", "rs_policy_value", "rs_sizeof_policy_config", "rs_policy_grad_workspace_bytes", "rs_policy_ppo_grad",
    "rs_pfgru_param_count", "rs_pfgru_predict", "rs_pfgru_peek", "rs_pfgru_restart", "rs_sizeof_pfgru_config",
]
MS_CELL_RANGE, MS_LOG_FULL, MS_PRED_RANGE = 1, 2, 4
MR_BAD_RANGE = 8


class RsConfig(C.Structure):
    _fields_ = [
        ("bbox", C.c_int32 * 4),
        ("obs_area", C.c_int32 * 2),
        ("enforce", C.c_int32),
        ("n_agents", C.c_int32),
        ("obstruction_count", C.c_int32),
        ("count_law", C.c_int32),
        ("max_ep_len", C.c_int32),
        ("k_max", C.c_int32),
        ("standardize", C.c_int32),
    ]


class RsState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "src", "rad", "rects", "meta", "det", "best", "aflags", "dsrc", "vis", "status", "reset_list", "reset_count",
        "epi", "nx_src", "nx_det", "nx_rad", "nx_best", "nx_dsrc", "nx_obs", "nx_seq", "refill_list", "refill_count",
        "ctr_dev", "st_mean", "st_m2", "raw_count", "ticket", "dsf", "nx_dsf")]


class RsMapsConfig(C.Structure):
    _fields_ = [
        ("n_agents", C.c_int32),
        ("dim_x", C.c_int32),
        ("dim_y", C.c_int32),
        ("base", C.c_int32),
        ("log_cap", C.c_int32),
        ("use_prediction", C.c_int32),
        ("resolution_accuracy", C.c_double),
        ("scale", C.c_double),
    ]


class RsMapsState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "actor", "critic", "log_cell", "log_val", "log_len", "last_cell", "last_pred", "std", "std_count",
        "visit_lut", "status")]


class RsPolicyConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("d_in", "hidden", "pi_hidden", "v_hidden", "activation")]


class RsPfgruConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("d_in", "hidden", "particles", "obs_hidden", "resample")] + [("alpha", C.c_float)]


class RadSearchLibraryError(RuntimeError):
    pass


_lib = None


def declare(lib, prefix="rs_"):
    """Attach argtypes/restype to the entry points of `lib` (also used for the host-emulation build in tests/)."""
    vp, i32, u32, u64, i64, f64 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64, C.c_int64, C.c_double
    cfgp, stp = C.POINTER(RsConfig), C.POINTER(RsState)
    tail = [vp] if prefix == "rs_" else []       # the emulation has no stream argument
    f = getattr(lib, prefix + "step")
    f.restype = i32
    f.argtypes = [cfgp, stp, vp, vp, vp, vp, vp, vp, vp, vp, i32, u32, u64, u64, vp, i32, i32] + tail
    f = getattr(lib, prefix + "reset")
    f.restype = i32
    f.argtypes = [cfgp, stp, vp, vp, vp, i32, u32, u64, u64, vp, i32, i32] + tail
    f = getattr(lib, prefix + "load_scenarios")
    f.restype = i32
    f.argtypes = [cfgp, stp, vp, vp, vp, vp, vp, i32, vp, vp, i32, u32, u64, u64, vp, i32] + tail
    f = getattr(lib, prefix + "prepare")
    f.restype = i32
    f.argtypes = [cfgp, stp, i32, u32, u64, i32] + tail
    f = getattr(lib, prefix + "query_shortest_path")
    f.restype = i32
    f.argtypes = [cfgp, stp, vp, vp, i32, i32] + tail
    if prefix == "rs_":
        lib.rs_gae.restype = i32
        lib.rs_gae.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, f64, f64, vp, i32, vp]
        lib.rs_adv_stats.restype = i32
        lib.rs_adv_stats.argtypes = [vp, i64, vp, vp, vp]
        lib.rs_adv_normalize.restype = i32
        lib.rs_adv_normalize.argtypes = [vp, i64, vp, vp, vp]
        lib.rs_bump_ctr.restype = i32
        lib.rs_bump_ctr.argtypes = [stp, vp]
        mcp, msp = C.POINTER(RsMapsConfig), C.POINTER(RsMapsState)
        lib.rs_maps_update.restype = i32
        lib.rs_maps_update.argtypes = [mcp, msp, vp, vp, vp, i32, i32, vp]
        lib.rs_maps_reset.restype = i32
        lib.rs_maps_reset.argtypes = [mcp, msp, vp, i32, i32, vp]
        lib.rs_pack_rollout.restype = i32
        lib.rs_pack_rollout.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
        lib.rs_episode_table.restype = i32
        lib.rs_episode_table.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
        lib.rs_rollout_pre.restype = i32
        lib.rs_rollout_pre.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
        lib.rs_rollout_post.restype = i32
        lib.rs_rollout_post.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
        lib.rs_rollout_pre_team.restype = i32
        lib.rs_rollout_pre_team.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
        lib.rs_rollout_post_team.restype = i32
        lib.rs_rollout_post_team.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32,
                                             vp]
        lib.rs_maps_replay.restype = i32
        lib.rs_maps_replay.argtypes = [mcp, msp, vp, vp, vp, i32, i32, vp, i32, vp, vp, vp, vp, vp]
        lib.rs_eval_step.restype = i32
        lib.rs_eval_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, f64, vp, vp, vp, i32, i32, i32, vp]
        pcp = C.POINTER(RsPolicyConfig)
        lib.rs_policy_param_count.restype = i32
        lib.rs_policy_param_count.argtypes = [pcp]
        lib.rs_policy_act.restype = i32
        lib.rs_policy_act.argtypes = [pcp, vp, vp, vp, vp, vp, vp, vp, i32, u32, u64, vp, vp, vp]
        lib.rs_policy_value.restype = i32
        lib.rs_policy_value.argtypes = [pcp, vp, vp, vp, vp, vp, i32, vp]
        lib.rs_sizeof_policy_config.restype = i32
        lib.rs_policy_grad_workspace_bytes.restype = i64
        lib.rs_policy_grad_workspace_bytes.argtypes = [pcp, i32, i32]
        lib.rs_policy_ppo_grad.restype = i32
        lib.rs_policy_ppo_grad.argtypes = [pcp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, f64, f64, f64, vp, vp, vp, vp,
                                           vp]
        fcp = C.POINTER(RsPfgruConfig)
        lib.rs_pfgru_param_count.restype = i32
        lib.rs_pfgru_param_count.argtypes = [fcp]
        lib.rs_pfgru_predict.restype = i32
        lib.rs_pfgru_predict.argtypes = [fcp, vp, vp, vp, vp, vp, i32, u32, u64, vp, vp, vp]
        lib.rs_pfgru_peek.restype = i32
        lib.rs_pfgru_peek.argtypes = [fcp, vp, vp, vp, vp, vp, vp, i32, i32, u32, u64, vp, vp]
        lib.rs_pfgru_restart.restype = i32
        lib.rs_pfgru_restart.argtypes = [fcp, vp, vp, vp, i32, i32, u32, u64, vp, vp]
        lib.rs_sizeof_pfgru_config.restype = i32
        lib.rs_sizeof_maps_config.restype = i32
        lib.rs_sizeof_maps_state.restype = i32
        lib.rs_last_error.restype = C.c_char_p
        lib.rs_version.restype = i32
        lib.rs_sizeof_config.restype = i32
        lib.rs_sizeof_state.restype = i32
    return lib


def load():
    """Load libradsearch_b200.so; raises RadSearchLibraryError when it has not been built (python -m radiation_ppo_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RadSearchLibraryError(
                f"{LIB_PATH} not found: build it with `python -m radiation_ppo_b200.build` (there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        missing = [s for s in EXPORTS if not hasattr(lib, s)]
        if missing:
            raise RadSearchLibraryError(f"{LIB_PATH} lacks symbols {missing}")
        declare(lib)
        if lib.rs_sizeof_config() != C.sizeof(RsConfig) or lib.rs_sizeof_state() != C.sizeof(RsState) or \
                lib.rs_sizeof_maps_config() != C.sizeof(RsMapsConfig) or lib.rs_sizeof_maps_state() != C.sizeof(RsMapsState) or \
                lib.rs_sizeof_policy_config() != C.sizeof(RsPolicyConfig) or \
                lib.rs_sizeof_pfgru_config() != C.sizeof(RsPfgruConfig):
            raise RadSearchLibraryError("struct layout mismatch between _lib.py and libradsearch_b200.so")
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        raise ValueError(f"{what}: {load().rs_last_error().decode()}")
    raise RadSearchLibraryError(f"{what}: CUDA error {rc}")
