"""ctypes binding of the C ABI declared in ``include/ssd_b200.h``.

There is no fallback: if ``libssd_b200.so`` is missing this module raises, and
every compute entry point needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SSD_B200_LIB") or os.path.join(
    PKG_DIR, "libssd_b200_check.so" if os.environ.get("SSD_B200_CHECKED") == "1" else "libssd_b200.so")

SSD_OK, SSD_ERR_INVALID, SSD_ERR_CUDA, SSD_ERR_SPAWN, SSD_ERR_MAP = 0, -1, -2, -3, -4
SSD_OBS_RGB, SSD_OBS_INDEX4 = 0, 1
SSD_MAX_VARIANTS = 256
# per-agent episode counters (ssd_set_stats): field index = position in STAT_NAMES
STAT_NAMES = ("apples", "apple_t", "fires", "hits_dealt", "hits_taken", "out_steps", "cleaned")
SSD_N_STATS = len(STAT_NAMES)
(SSD_STAT_APPLES, SSD_STAT_APPLE_T, SSD_STAT_FIRES, SSD_STAT_HITS_DEALT, SSD_STAT_HITS_TAKEN, SSD_STAT_OUT_STEPS,
 SSD_STAT_CLEANED) = range(SSD_N_STATS)

# every symbol include/ssd_b200.h declares (checked by tests/test_capi_symbols.py against the header text)
EXPORTS = ("ssd_abi_version", "ssd_error_string", "ssd_last_cuda_error", "ssd_prob_to_threshold",
           "ssd_create", "ssd_destroy", "ssd_get_layout", "ssd_get_obs_layout", "ssd_set_obs_format", "ssd_expand_obs",
           "ssd_get_state_layout", "ssd_set_state_format", "ssd_expand_state",
           "ssd_reset", "ssd_step", "ssd_step_range", "ssd_step_autoreset", "ssd_render",
           "ssd_set_variants", "ssd_set_env_variants", "ssd_set_stats", "ssd_set_reward_shaping",
           "ssd_step_host", "ssd_incentive", "ssd_launch_count", "ssd_debug_oob_count",
           "ssd_select_actions", "ssd_policy_last_cuda_error",
           "ssd_frontend_create", "ssd_frontend_forward", "ssd_frontend_forward_index4", "ssd_frontend_destroy",
           "ssd_frontend_last_cuda_error")


class SsdConfig(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_envs", C.c_int32), ("n_agents", C.c_int32),
                ("height", C.c_int32), ("width", C.c_int32), ("view", C.c_int32),
                ("episode_limit", C.c_int32), ("fire_cost", C.c_int32), ("hit_penalty", C.c_int32),
                ("beam_len", C.c_int32), ("random_spawn_point", C.c_int32), ("spawn_rotation", C.c_int32),
                ("device", C.c_int32), ("tag_timeout", C.c_int32),
                ("seed", C.c_uint64), ("env_gid_base", C.c_uint32), ("n_waste_lut", C.c_uint32),
                ("ascii_map", C.c_char_p), ("thr_apple", C.c_void_p), ("thr_waste", C.c_void_p),
                ("thr_harvest", C.c_uint32 * 4), ("color_lut", (C.c_uint8 * 4) * 16)]


class SsdVariant(C.Structure):
    _fields_ = [("ascii_map", C.c_char_p), ("n_waste_lut", C.c_uint32), ("thr_apple", C.c_void_p), ("thr_waste", C.c_void_p),
                ("thr_harvest", C.c_uint32 * 4), ("fire_cost", C.c_int32), ("hit_penalty", C.c_int32), ("tag_timeout", C.c_int32)]


class SsdShaping(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("alpha", "beta", "decay", "prosocial")]


class SsdLayout(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("n_actions", "n_cells", "obs_n", "grid_stride", "agent_stride",
                                          "obs_plane_stride", "obs_agent_stride", "obs_env_stride",
                                          "n_apple_pts", "n_waste_pts", "n_spawn_pts", "obs_row_stride")]


class SsdObsLayout(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("format", "row_stride", "plane_stride", "agent_stride", "env_stride")]


class SsdStateLayout(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("format", "row_stride", "plane_stride", "env_stride")]


class SsdState(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("grid", "agent", "ep_ret", "t", "tick", "counts")]


class SsdStepOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("reward", "clean", "apple_cnt", "done", "obs", "state_rgb")]


class SsdDraws(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("prio", "u_apple", "u_waste", "wkey", "spawn_key", "rot")]


class SsdEpisodeEnd(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("obs", "state_rgb", "ep_ret")]


class SsdError(RuntimeError):
    def __init__(self, code, cuda_error=0, msg=""):
        self.code, self.cuda_error = code, cuda_error
        super().__init__(f"ssd_b200 error {code}: {msg}" + (f" (cudaError {cuda_error})" if code == SSD_ERR_CUDA else ""))


_lib = None


def load():
    """dlopen the in-tree library; loud failure if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing -- run `python -m homophily_marl_b200._build` "
                          "(or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.ssd_abi_version.restype = C.c_int
    L.ssd_error_string.restype = C.c_char_p
    L.ssd_error_string.argtypes = [C.c_int]
    L.ssd_last_cuda_error.restype = C.c_int
    L.ssd_prob_to_threshold.restype = C.c_uint32
    L.ssd_prob_to_threshold.argtypes = [C.c_double]
    L.ssd_create.argtypes = [C.POINTER(SsdConfig), C.POINTER(C.c_void_p)]
    L.ssd_destroy.argtypes = [C.c_void_p]
    L.ssd_get_layout.argtypes = [C.c_void_p, C.POINTER(SsdLayout)]
    L.ssd_get_obs_layout.argtypes = [C.c_void_p, C.c_int32, C.POINTER(SsdObsLayout)]
    L.ssd_set_obs_format.argtypes = [C.c_void_p, C.c_int32]
    L.ssd_expand_obs.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.ssd_get_state_layout.argtypes = [C.c_void_p, C.c_int32, C.POINTER(SsdStateLayout)]
    L.ssd_set_state_format.argtypes = [C.c_void_p, C.c_int32]
    L.ssd_expand_state.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.ssd_set_variants.argtypes = [C.c_void_p, C.c_int32, C.POINTER(SsdVariant)]
    L.ssd_set_env_variants.argtypes = [C.c_void_p, C.c_void_p]
    L.ssd_set_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.ssd_set_reward_shaping.argtypes = [C.c_void_p, C.c_int32, C.POINTER(SsdShaping), C.c_void_p, C.c_void_p]
    L.ssd_reset.argtypes = [C.c_void_p, C.POINTER(SsdState), C.c_void_p, C.POINTER(SsdDraws), C.c_void_p, C.c_void_p]
    L.ssd_step.argtypes = [C.c_void_p, C.POINTER(SsdState), C.c_void_p, C.POINTER(SsdDraws), C.POINTER(SsdStepOut), C.c_void_p]
    L.ssd_step_range.argtypes = [C.c_void_p, C.POINTER(SsdState), C.c_void_p, C.POINTER(SsdDraws), C.POINTER(SsdStepOut),
                                 C.c_int32, C.c_int32, C.c_void_p]
    L.ssd_step_autoreset.argtypes = [C.c_void_p, C.POINTER(SsdState), C.c_void_p, C.POINTER(SsdDraws), C.POINTER(SsdStepOut),
                                     C.POINTER(SsdEpisodeEnd), C.c_int32, C.c_int32, C.c_void_p]
    L.ssd_render.argtypes = [C.c_void_p, C.POINTER(SsdState), C.c_void_p, C.c_void_p, C.c_void_p]
    L.ssd_step_host.argtypes = [C.c_void_p, C.POINTER(SsdState), C.c_void_p, C.c_void_p,
                                C.POINTER(SsdStepOut), C.POINTER(SsdStepOut), C.c_void_p]
    L.ssd_incentive.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_float, C.c_float,
                                C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ssd_select_actions.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                     C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]
    L.ssd_frontend_create.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int32,
                                      C.POINTER(C.c_void_p)]
    L.ssd_frontend_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.ssd_frontend_forward_index4.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                              C.c_void_p]
    L.ssd_frontend_destroy.argtypes = [C.c_void_p]
    L.ssd_launch_count.restype = C.c_int64
    L.ssd_launch_count.argtypes = [C.c_void_p]
    L.ssd_debug_oob_count.restype = C.c_int64
    for name in EXPORTS:
        getattr(L, name)
    _lib = L
    return L


def check(rc: int):
    if rc != SSD_OK:
        L = load()
        raise SsdError(rc, L.ssd_last_cuda_error(), L.ssd_error_string(rc).decode())
