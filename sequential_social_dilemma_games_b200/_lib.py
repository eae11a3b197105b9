"""ctypes binding of libssd_b200.so (include/ssd_b200.h).  There is no CPU fallback: if the CUDA
library is missing the import of this module raises."""
import ctypes as C
import os

from ._names import STAT_NAMES  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libssd_b200.so")

ABI_VERSION = 2
MAX_AGENTS = 16
NUM_STATS = 8
OPT_CHAIN_STEPS = 1
OPT_GENERAL_KERNEL = 2
PHASE_MOVES, PHASE_CONSUME, PHASE_BEAMS, PHASE_SPAWN, PHASE_RENDER, PHASE_ALL = 1, 2, 4, 8, 16, 31
ACT_SAMPLE, ACT_GREEDY, ACT_GIVEN = 0, 1, 2
DIV_KL, DIV_JSD = 0, 1
ADV_GAE, ADV_RETURNS = 0, 1
DTYPE_I32, DTYPE_F32 = 0, 1

# every symbol include/ssd_b200.h declares (tests/test_cabi.py checks the list against the header)
SYMBOLS = ("ssd_last_error", "ssd_abi_version", "ssd_create", "ssd_destroy", "ssd_num_apple_points",
           "ssd_num_waste_points", "ssd_obs_bytes_per_env", "ssd_envs_per_cta",
           "ssd_algorithmic_bytes_per_env_step", "ssd_seed", "ssd_get_counter", "ssd_set_state",
           "ssd_get_state", "ssd_reset", "ssd_reset_rows", "ssd_step", "ssd_rollout", "ssd_step_phases", "ssd_get_beams", "ssd_render", "ssd_render_map", "ssd_step_host",
           "ssd_set_option", "ssd_stats", "ssd_launch_count", "ssd_philox_selftest",
           "ssd_policy_create", "ssd_policy_features", "ssd_policy_destroy", "ssd_policy_lstm_cell",
           "ssd_policy_set_head", "ssd_policy_lstm_heads", "ssd_policy_create_n", "ssd_policy_set_head_n",
           "ssd_policy_create_pool", "ssd_policy_pool_features", "ssd_policy_pool_lstm_heads", "ssd_policy_lstm_heads_dist",
           "ssd_policy_pool_lstm_heads_dist", "ssd_moa_create", "ssd_moa_destroy", "ssd_moa_step", "ssd_moa_create_pool",
           "ssd_moa_pool_step", "ssd_advantages_workspace_bytes", "ssd_advantages", "ssd_vtrace")


class SsdConfig(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("kind", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
                ("num_agents", C.c_int32), ("view_radius", C.c_int32), ("beam_len", C.c_int32),
                ("num_envs", C.c_int32), ("device", C.c_int32), ("envs_per_cta", C.c_int32),
                ("env_id_offset", C.c_uint64),
                ("base_map", C.c_void_p), ("color_lut", C.c_void_p), ("harvest_spawn_prob", C.c_void_p),
                ("cleanup_apple_prob", C.c_void_p), ("cleanup_waste_prob", C.c_void_p),
                ("potential_waste_area", C.c_int32), ("num_spawn_points", C.c_int32),
                ("spawn_points", C.c_void_p)]


class SsdTape(C.Structure):
    _fields_ = [("move_order", C.c_void_p), ("uniforms", C.c_void_p), ("u_stride", C.c_int32),
                ("waste_order", C.c_void_p), ("n_draws_out", C.c_void_p)]


class SsdError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libssd_b200.so is not built (%s). Build it with `python -m sequential_social_dilemma_games_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    try:  # make sure libcudart.so.12 is resolvable (PyTorch ships it)
        import torch  # noqa: F401
    except Exception:  # pragma: no cover
        pass
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, u32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_uint32
    sig = {
        "ssd_last_error": (C.c_char_p, []),
        "ssd_abi_version": (i32, []),
        "ssd_create": (i32, [C.POINTER(SsdConfig), C.POINTER(vp)]),
        "ssd_destroy": (i32, [vp]),
        "ssd_num_apple_points": (i32, [vp]),
        "ssd_num_waste_points": (i32, [vp]),
        "ssd_obs_bytes_per_env": (i64, [vp]),
        "ssd_envs_per_cta": (i32, [vp]),
        "ssd_algorithmic_bytes_per_env_step": (i64, [vp]),
        "ssd_seed": (i32, [vp, u64, u32]),
        "ssd_get_counter": (i32, [vp, C.POINTER(u32)]),
        "ssd_set_state": (i32, [vp, vp, vp, vp, vp]),
        "ssd_get_state": (i32, [vp, vp, vp, vp, vp]),
        "ssd_reset": (i32, [vp, vp, vp, vp]),
        "ssd_reset_rows": (i32, [vp, vp, i32, vp, vp]),
        "ssd_step": (i32, [vp, vp, vp, C.POINTER(SsdTape), vp, vp, vp]),
        "ssd_rollout": (i32, [vp, i32, vp, vp, i32, vp, vp]),
        "ssd_step_phases": (i32, [vp, i32, vp, vp, C.POINTER(SsdTape), vp, vp, vp]),
        "ssd_get_beams": (i32, [vp, vp, vp]),
        "ssd_render": (i32, [vp, i32, vp, vp]),
        "ssd_render_map": (i32, [vp, vp, vp]),
        "ssd_step_host": (i32, [vp, vp, vp, vp, vp]),
        "ssd_set_option": (i32, [vp, i32, i64]),
        "ssd_stats": (i32, [vp, vp, vp]),
        "ssd_launch_count": (i64, [vp]),
        "ssd_philox_selftest": (i32, [i32, vp, vp, vp]),
        "ssd_policy_create": (i32, [i32, i32, vp, vp, vp, vp, vp, vp, C.POINTER(vp)]),
        "ssd_policy_features": (i32, [vp, vp, i64, vp, vp]),
        "ssd_policy_destroy": (None, [vp]),
        "ssd_policy_lstm_cell": (i32, [vp, vp, vp, vp, vp, vp, i64, i32, vp]),
        "ssd_policy_set_head": (i32, [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
        "ssd_policy_lstm_heads": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, C.c_uint64, C.c_uint32, vp]),
        "ssd_policy_create_n": (i32, [i32, i32, i32, vp, vp, vp, vp, vp, vp, C.POINTER(vp)]),
        "ssd_policy_set_head_n": (i32, [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
        "ssd_policy_create_pool": (i32, [i32, i32, i32, i32, i32] + [vp] * 13 + [C.POINTER(vp)]),
        "ssd_policy_pool_features": (i32, [vp, vp, vp, i64, vp, vp]),
        "ssd_policy_pool_lstm_heads": (i32, [vp] + [vp] * 9 + [i64, C.c_uint64, C.c_uint32, vp]),
        "ssd_policy_lstm_heads_dist": (i32, [vp] * 8 + [i32] + [vp] * 3 + [i64, C.c_uint64, C.c_uint32, vp]),
        "ssd_policy_pool_lstm_heads_dist": (i32, [vp] * 9 + [i32] + [vp] * 3 + [i64, C.c_uint64, C.c_uint32, vp]),
        "ssd_moa_create": (i32, [i32, i32, i32, i32] + [vp] * 5 + [C.POINTER(vp)]),
        "ssd_moa_destroy": (None, [vp]),
        "ssd_moa_step": (i32, [vp] * 12 + [i64, i32, C.c_float, vp]),
        "ssd_moa_create_pool": (i32, [i32, i32, i32, i32] + [vp] * 5 + [C.POINTER(vp)]),
        "ssd_moa_pool_step": (i32, [vp] * 13 + [i64, i32, C.c_float, vp]),
        "ssd_advantages_workspace_bytes": (i64, [i64, i64]),
        "ssd_advantages": (i32, [i32, i64, i64, i32, vp, i32, vp, C.c_float, vp, vp, vp, C.c_float, C.c_float, vp, vp, vp, i64, vp]),
        "ssd_vtrace": (i32, [i64, i64, i32, vp, i32, vp, C.c_float, vp, vp, vp, vp, vp, C.c_float, C.c_float, C.c_float, vp, vp, vp,
                             i64, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.ssd_abi_version() != ABI_VERSION:
        raise ImportError("libssd_b200.so ABI %d != binding ABI %d; rebuild" % (lib.ssd_abi_version(), ABI_VERSION))
    return lib


lib = _load()


def check(rc):
    if rc != 0:
        raise SsdError("libssd_b200 error %d: %s" % (rc, lib.ssd_last_error().decode()))
