"""ctypes binding of the C-ABI in include/sf_b200.h (libsf_b200.so, built in-tree by build.py).

This is the ONLY implementation of the hot path. If the library cannot be loaded, or there is no CUDA
device, every entry point raises: there is no CPU or PyTorch fallback.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SF_B200_LIB: a variant build of the same library (tools/: -D instrumented builds); never another implementation
LIB_PATH = os.environ.get("SF_B200_LIB") or os.path.join(HERE, "libsf_b200.so")

SF_OK, SF_ERR_INVALID, SF_ERR_CUDA, SF_ERR_UNSUPPORTED = 0, 1, 2, 3
MAX_MISSILES = 20
MAX_SHELLS = 20
NUM_STATS = 13
NUM_EPISODE_STATS = 24
OBS_H = OBS_W = 84
NATIVE_H, NATIVE_W = 92, 90

KEY_FIRE, KEY_THRUST, KEY_LEFT, KEY_RIGHT = 1, 2, 4, 8
MAX_HOST_MIRRORS = 4  # SF_MAX_MIRRORS: host observation buffers whose contents the library remembers per handle
FLAG_RENDER, FLAG_NO_AUTORESET, FLAG_ACTIONS_ARE_KEYMASKS, FLAG_NATIVE_OBS, FLAG_RAW_REWARD, FLAG_HOST_DELTA = 1, 2, 4, 8, 16, 32

ENV_BLOB_BYTES = 832  # SF_ENV_BLOB_BYTES: one env's complete game state as one row (sf_save_envs / sf_load_envs)
ENV_BLOB_VERSION = 1  # SF_ENV_BLOB_VERSION
MAX_ACTION_REPEAT = 5295  # SF_MAX_ACTION_REPEAT: ticks per agent step at most (one episode)

OBS_TYPES = {"image": 0, "features": 1, "normalized-features": 2, "monitors": 3}  # ssf_env.py:51

EVENT_BITS = {
    "missile-fired": 1 << 0, "fortress-fired": 1 << 1, "hit-fortress": 1 << 2, "vlner-increased": 1 << 3,
    "vlner-reset": 1 << 4, "fortress-destroyed": 1 << 5, "hit-dead-fortress": 1 << 6, "explode-bighex": 1 << 7,
    "explode-smallhex": 1 << 8, "shell-hit-ship": 1 << 9, "ship-respawn": 1 << 10, "fortress-respawn": 1 << 11,
}
COLLISION_BITS = {"bighex": 1 << 12, "smallhex": 1 << 13, "missile": 1 << 14, "shell": 1 << 15}
EV_EPISODE_RESET = 1 << 21
EV_STICKY = 1 << 22  # SF_EV_STICKY: a tick of the agent step kept the held keys (sticky actions)

EPISODE_STAT_NAMES = ["episodes", "sum_return", "sum_return_sq", "sum_length", "bigHexDeaths", "smallHexDeaths",
                      "shellDeaths", "shipDeaths", "resets", "destroyedFortresses", "missedShots", "totalShots",
                      "totalThrusts", "totalLefts", "totalRights", "vlnerIncs", "maxVlner_sum", "sum_points_int",
                      "sum_raw_points_milli", "fort_kills", "maxVlner_max", "reserved0", "reserved1", "reserved2"]


class StateRecord(C.Structure):
    """sf_state_record (include/sf_b200.h): the reference's public Game members (game.hh:84-107)."""
    _fields_ = [
        ("ship_x", C.c_double), ("ship_y", C.c_double), ("ship_vx", C.c_double), ("ship_vy", C.c_double),
        ("ship_angle", C.c_double), ("fortress_angle", C.c_double), ("fortress_last_angle", C.c_double),
        ("missile_x", C.c_double * MAX_MISSILES), ("missile_y", C.c_double * MAX_MISSILES),
        ("missile_vx", C.c_double * MAX_MISSILES), ("missile_vy", C.c_double * MAX_MISSILES),
        ("missile_angle", C.c_double * MAX_MISSILES),
        ("shell_x", C.c_double * MAX_SHELLS), ("shell_y", C.c_double * MAX_SHELLS),
        ("shell_vx", C.c_double * MAX_SHELLS), ("shell_vy", C.c_double * MAX_SHELLS),
        ("shell_angle", C.c_double * MAX_SHELLS),
        ("points", C.c_float), ("raw_points", C.c_float),
        ("missile_mask", C.c_uint32), ("shell_mask", C.c_uint32),
        ("ship_alive", C.c_int32), ("fortress_alive", C.c_int32),
        ("ship_death_timer", C.c_int32), ("fire_timer", C.c_int32), ("thrust_timer", C.c_int32),
        ("left_timer", C.c_int32), ("right_timer", C.c_int32),
        ("thrust_flag", C.c_int32), ("fire_flag", C.c_int32), ("left_flag", C.c_int32), ("right_flag", C.c_int32),
        ("turn_flag", C.c_int32),
        ("fortress_timer", C.c_int32), ("fortress_death_timer", C.c_int32), ("fortress_vuln_timer", C.c_int32),
        ("vulnerability", C.c_int32), ("tick", C.c_int32), ("time", C.c_int32),
        ("stats", C.c_int32 * NUM_STATS),
        ("prev_vlner", C.c_int32), ("rng_seed", C.c_uint32), ("rng_count", C.c_uint32), ("ep_return", C.c_int32),
    ]


class SFError(RuntimeError):
    pass


_LIB = None

_PROTOTYPES = {
    "sf_last_error": (C.c_char_p, []),
    "sf_version": (C.c_int, []),
    "sf_create": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "sf_destroy": (C.c_int, [C.c_void_p]),
    "sf_num_envs": (C.c_int, [C.c_void_p]),
    "sf_num_actions": (C.c_int, [C.c_void_p]),
    "sf_action_keymask": (C.c_int, [C.c_void_p, C.c_int]),
    "sf_state_bytes": (C.c_longlong, [C.c_void_p]),
    "sf_seed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "sf_set_ticks": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sf_policy_input": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sf_policy_input_f32": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sf_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "sf_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "sf_rollout": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "sf_synthetic_action": (C.c_int, [C.c_uint32, C.c_longlong, C.c_longlong, C.c_int]),
    "sf_set_action_repeat": (C.c_int, [C.c_void_p, C.c_int]),
    "sf_action_repeat": (C.c_int, [C.c_void_p]),
    "sf_set_sticky_actions": (C.c_int, [C.c_void_p, C.c_double, C.c_uint32]),
    "sf_sticky_actions": (C.c_double, [C.c_void_p]),
    "sf_sticky_draw": (C.c_int, [C.c_uint32, C.c_longlong, C.c_uint32, C.c_int32, C.c_double]),
    "sf_set_final_obs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sf_final_obs_enabled": (C.c_int, [C.c_void_p]),
    "sf_render": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "sf_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "sf_host_delta_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sf_host_forget": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sf_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_longlong]),
    "sf_host_free": (C.c_int, [C.c_void_p]),
    "sf_get_state": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "sf_set_state": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "sf_save_envs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "sf_load_envs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "sf_episode_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "sf_num_features": (C.c_int, [C.c_void_p, C.c_int]),
    "sf_features": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "sf_features_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "sf_rollout_features": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint32, C.c_longlong, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "sf_step_host_features": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "sf_set_glyph_masks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sf_background": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sf_host_static_frame": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
}
EXPORTED_SYMBOLS = sorted(_PROTOTYPES)


def lib():
    """Load libsf_b200.so (raises SFError if it has not been built: run `python -m spacefortress_b200.build`)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise SFError("%s is missing; build it with `python spacefortress_b200/build.py` "
                          "(there is no fallback implementation)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOTYPES.items():
            if os.environ.get("SF_B200_LIB") and not hasattr(L, name):
                continue  # an older variant build under test (tools/gpu_ab.py); the product library must export everything
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(rc):
    if rc != SF_OK:
        msg = lib().sf_last_error()
        raise SFError("sf_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))


class _PinnedBlock(object):
    """Owns one sf_host_alloc block; freed when the last numpy view of it is garbage collected."""

    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            if self.ptr is not None and _LIB is not None:
                _LIB.sf_host_free(self.ptr)
            self.ptr = None
        except Exception:
            pass


def pinned_array(shape, dtype):
    """numpy array over page-locked host memory (sf_host_alloc): device<->host copies DMA straight into it. The
    memory belongs to the array: it is released (sf_host_free) when the last view of it dies, never while a caller
    still holds an observation it was handed."""
    import numpy as np
    dt = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dt.itemsize
    p = C.c_void_p()
    check(lib().sf_host_alloc(C.byref(p), max(nbytes, 1)))
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
    buf._owner = _PinnedBlock(p)  # numpy keeps `buf` alive through .base; `buf` keeps the block alive
    arr = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)
    return arr
