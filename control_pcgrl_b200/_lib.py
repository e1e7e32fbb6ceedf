"""ctypes binding of libpcgrl_sm100.so (the C ABI declared in include/pcgrl_b200.h).

There is deliberately no fallback: if the shared library is missing the import of any compute entry
point raises, so a GPU box can never silently run something else.
"""
from __future__ import annotations

import ctypes as C
import os

PCGRL_ABI_VERSION = 5
MAX_STATS = 16
MAX_TILES = 16

PROB_IDS = {"binary": 0, "zelda": 1, "sokoban": 2, "smb": 3, "minecraft_3D_maze": 4, "binary_holey": 5,
            "minecraft_2D_maze": 6, "minecraft_3D_holey_maze": 7, "minecraft_3D_dungeon_holey": 8}
HOLES_GIVEN, HOLES_FIXED, HOLES_RANDOM = 0, 1, 2
REP_IDS = {"narrow": 0, "turtle": 1, "wide": 2, "cellular": 3}
ACT_INT32, ACT_WIDE_COORDS, ACT_WIDE_FLAT, ACT_CA_TILES, ACT_CA_LOGITS, ACT_PATCH = range(6)
REWARD_CONTROL, REWARD_RANGE = 0, 1

LIB_NAME = "libpcgrl_sm100.so"
# PCGRL_B200_LIB lets kernel experiments load an alternative build of the same ABI (scripts/ab_variants.sh)
LIB_PATH = os.environ.get("PCGRL_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("problem", C.c_int32), ("representation", C.c_int32),
        ("action_kind", C.c_int32), ("ndim", C.c_int32), ("dims", C.c_int32 * 3), ("n_tiles", C.c_int32),
        ("n_stats", C.c_int32), ("row_stride", C.c_int32), ("max_iterations", C.c_int32),
        ("max_changes", C.c_int32), ("act_h", C.c_int32), ("act_w", C.c_int32),
        ("targets_per_env", C.c_int32), ("init_random_probs", C.c_int32), ("reward_mode", C.c_int32),
        ("init_probs", C.c_float * MAX_TILES), ("weights", C.c_double * MAX_STATS),
        ("act_window", C.c_int32 * 3), ("static_prob", C.c_float), ("n_static_walls", C.c_int32),
        ("wall_tile", C.c_int32), ("static_eval_mode", C.c_int32), ("hole_mode", C.c_int32),
        ("action_elem_bytes", C.c_int32), ("record_stat_bytes", C.c_int32),
    ]


class State(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int64), ("env_offset", C.c_int64), ("grids", C.c_void_p), ("pos", C.c_void_p),
        ("n_step", C.c_void_p), ("iteration", C.c_void_p), ("changes", C.c_void_p), ("stats", C.c_void_p),
        ("targets", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p), ("changed", C.c_void_p),
        ("status", C.c_void_p), ("scratch", C.c_void_p), ("static_mask", C.c_void_p), ("holes", C.c_void_p),
        ("records", C.c_void_p), ("worklist", C.c_void_p), ("cache", C.c_void_p),
    ]


class ObsArgs(C.Structure):
    _fields_ = [
        ("crop", C.c_int32), ("obs_dims", C.c_int32 * 3), ("n_ctrl", C.c_int32),
        ("ctrl_idx", C.c_int32 * MAX_STATS), ("ctrl_range", C.c_double * MAX_STATS),
        ("out_kind", C.c_int32), ("out", C.c_void_p), ("static_channel", C.c_int32),
        ("holey_border_tile", C.c_int32),
    ]


# name -> (restype, argtypes); every symbol include/pcgrl_b200.h declares
SYMBOLS = {
    "pcgrl_abi_version": (C.c_int32, []),
    "pcgrl_last_error": (C.c_char_p, []),
    "pcgrl_config_check": (C.c_int32, [C.POINTER(Config)]),
    "pcgrl_scratch_bytes": (C.c_int64, [C.POINTER(Config), C.c_int64]),
    "pcgrl_step_bytes": (C.c_int64, [C.POINTER(Config)]),
    "pcgrl_step": (C.c_int32, [C.POINTER(Config), C.POINTER(State), C.c_void_p, C.c_void_p]),
    "pcgrl_update": (C.c_int32, [C.POINTER(Config), C.POINTER(State), C.c_void_p, C.c_void_p]),
    "pcgrl_reset": (C.c_int32, [C.POINTER(Config), C.POINTER(State), C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_uint64, C.c_uint64, C.c_void_p]),
    "pcgrl_stats": (C.c_int32, [C.POINTER(Config), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "pcgrl_stats_holey": (C.c_int32, [C.POINTER(Config), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                      C.c_void_p]),
    "pcgrl_observe": (C.c_int32, [C.POINTER(Config), C.POINTER(State), C.POINTER(ObsArgs), C.c_void_p]),
    "pcgrl_step_host": (C.c_int32, [C.POINTER(Config), C.POINTER(State), C.c_void_p, C.c_void_p, C.c_int64,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcgrl_step_host_packed": (C.c_int32, [C.POINTER(Config), C.POINTER(State), C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_void_p, C.c_void_p]),
    "pcgrl_record_stride": (C.c_int32, [C.POINTER(Config)]),
    "pcgrl_worklist_ints": (C.c_int64, [C.POINTER(Config), C.c_int64]),
    "pcgrl_cache_stride": (C.c_int32, [C.POINTER(Config)]),
    "pcgrl_launch_count": (C.c_int64, []),
}

_lib = None


class PcgrlError(RuntimeError):
    pass


def load():
    """Load the CUDA library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PcgrlError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). control_pcgrl_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.pcgrl_abi_version() != PCGRL_ABI_VERSION:
        raise PcgrlError("libpcgrl_sm100.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc, what="pcgrl call"):
    if rc != 0:
        msg = load().pcgrl_last_error().decode("utf-8", "replace")
        raise PcgrlError(f"{what} failed ({rc}): {msg}")
