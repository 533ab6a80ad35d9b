"""ctypes binding of include/lle_b200.h (lle_b200/_native/liblle_b200.so).

There is no CPU fallback: if the CUDA extension is missing or no CUDA device is usable, the product
raises.  (The oracle under oracle/ is test infrastructure and is never imported from here.)
"""
from __future__ import annotations

import ctypes as C
import os

from .types import InvalidActionError, InvalidLevelError, InvalidWorldStateError, ParsingError

_HERE = os.path.dirname(os.path.abspath(__file__))
# LLE_B200_LIB: development aid (A/B timing of two builds of this same library on one GPU box)
LIB_PATH = os.environ.get("LLE_B200_LIB") or os.path.join(_HERE, "_native", "liblle_b200.so")

SYMBOLS = [
    "lle_last_error", "lle_version", "lle_map_parse", "lle_map_level", "lle_map_free", "lle_map_get_info",
    "lle_map_positions", "lle_map_start_candidates", "lle_map_sources", "lle_map_lasers", "lle_map_text", "lle_vec_default_options", "lle_vec_create",
    "lle_vec_destroy", "lle_vec_get_buffers", "lle_vec_reset", "lle_vec_refresh", "lle_vec_step", "lle_vec_rollout", "lle_vec_step_host", "lle_vec_pipeline_submit",
    "lle_vec_pipeline_wait", "lle_vec_set_source", "lle_vec_get_sources", "lle_vec_set_exits", "lle_vec_collect_gem", "lle_vec_set_state",
    "lle_vec_export_raw", "lle_vec_set_seed", "lle_vec_get_step_count", "lle_vec_set_step_count", "lle_vec_launch_count",
    "lle_vec_timing_begin", "lle_vec_timing_end", "lle_vec_debug_timeline", "lle_host_alloc", "lle_host_free", "lle_vec_fetch", "lle_vec_export_raw_state", "lle_vec_import_raw_state",
    "lle_vec_get_reset_count", "lle_vec_set_reset_count",
    "lle_vec_parts_begin", "lle_vec_parts_count", "lle_vec_parts_range", "lle_vec_parts_launch", "lle_vec_parts_feed", "lle_vec_parts_wait",
    "lle_vec_parts_end", "lle_vec_parts_abort",
    "lle_gen_default_options", "lle_gen_create", "lle_gen_destroy", "lle_gen_attempt_seeds", "lle_gen_run", "lle_gen_get_buffers",
    "lle_gen_fetch", "lle_gen_geometry_valid", "lle_gen_cells_to_text", "lle_plan",
    "lle_vec_expert_build", "lle_vec_expert_act", "lle_vec_expert_table",
]


class MapInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("height", "width", "n_agents", "n_gems", "n_sources", "n_channels", "n_exits",
                                          "n_walls", "n_voids", "n_laser_cells", "n_lasers", "obs_invalid", "max_beam_len")] + [
        ("gem_toplevel", C.c_uint64)]


class VecOptions(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("device", "reward_dim", "walkable_lasers", "auto_reset", "lle_semantics", "write_obs")] + [
        ("seed", C.c_uint64), ("env_id_base", C.c_uint64), ("n_extras", C.c_int32), ("extras_src", C.c_int32 * 64),
        ("pbrs", C.c_int32), ("n_pbrs", C.c_int32), ("pbrs_src", C.c_int32 * 64), ("pbrs_gamma", C.c_double),
        ("pbrs_reward_value", C.c_double), ("obs_type", C.c_int32), ("obs_param", C.c_int32), ("randomize_lasers", C.c_int32),
        ("state_type", C.c_int32), ("state_param", C.c_int32), ("episode_stats", C.c_int32), ("obs_dtype", C.c_int32)]


class VecBuffers(C.Structure):
    _fields_ = [("n_envs", C.c_int64)] + [(n, C.c_int32) for n in ("n_agents", "n_gems", "n_channels", "height", "width",
                                                                   "reward_dim", "state_dim", "n_beams_max")] + [
        ("obs_stride", C.c_int64), ("obs", C.c_void_p), ("state", C.c_void_p), ("avail", C.c_void_p), ("reward", C.c_void_p),
        ("done", C.c_void_p), ("events", C.c_void_p), ("actions", C.c_void_p), ("err", C.c_void_p), ("record_bytes", C.c_int64), ("extras", C.c_void_p), ("extras_dim", C.c_int32), ("pad", C.c_int32)] + [
        (n, C.c_int32) for n in ("obs_type", "obs_param", "obs_view_agents", "obs_c", "obs_h", "obs_w", "obs_invalid", "pad2")] + [
        ("map_index", C.c_void_p), ("n_variants", C.c_int32), ("pad3", C.c_int32), ("state_obs", C.c_void_p), ("state_obs_stride", C.c_int64)] + [
        (n, C.c_int32) for n in ("state_type", "state_param", "state_view_agents", "state_c", "state_h", "state_w")] + [
        (n, C.c_void_p) for n in ("info", "ep_return", "ep_length", "last_return", "last_length")] + [
        ("obs_i8", C.c_void_p), ("obs_dtype", C.c_int32), ("pad4", C.c_int32)]

# lle_vec_options.obs_dtype
DTYPE_F32, DTYPE_I8 = 0, 1


class RawState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("pos", "alive", "arrived", "slot", "beam_on", "collected", "counters", "avail_cache",
                                          "subgoals_extras", "subgoals_pbrs")]


class GenOptions(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("width", "height", "n_agents", "starts", "exits", "n_lasers", "n_gems", "laser_placement",
                                          "laser_span", "n_walls", "walls_shapes", "n_rooms_rows", "n_rooms_cols", "door_size",
                                          "cluster_h", "cluster_w")]


class GenBuffers(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("n", C.c_int64), ("height", C.c_int32), ("width", C.c_int32), ("cells", C.c_void_p),
                ("status", C.c_void_p), ("labels", C.c_void_p), ("tries", C.c_void_p)]


_lib = None


def lib():
    """Load the extension; fail loudly when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"lle_b200: the CUDA extension {LIB_PATH} is missing. Build it with `python -m lle_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    for name in SYMBOLS:
        getattr(L, name)  # AttributeError if the library is stale
    L.lle_last_error.restype = C.c_char_p
    L.lle_version.restype = C.c_char_p
    L.lle_map_text.restype = C.c_char_p
    L.lle_map_text.argtypes = [C.c_void_p]
    L.lle_map_free.argtypes = [C.c_void_p]
    L.lle_map_free.restype = None
    L.lle_vec_default_options.restype = None
    L.lle_map_parse.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.lle_map_level.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.lle_map_get_info.argtypes = [C.c_void_p, C.POINTER(MapInfo)]
    L.lle_map_positions.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]
    L.lle_map_start_candidates.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]
    L.lle_map_sources.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]
    L.lle_map_lasers.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]
    L.lle_vec_create.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.POINTER(C.c_int32), C.c_int64, C.POINTER(VecOptions),
                                 C.POINTER(C.c_void_p)]
    L.lle_vec_destroy.argtypes = [C.c_void_p]
    L.lle_vec_get_buffers.argtypes = [C.c_void_p, C.POINTER(VecBuffers)]
    L.lle_vec_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_refresh.argtypes = [C.c_void_p, C.c_void_p]
    L.lle_vec_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_rollout.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.lle_vec_step_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_pipeline_submit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_pipeline_wait.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
    L.lle_vec_parts_begin.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_parts_count.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
    L.lle_vec_parts_range.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    for name in ("lle_vec_parts_launch", "lle_vec_parts_end", "lle_vec_parts_abort"):
        getattr(L, name).argtypes = [C.c_void_p]
    L.lle_vec_parts_feed.argtypes = [C.c_void_p, C.c_int32]
    L.lle_vec_parts_wait.argtypes = [C.c_void_p, C.c_int32]
    L.lle_vec_set_source.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    L.lle_vec_get_sources.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]
    L.lle_vec_set_exits.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_void_p]
    L.lle_vec_collect_gem.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    L.lle_vec_set_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_export_raw.argtypes = [C.c_void_p] + [C.c_void_p] * 8
    L.lle_vec_set_seed.argtypes = [C.c_void_p, C.c_uint64]
    L.lle_vec_get_step_count.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    L.lle_vec_set_step_count.argtypes = [C.c_void_p, C.c_uint64]
    L.lle_vec_launch_count.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    L.lle_vec_timing_begin.argtypes = [C.c_void_p, C.c_void_p]
    L.lle_vec_timing_end.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint64)]
    L.lle_vec_debug_timeline.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    L.lle_vec_export_raw_state.argtypes = [C.c_void_p, C.POINTER(RawState), C.c_void_p]
    L.lle_vec_import_raw_state.argtypes = [C.c_void_p, C.POINTER(RawState), C.c_void_p]
    L.lle_vec_get_reset_count.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    L.lle_vec_set_reset_count.argtypes = [C.c_void_p, C.c_uint32]
    L.lle_vec_fetch.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p]
    L.lle_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    L.lle_host_free.argtypes = [C.c_void_p]
    L.lle_gen_default_options.argtypes = [C.POINTER(GenOptions)]
    L.lle_gen_default_options.restype = None
    L.lle_gen_create.argtypes = [C.POINTER(GenOptions), C.c_int32, C.c_int64, C.POINTER(C.c_void_p)]
    L.lle_gen_destroy.argtypes = [C.c_void_p]
    L.lle_gen_attempt_seeds.argtypes = [C.c_uint64, C.c_int64, C.c_void_p]
    L.lle_gen_run.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64, C.c_int32, C.c_uint32, C.c_void_p]
    L.lle_gen_get_buffers.argtypes = [C.c_void_p, C.POINTER(GenBuffers)]
    L.lle_gen_fetch.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_gen_geometry_valid.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]
    L.lle_gen_cells_to_text.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.lle_plan.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_expert_build.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    L.lle_vec_expert_act.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lle_vec_expert_table.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    _lib = L
    return L


def last_error() -> str:
    return lib().lle_last_error().decode()


def check(status: int):
    """Map a status code to the exception the reference raises (src/bindings/pyexceptions.rs:43-183)."""
    if status == 0:
        return
    msg = last_error()
    if status == 5:
        raise InvalidLevelError(msg)
    if 1 <= status < 100:
        raise ParsingError(msg)
    if status == 101:
        raise InvalidActionError(msg)
    if status in (102, 103, 104, 107):
        raise InvalidWorldStateError(msg)
    if status in (105, 201):
        raise IndexError(msg)
    if status in (106, 110, 202):
        raise ValueError(msg)
    raise RuntimeError(f"lle_b200 error {status}: {msg}")
