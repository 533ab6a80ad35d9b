"""Exact shortest death-free joint plans for batches of maps, searched on the device (include/lle_b200.h: lle_plan).

`plan(maps)` answers, per map and for this library's own rules, whether every agent can reach an exit without anybody dying,
in how many steps at least (a difficulty measure for curricula), and with which joint actions (an expert demonstration).
The search is a breadth-first search over joint states, one map per CTA; its rules, limits and the unique plan it returns
are documented with lle_plan.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Sequence

import numpy as np

from ._native import check, lib
from .vec_world import Map

PLAN_ALL_GEMS = 1  # LLE_PLAN_ALL_GEMS


class Plans(NamedTuple):
    length: np.ndarray    # int32 [M]: steps of the shortest plan, 0 when the reset state is a goal, -1 when none within max_steps
    n_states: np.ndarray  # int64 [M]: joint states the search reached
    actions: np.ndarray   # int8 [M, max_steps, 4]: Action values of agent a in column a; -1 past the plan and past n_agents


def plan(maps: Sequence[Map | str | int], *, max_steps: int = 64, all_gems: bool = False, device: int = 0) -> Plans:
    """Shortest plans of `maps` (`Map` objects, map texts or level numbers, as `VecWorld` takes them; the maps may differ in
    shape).  A goal is every agent on an exit, and with `all_gems` every gem collected as well.  Limits: at most 4 agents,
    (standable cells)^n_agents (times 2^n_gems with `all_gems`) <= 2^22, beams <= 32 cells, <= 32 gems, no random starts,
    1 <= max_steps <= 1024."""
    handles = [m if isinstance(m, Map) else (Map(level=m) if isinstance(m, int) else Map(m)) for m in maps]
    n = len(handles)
    length = np.zeros(n, np.int32)
    n_states = np.zeros(n, np.int64)
    actions = np.zeros((n, max(int(max_steps), 0), 4), np.int8)
    arr = (C.c_void_p * max(1, n))(*[m._h.value for m in handles])
    check(lib().lle_plan(arr, n, int(max_steps), PLAN_ALL_GEMS if all_gems else 0, int(device), length.ctypes.data_as(C.c_void_p),
                         n_states.ctypes.data_as(C.c_void_p), actions.ctypes.data_as(C.c_void_p)))
    return Plans(length, n_states, actions)
