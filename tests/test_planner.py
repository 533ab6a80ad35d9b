"""The planner (lle_plan, lle_b200/planner.py): exact shortest death-free joint plans.

  * CPU: the planning core (lle_b200/csrc/plan_core.cuh, built with g++ through tests/host_shim/plan_host.cpp) against an
    independent breadth-first search over the oracle engine that rebuilds every state from its key with `set_state` — same
    length and same number of reached states; every host plan replayed on the oracle `LLE`; the argument and limit refusals
    of lle_plan, which happen before any device call.
  * GPU: the device planner byte for byte against the host core (config 3's 1,024 maps and three other generator
    configurations), its plans replayed through `VecWorld`, and `GeneratorBuilder.plannable`.
"""
import ctypes as C
import itertools
import json
import os
import subprocess

import numpy as np
import pytest

from _util import GOLDEN, level_text
from oracle import generator as og
from oracle import lle_oracle as lo

HERE = os.path.dirname(os.path.abspath(__file__))


def build_plan_host_shim() -> str:
    """g++ build of tests/host_shim/plan_host.cpp: the planning core (lle_b200/csrc/plan_core.cuh, __host__ __device__) plus
    the product's host map compiler, for the test-suite.  Test infrastructure only."""
    csrc = os.path.join(os.path.dirname(HERE), "lle_b200", "csrc")
    srcs = [os.path.join(HERE, "host_shim", "plan_host.cpp"), os.path.join(csrc, "map_compiler.cpp"), os.path.join(csrc, "toml_config.cpp")]
    out_dir = os.path.join(HERE, "host_shim", "_build")
    out = os.path.join(out_dir, "libplan_host.so")
    deps = srcs + [os.path.join(csrc, f) for f in ("plan_core.cuh", "tiny_core.cuh", "step_common.cuh", "static_map.h", "map_compiler.hpp", "toml_lite.hpp")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{out}.{os.getpid()}.tmp"
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++"] + srcs + ["-o", tmp], check=True)
        os.replace(tmp, out)
    return out


_SHIM = None


def host_plan(texts, max_steps=64, all_gems=False):
    """The host core on map texts: (length i32[n], n_states i64[n], actions i8[n, max_steps, 4])."""
    global _SHIM
    if _SHIM is None:
        _SHIM = C.CDLL(build_plan_host_shim())
    n = len(texts)
    arr = (C.c_char_p * max(1, n))(*[t.encode() for t in texts])
    length, n_states = np.zeros(n, np.int32), np.zeros(n, np.int64)
    actions = np.zeros((n, max_steps, 4), np.int8)
    err = C.create_string_buffer(512)
    rc = _SHIM.plan_host(arr, n, max_steps, int(all_gems), length.ctypes.data_as(C.c_void_p), n_states.ctypes.data_as(C.c_void_p),
                         actions.ctypes.data_as(C.c_void_p), err, 512)
    assert rc == 0, err.value.decode()
    return length, n_states, actions


def host_limit_status(text, all_gems=False):
    """0 when the map is within the planner's limits, else the LLE_* status of the host core."""
    global _SHIM
    if _SHIM is None:
        _SHIM = C.CDLL(build_plan_host_shim())
    arr = (C.c_char_p * 1)(text.encode())
    length, n_states, actions = np.zeros(1, np.int32), np.zeros(1, np.int64), np.zeros((1, 1, 4), np.int8)
    # max_steps = 1: a one-depth search, cheap for any map within the limits
    return _SHIM.plan_host(arr, 1, 1, int(all_gems), length.ctypes.data_as(C.c_void_p), n_states.ctypes.data_as(C.c_void_p),
                           actions.ctypes.data_as(C.c_void_p), None, 0)


def oracle_bfs(text, max_steps, all_gems=False):
    """An independent search over the oracle engine: every state is rebuilt from its key (positions, and the gem mask with
    all_gems) with World.set_state before each joint action; successors in which an agent died are dropped.  Same stop rule
    as the planner.  Returns (length, n_states).
    set_state enters the agents one after the other, so it refuses a state where an agent stands in a beam that only a later
    agent blocks (InvalidWorldState); such a state is rebuilt by replaying, from reset, the path that first reached it."""
    w = lo.World(text)
    w.reset()
    blocked = set(w.wall_pos) | set(w.void_pos) | {s.pos for s in w.laser_sources}
    cells = [(i, j) for i in range(w.height) for j in range(w.width) if (i, j) not in blocked]
    index = {c: k for k, c in enumerate(cells)}
    A, G, nc = w.n_agents, w.n_gems, len(cells)
    gem_cells = [g.pos for g in w.gems]

    def key(state):
        k = sum(1 << g for g, c in enumerate(state.gems_collected) if c) if all_gems else 0
        for p in reversed(state.agents_positions):
            k = k * nc + index[tuple(p)]
        return k

    def rebuild(k):
        pos, rest = [], k
        for _ in range(A):
            pos.append(cells[rest % nc])
            rest //= nc
        # without all_gems the key holds no gem mask; a gem under an agent is collected in every state that reaches it
        try:
            w.set_state(lo.WorldState(pos, [bool((rest >> g) & 1) or gem_cells[g] in pos for g in range(G)], [True] * A))
        except lo.InvalidWorldStateError:
            path = []
            while k != start:
                k, joint = parent[k]
                path.append(joint)
            w.reset()
            for joint in reversed(path):
                w.step(joint)

    def over():
        return all(a.has_arrived for a in w.agents)

    def goal():
        return over() and (not all_gems or all(w.get_state().gems_collected))

    start = key(w.get_state())
    parent = {start: None}
    if goal():
        return 0, 1
    if over():
        return -1, 1
    frontier = [start]
    for depth in range(max_steps):
        nxt, found = [], False
        for k in frontier:
            rebuild(k)
            for joint in itertools.product(*w.available_actions()):
                rebuild(k)
                w.step(list(joint))
                if not all(a.is_alive for a in w.agents):
                    continue
                k2 = key(w.get_state())
                if k2 in parent:
                    continue
                parent[k2] = (k, list(joint))
                if goal():
                    found = True
                elif not over():
                    nxt.append(k2)
        if found:
            return depth + 1, len(parent)
        if not nxt:
            return -1, len(parent)
        frontier = nxt
    return -1, len(parent)


def replay_on_oracle(text, length, actions, all_gems=False):
    """Replays one plan on the oracle LLE from reset: nobody dies, everybody arrives at the last step and not before, and with
    all_gems every gem is collected by then."""
    env = lo.LLE(text)
    env.reset()
    A, G = env.n_agents, env.n_gems
    assert (actions[length:] == -1).all() and (actions[:, A:] == -1).all()
    if length == 0:
        assert env.n_arrived == A
    for t in range(length):
        assert env.n_arrived < A, t
        step = env.step([int(a) for a in actions[t, :A]])
        assert not any(e.event_type == lo.EventType.AGENT_DIED for e in step.events), t
        assert step.done == (t == length - 1), t
    assert env.n_arrived == A
    if all_gems:
        assert env.state_array()[2 * A:2 * A + G].all()


# ---- maps
GEM_MAPS = [
    "S0 . G . X",
    "S0 . . G\n. @ . .\nG . . X",
    "S0 S1 . G\n. @ . .\nG . X X",
    ". G . S0\nL1E . . .\nS1 . G X\n. . . X",
]
NEEDS_BLOCKER = "S0 . .\nL1E . .\nX S1 X"    # agent 0 crosses the beam of colour 1 only while agent 1 stands in it
CORRIDOR_WAIT = "@ S1 @ @\nS0 . . X\n@ X @ @"  # both agents must pass the corridor cell (1, 1), one after the other


def layouts_in_limit():
    with open(os.path.join(GOLDEN, "layouts.json")) as f:
        layouts = json.load(f)
    return {name: text for name, text in layouts.items() if host_limit_status(text) == 0}


def oracle_generated_maps(n=48, seed=3):
    """`n` distinct 5x5, 2-agent, 2-laser maps of the oracle generator that the map compiler accepts."""
    cfg = og.GenConfig(width=5, height=5, n_agents=2, n_lasers=2)
    out = []
    for s in og.attempt_seeds(seed, 2000):
        lay = og.try_generate(cfg, s)
        if lay is None:
            continue
        text = lay.to_v1()
        try:
            lo.World(text)
        except lo.ParsingError:
            continue
        if text not in out:
            out.append(text)
        if len(out) == n:
            return out
    raise AssertionError(f"only {len(out)} maps")


# ------------------------------------------------------------------------------------------------------------------- CPU
def _compare(texts, max_steps, all_gems=False):
    length, n_states, actions = host_plan(texts, max_steps, all_gems)
    for k, text in enumerate(texts):
        assert (int(length[k]), int(n_states[k])) == oracle_bfs(text, max_steps, all_gems), (k, text)
        if length[k] >= 0:
            replay_on_oracle(text, int(length[k]), actions[k], all_gems)
    return length, n_states


def test_host_core_level1_and_layouts_match_an_oracle_search():
    layouts = layouts_in_limit()
    assert "blocked-unsolvable" in layouts and len(layouts) >= 20
    names = sorted(layouts)
    length, _ = _compare([level_text(1)] + [layouts[n] for n in names], 24)
    assert length[0] == 10
    assert length[1 + names.index("blocked-unsolvable")] == -1


def test_host_core_generated_maps_match_an_oracle_search():
    length, _ = _compare(oracle_generated_maps(48), 16)
    assert (length > 0).sum() > 10 and (length == -1).sum() > 0


@pytest.mark.parametrize("all_gems", [False, True])
def test_host_core_gem_maps_match_an_oracle_search(all_gems):
    length, _ = _compare(GEM_MAPS, 20, all_gems)
    plain, _, _ = host_plan(GEM_MAPS, 20, False)
    assert (length >= plain).all() and (length > plain).any() == all_gems


def test_host_core_hand_made_cases():
    length, _ = _compare([NEEDS_BLOCKER, CORRIDOR_WAIT], 16)
    _, _, act = host_plan([NEEDS_BLOCKER, CORRIDOR_WAIT], 16)
    # needs a blocker: agent 1 steps north into its own beam at some point, although its exits are beside it
    assert length[0] > 0 and (act[0, : length[0], 1] == 0).any()
    # the corridor: an agent cannot enter an occupied cell, so one agent waits while the other clears (1, 1)
    assert length[1] == 4 and (act[1, :4, :2] == 4).any()


def test_host_core_stops_at_once_when_the_reset_state_is_over():
    """The search of a map whose agents cannot move at all: only the reset state is reached.  (A reset state that is already a
    goal - length 0 - would need a start on an exit, which the parser refuses: AgentWithoutStart.)"""
    length, n_states, act = host_plan(["S0 @ X"], 8)
    assert (int(length[0]), int(n_states[0])) == (-1, 1) == oracle_bfs("S0 @ X", 8) and (act == -1).all()
    with pytest.raises(lo.ParsingError):
        lo.World('world_string = """\nX . .\n"""\n[[agents]]\nstart_positions = [{ i = 0, j = 0 }]\n')


def test_argument_and_limit_refusals_before_any_device_call():
    """lle_plan checks every argument and every map before it touches a device (this runs without one)."""
    from lle_b200 import _native
    from lle_b200.planner import plan
    from lle_b200.types import ParsingError

    L = _native.lib()
    length, n_states, actions = np.zeros(2, np.int32), np.zeros(2, np.int64), np.zeros((2, 8, 4), np.int8)
    ok = lo.level_text(1)
    from lle_b200.vec_world import Map

    maps = [Map(ok), Map(level=6)]
    handles = (C.c_void_p * 2)(maps[0]._h.value, maps[1]._h.value)
    args = lambda n, steps, flags, dev: (handles, n, steps, flags, dev, length.ctypes.data, n_states.ctypes.data, actions.ctypes.data)
    assert L.lle_plan(*args(1, 0, 0, 0)) == 202
    assert L.lle_plan(*args(1, 1025, 0, 0)) == 202
    assert L.lle_plan(*args(1, 8, 2, 0)) == 202
    assert L.lle_plan(*args(1, 8, 0, -1)) == 202
    assert L.lle_plan(*args(-1, 8, 0, 0)) == 202
    assert L.lle_plan(handles, 1, 8, 0, 0, None, None, None) == 202
    assert L.lle_plan(*args(2, 8, 0, 0)) == 21 and "map 1" in _native.last_error()
    nulls = (C.c_void_p * 2)(maps[0]._h.value, None)
    assert L.lle_plan(nulls, 2, 8, 0, 0, length.ctypes.data, n_states.ctypes.data, actions.ctypes.data) == 202
    assert L.lle_plan(None, 0, 8, 0, 0, None, None, None) == 0  # nothing to plan
    with pytest.raises(ValueError):
        plan([ok], max_steps=0)
    with pytest.raises(ParsingError, match="more than 4 agents"):
        plan([ok, lo.level_text(1), json.load(open(os.path.join(GOLDEN, "layouts.json")))["eight-agent-interdependent-8"]])
    with pytest.raises(ParsingError, match="2\\^22"):
        plan([6])
    with pytest.raises(ValueError, match="random start"):
        plan(['world_string = """\n. . X\n. . X\n"""\n[[agents]]\nstarts = [{ i = 0, j = 0 }, { i = 0, j = 1 }]\n[[agents]]\nstarts = [{ i = 0, j = 0 }]\n'])
    assert plan([], max_steps=4).length.shape == (0,)


# ------------------------------------------------------------------------------------------------------------------- GPU
def _other_generator_maps():
    from lle_b200.generator import WorldGenerator

    configs = [
        dict(width=8, height=7, n_agents=3, starts="edge", exits="opposite", n_lasers=2, laser_placement="cross-agent", n_walls=5,
             walls_style="shapes", n_gems=3),
        dict(width=9, height=9, n_agents=4, n_lasers=3, n_gems=4, n_rooms_rows=2, n_rooms_cols=2, door_size=1),
        dict(width=10, height=6, n_agents=2, starts="clustered", exits="opposite", n_lasers=2, laser_placement="cross-cluster",
             cluster_shape=(2, 1), n_walls=4, n_gems=2),
    ]
    out = []
    for kw in configs:
        maps = list(WorldGenerator(**kw, batch=4096).generate_n(160, seed=21, distinct=True))
        out.append([m for m in maps if host_limit_status(m) == 0])
    return out


def _device_matches_host(texts, max_steps, all_gems=False):
    from lle_b200.planner import plan

    got = plan(texts, max_steps=max_steps, all_gems=all_gems)
    length, n_states, actions = host_plan(texts, max_steps, all_gems)
    assert np.array_equal(got.length, length) and np.array_equal(got.n_states, n_states)
    assert got.actions.tobytes() == actions.tobytes()
    return got


def _replay_on_vec(texts, got):
    """One env per map, supplied actions, LLE semantics, no auto-reset: every plan ends done with every agent arrived."""
    import torch

    import lle_b200

    keep = [k for k in range(len(texts)) if got.length[k] > 0]
    if not keep:
        return
    maps = [texts[k] for k in keep]
    lengths = got.length[keep]
    vec = lle_b200.VecWorld(maps, len(maps), map_of_env=list(range(len(maps))), device=0, auto_reset=False, episode_stats=True)
    A = vec.n_agents
    finished = np.zeros(len(maps), bool)
    for t in range(int(lengths.max())):
        act = np.where((t < lengths)[:, None], got.actions[keep, min(t, got.actions.shape[1] - 1), :A], 4).astype(np.int8)
        vec.step(torch.from_numpy(act).to(vec.device))
        done, err, info = vec.done.cpu().numpy(), vec.err.cpu().numpy(), vec.info_bytes.cpu().numpy()
        live = t < lengths
        assert (err[live] == 0).all(), t
        assert (done[live] == (t == lengths - 1)[live]).all(), t
        last = t == lengths - 1
        assert (info[last, 1] == A).all(), t  # n_arrived
        finished |= last
    assert finished.all()


@pytest.mark.gpu
def test_device_plans_config3_maps_equal_the_host_core():
    from lle_b200.workloads import generated_maps

    texts = generated_maps(1024)
    got = _device_matches_host(texts, 64)
    assert (got.length > 0).sum() > 100
    _replay_on_vec(texts, got)
    got = _device_matches_host(texts, 64, all_gems=True)  # no gems on these maps: the same plans
    _replay_on_vec(texts, got)


@pytest.mark.gpu
def test_device_plans_other_generated_shapes_equal_the_host_core():
    groups = _other_generator_maps()
    assert sum(len(g) for g in groups) >= 160
    for texts in groups:
        if not texts:
            continue
        got = _device_matches_host(texts, 40)
        _replay_on_vec(texts, got)
    _device_matches_host(groups[2][:40], 40, all_gems=True)  # 10x6 maps with 2 gems


@pytest.mark.gpu
def test_device_plans_levels_layouts_and_hand_made_maps():
    layouts = layouts_in_limit()
    texts = [level_text(1), NEEDS_BLOCKER, CORRIDOR_WAIT] + [layouts[n] for n in sorted(layouts)] + GEM_MAPS
    for all_gems in (False, True):
        for steps in (1, 7, 64):
            _device_matches_host(texts, steps, all_gems)


@pytest.mark.gpu
def test_generator_plannable_filter():
    from lle_b200.generator import generate
    from lle_b200.types import ParsingError
    from lle_b200.vec_world import Map

    got = list(generate(5, 5, 2).lasers(2).plannable(12).take(64, seed=0, texts=True))
    candidates = []
    for text in generate(5, 5, 2).lasers(2).take(4096, seed=0, texts=True):
        try:
            Map(text)
        except ParsingError:
            continue
        candidates.append(text)
    length, _, _ = host_plan(candidates, 12)
    want = [t for t, n in zip(candidates, length) if n >= 0][:64]
    assert len(want) == 64 and got == want
    world = generate(5, 5, 2).lasers(2).plannable(12).build(seed=0)
    assert world is not None and world.world_string == want[0]
    with pytest.raises(NotImplementedError):
        generate(5, 5, 2).solvable()
