"""The device expert (lle_vec_expert_*, VecWorld.build_expert / expert_actions / expert_table): exact distance-to-goal tables.

  * CPU: the expert core (lle_b200/csrc/expert_core.cuh, built with g++ through tests/host_shim/expert_host.cpp) against an
    independent computation over the oracle engine (a forward search over `World` that rebuilds states with `set_state`, then a
    reverse breadth-first search from the goals): the same reached set and the same dist for every key; every joint action of the
    table available, death-free, one step closer on the oracle, and the smallest such; dist at reset equal to the planner's length.
  * GPU: device tables byte-equal to the host core; expert_actions equal to a host lookup through the fetched tables from the
    raw engine state; closed loops on the device; set_state / dead agents / set_source invalidation; every refusal.
"""
import ctypes as C
import itertools
import os
import subprocess
from collections import defaultdict, deque

import numpy as np
import pytest

from _util import level_text
from oracle import lle_oracle as lo
from test_planner import CORRIDOR_WAIT, GEM_MAPS, NEEDS_BLOCKER, host_plan, layouts_in_limit, oracle_generated_maps

HERE = os.path.dirname(os.path.abspath(__file__))


def build_expert_host_shim() -> str:
    """g++ build of tests/host_shim/expert_host.cpp: the expert core plus the product's host map compiler.  Test infrastructure."""
    csrc = os.path.join(os.path.dirname(HERE), "lle_b200", "csrc")
    srcs = [os.path.join(HERE, "host_shim", "expert_host.cpp"), os.path.join(csrc, "map_compiler.cpp"), os.path.join(csrc, "toml_config.cpp")]
    out_dir = os.path.join(HERE, "host_shim", "_build")
    out = os.path.join(out_dir, "libexpert_host.so")
    deps = srcs + [os.path.join(csrc, f) for f in ("expert_core.cuh", "plan_core.cuh", "tiny_core.cuh", "step_common.cuh", "static_map.h",
                                                   "map_compiler.hpp", "toml_lite.hpp")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{out}.{os.getpid()}.tmp"
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++"] + srcs + ["-o", tmp], check=True)
        os.replace(tmp, out)
    return out


_SHIM = None


def host_expert(text, all_gems=False):
    """The host core on one map text: (dist i32[K], joint i16[K], n_states)."""
    global _SHIM
    if _SHIM is None:
        _SHIM = C.CDLL(build_expert_host_shim())
    K, n = C.c_int64(0), C.c_int64(0)
    err = C.create_string_buffer(512)
    rc = _SHIM.expert_host_build(text.encode(), int(all_gems), C.byref(K), C.byref(n), err, 512)
    assert rc == 0, err.value.decode()
    dist, joint = np.zeros(K.value, np.int32), np.zeros(K.value, np.int16)
    _SHIM.expert_host_fetch(dist.ctypes.data_as(C.c_void_p), joint.ctypes.data_as(C.c_void_p), None, None)
    return dist, joint, n.value


def standable_cells(text):
    """The standable cells (not wall, laser source or void) in row-major order, from the oracle: the digits of a state key."""
    w = lo.World(text)
    blocked = set(w.wall_pos) | set(w.void_pos) | {s.pos for s in w.laser_sources}
    return [(i, j) for i in range(w.height) for j in range(w.width) if (i, j) not in blocked]


def oracle_expert(text, all_gems=False):
    """An independent computation over the oracle engine.  Forward: every state reachable from reset without a death, each rebuilt
    from its key with `World.set_state` before each joint action (by replaying its first path from reset when set_state refuses
    it, as test_planner.oracle_bfs does); a state where every agent has arrived is not expanded.  Backward: a breadth-first search
    from the goals over the reversed transitions.  Returns (dist {key: d or -1}, edges {key: [(joint index, successor key)]})."""
    w = lo.World(text)
    w.reset()
    cells = standable_cells(text)
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
    is_over, is_goal = {start: over()}, {start: goal()}
    order, edges = [start], {}
    for k in order:  # grows while it is walked: a breadth-first enumeration
        if is_over[k]:
            continue
        rebuild(k)
        out = []
        for joint in itertools.product(*w.available_actions()):
            rebuild(k)
            w.step(list(joint))
            if not all(a.is_alive for a in w.agents):
                continue
            k2 = key(w.get_state())
            out.append((sum(int(a) * 5 ** i for i, a in enumerate(joint)), k2))
            if k2 not in parent:
                parent[k2] = (k, list(joint))
                is_over[k2], is_goal[k2] = over(), goal()
                order.append(k2)
        edges[k] = out
    preds = defaultdict(set)
    for k, out in edges.items():
        for _, k2 in out:
            preds[k2].add(k)
    dist = {k: 0 for k in order if is_goal[k]}
    queue = deque(dist)
    while queue:
        k = queue.popleft()
        for p in preds[k]:
            if p not in dist:
                dist[p] = dist[k] + 1
                queue.append(p)
    return {k: dist.get(k, -1) for k in order}, edges


# ------------------------------------------------------------------------------------------------------------------- CPU
def _check_against_oracle(texts, all_gems=False):
    for text in texts:
        dist, joint, n_states = host_expert(text, all_gems)
        want, edges = oracle_expert(text, all_gems)
        reached = np.flatnonzero(dist != -2)
        assert n_states == len(want) == len(reached), text
        assert set(reached.tolist()) == set(want), text
        assert all(dist[k] == d for k, d in want.items()), text
        assert (joint[dist <= 0] == -1).all(), text
        for k in np.flatnonzero(dist > 0).tolist():
            out = dict(edges[k])  # joint index -> successor: the available, death-free joint actions of the oracle
            j = int(joint[k])
            assert j in out and dist[out[j]] == dist[k] - 1, (text, k)
            assert all(dist[k2] != dist[k] - 1 for j2, k2 in out.items() if j2 < j), (text, k)
        length, _, _ = host_plan([text], 1024, all_gems)
        assert int(length[0]) == int(dist[_reset_key(text, all_gems)]), text


def _reset_key(text, all_gems=False):
    w = lo.World(text)
    w.reset()
    st = w.get_state()
    cells = standable_cells(text)
    index = {c: k for k, c in enumerate(cells)}
    k = sum(1 << g for g, c in enumerate(st.gems_collected) if c) if all_gems else 0
    for p in reversed(st.agents_positions):
        k = k * len(cells) + index[tuple(p)]
    return k


def test_host_core_level1_and_small_layouts_match_the_oracle():
    layouts = layouts_in_limit()
    small = [layouts[n] for n in sorted(layouts) if not n.startswith("level-")]  # levels 2-4: next test
    assert len(small) >= 20
    _check_against_oracle([level_text(1)] + small)


def test_host_core_levels_2_to_4_match_the_oracle():
    layouts = layouts_in_limit()
    _check_against_oracle([layouts[f"level-{n}"] for n in (2, 3, 4)])


def test_host_core_generated_maps_match_the_oracle():
    maps = oracle_generated_maps(48)
    _check_against_oracle(maps)
    d = [host_expert(t)[0] for t in maps]
    assert sum((x[_reset_key(t)] > 0) for x, t in zip(d, maps)) > 10 and any((x == -1).any() for x in d)


@pytest.mark.parametrize("all_gems", [False, True])
def test_host_core_gem_maps_match_the_oracle(all_gems):
    _check_against_oracle(GEM_MAPS, all_gems)


def test_host_core_blocker_and_corridor_maps_match_the_oracle():
    _check_against_oracle([NEEDS_BLOCKER, CORRIDOR_WAIT])
    dist, joint, _ = host_expert(CORRIDOR_WAIT)
    assert dist[_reset_key(CORRIDOR_WAIT)] == 4


def test_null_arguments_are_refused_without_a_device():
    from lle_b200 import _native

    L = _native.lib()
    n = C.c_int64(0)
    assert L.lle_vec_expert_build(None, 0, None, None) == 202
    assert L.lle_vec_expert_act(None, None, None, None) == 202
    assert L.lle_vec_expert_table(None, 0, None, None, 0, C.byref(n)) == 202


# ------------------------------------------------------------------------------------------------------------------- GPU
def _vec(maps, n_envs, **kw):
    import lle_b200

    return lle_b200.VecWorld(maps, n_envs, map_of_env=[e % len(maps) for e in range(n_envs)], device=0, **kw)


def _tables_match_host(texts, all_gems=False, **kw):
    vec = _vec(texts, len(texts), **kw)
    n_states = vec.build_expert(all_gems)
    for m, text in enumerate(texts):
        dist, joint, n = host_expert(text, all_gems)
        got_d, got_j = vec.expert_table(m)
        assert n_states[m] == n, m
        assert got_d.tobytes() == dist.tobytes() and got_j.tobytes() == joint.tobytes(), m
    return vec, n_states


def _config3_maps():
    from lle_b200.workloads import generated_maps

    return generated_maps(1024)


@pytest.mark.gpu
@pytest.mark.parametrize("all_gems", [False, True])
def test_device_tables_config3_equal_the_host_core(all_gems):
    _tables_match_host(_config3_maps(), all_gems)


@pytest.mark.gpu
def test_device_tables_levels_equal_the_host_core():
    for n in (1, 2, 3, 4):
        vec, n_states = _tables_match_host([level_text(n)])
        assert n_states[0] > 1


@pytest.mark.gpu
def test_device_tables_other_generator_shapes_equal_the_host_core():
    from test_planner import _other_generator_maps

    def small(texts, n):  # the host core's cost grows with K: the n maps of smallest K
        return sorted(texts, key=lambda t: len(standable_cells(t)) ** lo.World(t).n_agents)[:n]

    groups = _other_generator_maps()
    assert groups[0] and groups[2]
    for texts, n in zip(groups, (12, 4, 32)):  # 8x7 with 3 agents, 9x9 rooms with 4 agents (none within the limits), 10x6 with 2
        if texts:
            _tables_match_host(small(texts, n))
    _tables_match_host(small(groups[2], 16), all_gems=True)  # 10x6 maps with 2 gems


def _host_lookup(vec, texts, tables, all_gems=False):
    """expert_actions of every env of `vec` computed on the host: key from export_raw (positions, alive flags, gems) through the
    oracle's standable cells, then the fetched table of the env's map."""
    raw = {k: v.cpu().numpy().astype(np.int64) for k, v in vec.export_raw().items()}
    N, A, HW = vec.n_envs, vec.n_agents, vec.height * vec.width
    moe = vec.map_index.cpu().numpy().astype(np.int64) if vec.map_index is not None else np.zeros(N, np.int64)
    ci = np.full((len(texts), HW), -1, np.int64)
    nc = np.zeros(len(texts), np.int64)
    for m, text in enumerate(texts):
        cells = standable_cells(text)
        nc[m] = len(cells)
        for k, (i, j) in enumerate(cells):
            ci[m, i * vec.width + j] = k
    off = np.concatenate([[0], np.cumsum([len(d) for d, _ in tables])])
    all_d = np.concatenate([d for d, _ in tables])
    all_j = np.concatenate([j for _, j in tables]).astype(np.int64)
    key = raw["collected"].copy() if all_gems else np.zeros(N, np.int64)
    for a in reversed(range(A)):
        key = key * nc[moe] + ci[moe, raw["pos"][:, a, 0] * vec.width + raw["pos"][:, a, 1]]
    alive = raw["alive"].all(axis=1)
    at = off[moe] + key
    dist = np.where(alive, all_d[np.where(alive, at, 0)], -2).astype(np.int32)
    j = np.where(dist > 0, all_j[np.where(alive, at, 0)], 4 * sum(5 ** a for a in range(A)))
    act = np.stack([(j // 5 ** a) % 5 for a in range(A)], axis=1).astype(np.int8)
    return act, dist


def _query_matches_host(texts, n_envs, steps=(0, 1, 37), **kw):
    vec = _vec(texts, n_envs, **kw)
    vec.build_expert()
    tables = [vec.expert_table(m) for m in range(len(texts))]
    done_steps = 0
    for t in steps:
        for _ in range(t - done_steps):
            vec.step(None)
        done_steps = t
        launches = vec.launch_count
        act, dist = vec.expert_actions()
        assert vec.launch_count == launches + 1
        want_act, want_dist = _host_lookup(vec, texts, tables)
        assert np.array_equal(dist.cpu().numpy(), want_dist), t
        assert np.array_equal(act.cpu().numpy(), want_act), t
        assert (want_dist >= -1).all()  # every world stepped without a death is in the table (deaths reset it)
    return vec


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [{}, {"obs_dtype": "int8"}, {"obs_type": "partial7x7"}, {"extras": "laser_subgoal"}],
                         ids=["f32", "int8", "partial7x7", "laser_subgoal"])
def test_expert_actions_config3_equal_a_host_lookup(kw):
    _query_matches_host(_config3_maps(), 65536, **kw)


@pytest.mark.gpu
def test_expert_actions_levels_equal_a_host_lookup():
    for n in (1, 2, 3, 4):
        _query_matches_host([level_text(n)], 4096)


@pytest.mark.gpu
def test_closed_loop_on_the_device():
    import torch

    texts = _config3_maps()
    vec = _vec(texts, 65536, auto_reset=False)
    vec.build_expert()
    act, dist = vec.expert_actions()
    d0 = dist.clone()
    assert (d0 >= -1).all() and (d0 > 0).sum() > 50000 and (d0 == -1).any()
    for t in range(int(d0.max())):
        vec.step(act)
        act, dist = vec.expert_actions(act, dist)
        live = d0 > t  # worlds whose episode includes step t
        assert (vec.err[live] == 0).all(), t
        finishing = d0 == t + 1
        assert torch.equal(vec.done[live].bool(), finishing[live]), t
        assert (dist[live] == d0[live] - t - 1).all(), t
        none = d0 == -1
        assert (vec.done[none] == 0).all() and (vec.err[none] == 0).all() and (dist[none] == -1).all(), t
    raw = vec.export_raw()
    solvable = d0 >= 0
    assert raw["alive"][solvable].all() and raw["arrived"][solvable].all()
    # auto-reset: every finished episode of a solvable map lasts exactly its reset distance
    vec = _vec(texts, 65536, episode_stats=True)
    vec.build_expert()
    act, dist = vec.expert_actions()
    d0 = dist.clone()
    for _ in range(int(d0.max())):
        vec.step(act)
        vec.expert_actions(act, dist)
    vec.synchronize()
    assert torch.equal(vec.last_length[d0 > 0], d0[d0 > 0]) and (vec.last_length[d0 == -1] == 0).all()


@pytest.mark.gpu
def test_states_outside_the_table():
    import torch

    text = "S0 . @ . X\n. . @ . ."  # the right half, with the exit, is out of reach
    vec = _vec([text], 2)
    n_states = vec.build_expert()
    assert n_states[0] == 4
    act, dist = vec.expert_actions()
    assert (dist == -1).all() and (act == 4).all()
    pos = torch.tensor([[[0, 3]], [[0, 0]]], dtype=torch.int32)
    vec.set_state(pos, torch.zeros((2, 0), dtype=torch.uint8), torch.tensor([[1], [0]], dtype=torch.uint8))
    act, dist = vec.expert_actions()
    assert dist.tolist() == [-2, -2] and (act == 4).all()  # not reached / a dead agent


@pytest.mark.gpu
def test_set_source_drops_the_tables_until_a_rebuild():
    vec = _vec([NEEDS_BLOCKER], 8)
    vec.build_expert()
    vec.set_source(0, enabled=False)
    with pytest.raises(ValueError, match="no tables"):
        vec.expert_actions()
    with pytest.raises(ValueError, match="no tables"):
        vec.expert_table(0)
    n_states = vec.build_expert()
    dist, joint, n = host_expert(NEEDS_BLOCKER.replace("L1E", "@"))
    got_d, got_j = vec.expert_table(0)
    assert n_states[0] == n and got_d.tobytes() == dist.tobytes() and got_j.tobytes() == joint.tobytes()
    vec.expert_actions()


@pytest.mark.gpu
def test_collect_gem_keeps_the_tables():
    vec = _vec([GEM_MAPS[1]], 8)
    vec.build_expert()
    vec.collect_gem(0)
    vec.refresh()
    vec.expert_actions()


@pytest.mark.gpu
def test_refusals():
    import torch

    import lle_b200
    from lle_b200 import _native

    L = _native.lib()
    ok = level_text(1)
    vec = _vec([ok], 64)
    n = C.c_int64(0)
    assert L.lle_vec_expert_act(vec._h, torch.zeros((64, 1), dtype=torch.int8, device="cuda").data_ptr(), None, None) == 202  # no build
    assert L.lle_vec_expert_table(vec._h, 0, None, None, 0, C.byref(n)) == 202
    assert L.lle_vec_expert_build(vec._h, 2, None, None) == 202  # unknown flag
    vec.build_expert()
    assert L.lle_vec_expert_act(vec._h, None, None, None) == 202
    assert L.lle_vec_expert_table(vec._h, 1, None, None, 0, C.byref(n)) == 202
    assert L.lle_vec_expert_table(vec._h, 0, None, None, -1, C.byref(n)) == 202
    assert L.lle_vec_expert_table(vec._h, 0, None, None, 0, None) == 202
    assert L.lle_vec_expert_table(vec._h, 0, None, None, 0, C.byref(n)) == 0 and n.value == 156
    for maps, match in (([5], "map 0"), ([6], "map 0")):
        with pytest.raises(lle_b200.types.ParsingError, match=match):
            _vec(maps, 4).build_expert()
    import json

    from _util import GOLDEN

    eight = json.load(open(os.path.join(GOLDEN, "layouts.json")))["eight-agent-interdependent-8"]
    with pytest.raises(lle_b200.types.ParsingError, match="more than 4 agents"):
        _vec([eight], 4).build_expert()
    with pytest.raises(ValueError, match="walkable_lasers"):
        _vec([ok], 4, walkable_lasers=False).build_expert()
    with pytest.raises(ValueError, match="randomize_lasers"):
        _vec([ok], 4, randomize_lasers=True).build_expert()
    starts = 'world_string = """\n. . X\n. . X\n"""\n[[agents]]\nstarts = [{ i = 0, j = 0 }, { i = 0, j = 1 }]\n[[agents]]\nstarts = [{ i = 0, j = 0 }]\n'
    with pytest.raises(ValueError, match="random start"):
        _vec([starts], 4).build_expert()
    # pipelined steps outstanding
    reward = torch.zeros((64, 1), dtype=torch.float32).pin_memory()
    done = torch.zeros(64, dtype=torch.uint8).pin_memory()
    vec.submit_host(None, reward, done)
    with pytest.raises(ValueError, match="outstanding"):
        vec.build_expert()
    with pytest.raises(ValueError, match="outstanding"):
        vec.expert_actions()
    vec.wait_host()
    vec.expert_actions()
    with pytest.raises(ValueError):
        vec.expert_actions(torch.zeros((64, 2), dtype=torch.int8, device="cuda"))
