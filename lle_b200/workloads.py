"""The five workloads of BASELINE.json (`configs[0..4]`, numbered 1..5 in SURVEY.md §8d) as batches of this library, and
the device-timed measurement `bench.py` and the parity tests share.

    1  World.level(1) — 1 agent, 1 gem, no beam — batched (the reference's CPU-runnable anchor)
    2  World.level(6) — 4 agents, 3 laser sources, 4 gems — 65,536 envs per GPU, layered observations (the headline)
    3  1,024 distinct generated 5x5 maps (2 agents, 2 sources) x 1,024 envs each: heterogeneous static planes in one batch.
       The maps come from this library's device generator (`lle_b200.generate(5, 5, 2).lasers(2)`: the reference's placement
       code re-implemented per seed, python/lle/generator/generator.py:188-228); the `cooperative()` SAT filter is NOT applied.
    4  the six built-in levels mixed, 2,097,152 envs per GPU, auto-reset: one sub-batch per level (channel counts differ),
       contiguous global env ids
    5  synthetic 64x64 map, 8 agents, 16 sources of mixed colours, 262,144 envs per GPU (86 GB of observations)
"""
from __future__ import annotations

import random
from dataclasses import dataclass

import numpy as np
import torch

from .env import VecWorldGroup
from .vec_world import Map, VecWorld

DEFAULT_ENVS = {1: 65536, 2: 65536, 3: 1 << 20, 4: 1 << 21, 5: 1 << 18}
DESCRIPTION = {
    1: "World.level(1), 1 agent (BASELINE configs[0] map, batched)",
    2: "World.level(6), 4 agents, 3 laser sources (BASELINE configs[1])",
    3: "1,024 device-generated 5x5 maps, 2 agents, 2 sources, x envs/1,024 each (BASELINE configs[2]; no cooperative() filter)",
    4: "levels 1-6 mixed, one sub-batch per level, auto-reset (BASELINE configs[3] per-GPU slice)",
    5: "synthetic 64x64, 8 agents, 16 sources of mixed colours (BASELINE configs[4])",
}


def synthetic_map(h: int, w: int, n_agents: int, n_sources: int, seed: int = 0, n_gems: int | None = None) -> str:
    """Seeded synthetic map in the v1 grammar (BASELINE config 5): border-free grid, starts on the first row,
    exits on the last row, laser sources of mixed colours and directions placed so that every beam is at most
    63 cells long and never crosses a start tile, a few walls and gems."""
    rng = random.Random(seed)
    grid = [["." for _ in range(w)] for _ in range(h)]
    start_cols = rng.sample(range(2, w - 2), n_agents)
    for a, j in enumerate(start_cols):
        grid[0][j] = f"S{a}"
    exit_cols = rng.sample(range(2, w - 2), n_agents)
    for j in exit_cols:
        grid[h - 1][j] = "X"
    used_rows, used_cols = {0, h - 1}, set(start_cols) | set(exit_cols)
    placed = 0
    attempts = 0
    while placed < n_sources and attempts < 10000:
        attempts += 1
        colour = placed % n_agents
        if rng.random() < 0.5:  # horizontal beam on a free row
            i = rng.randrange(2, h - 2)
            if i in used_rows:
                continue
            used_rows.add(i)
            if rng.random() < 0.5:
                grid[i][0] = f"L{colour}E"
            else:
                grid[i][w - 1] = f"L{colour}W"
            # a wall somewhere keeps the beam <= 63 cells on 64-wide maps
            grid[i][rng.randrange(w // 2, w - 1) if grid[i][0].startswith("L") else rng.randrange(1, w // 2)] = "@"
        else:  # vertical beam on a free column, starting below the start row
            j = rng.randrange(1, w - 1)
            if j in used_cols:
                continue
            used_cols.add(j)
            grid[1][j] = f"L{colour}S"
            grid[rng.randrange(h // 2, h - 1)][j] = "@"
        placed += 1
    free = [(i, j) for i in range(1, h - 1) for j in range(w) if grid[i][j] == "."]
    rng.shuffle(free)
    n_gems = n_agents if n_gems is None else n_gems
    for i, j in free[:n_gems]:
        grid[i][j] = "G"
    for i, j in free[n_gems : n_gems + (h * w) // 40]:
        grid[i][j] = "@"
    return "\n".join(" ".join(f"{t:>4}" for t in row) for row in grid)


def generated_maps(n: int = 1024, seed: int = 2026, device: int = 0) -> list[str]:
    """`n` distinct 5x5 / 2 agents / 2 sources layouts from the device generator that the map compiler accepts (a layout whose
    beam kills a start is refused by the reference's `World` constructor too: AgentWithoutStart)."""
    from .generator import generate
    from .types import ParsingError

    out = []
    for text in generate(5, 5, 2).lasers(2).take(4 * n, seed=seed, device=device, distinct=True, texts=True):
        try:
            Map(text)
        except ParsingError:
            continue
        out.append(text)
        if len(out) == n:
            return out
    raise RuntimeError(f"the generator produced only {len(out)} of {n} distinct maps")


@dataclass
class Workload:
    config: int
    parts: list[VecWorld]
    texts: list[str]               # the map texts (config 3: the generated maps; config 4: the six levels)
    map_of_env: np.ndarray | None  # config 3: map index of each local env
    description: str

    @property
    def n_envs(self) -> int:
        return sum(p.n_envs for p in self.parts)

    @property
    def agent_envs(self) -> int:
        return sum(p.n_envs * p.n_agents for p in self.parts)

    def step(self):
        """One lockstep step of every env with device-sampled actions (adjacent launches overlap, see VecWorldGroup)."""
        for p in self.parts:
            p.step(None)

    def algorithmic_bytes(self) -> int:
        """SURVEY.md §8(d): bytes that must cross HBM per step of the whole workload on this GPU."""
        return sum(algorithmic_bytes(p)["total"] * p.n_envs for p in self.parts)

    def measure(self, steps: int, warmup: int = 3) -> float:
        """ms per step, CUDA events on the launching stream, `warmup` untimed steps first."""
        for _ in range(max(warmup, 0)):
            self.step()
        dev = self.parts[0].device
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(dev))
        for _ in range(steps):
            self.step()
        e1.record(torch.cuda.current_stream(dev))
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / steps


def algorithmic_bytes(vec: VecWorld) -> dict:
    """SURVEY.md §8(d): B = OBS + ST + AV + AC + RDE + 2*S for one env-step of `vec`; OBS = the block `vec.obs` holds per env."""
    A, G, R = vec.n_agents, vec.n_gems, vec.reward_dim
    # the elements the observation generator materialises per env (layered / state: one copy viewed by every agent), at the
    # vec's element size (4 bytes, or 1 for obs_dtype=torch.int8)
    obs = vec.obs.element_size() * int(np.prod(vec.obs.shape[1:])) if vec.obs is not None else 0
    st, av, ac = 4 * (3 * A + G), 5 * A, A
    rde = 4 * R + 1 + A + 1  # reward, done, events, err
    return dict(obs=obs, state=st, avail=av, actions=ac, reward_done_events=rde, record_rw=2 * vec.record_bytes,
                total=obs + st + av + ac + rde + 2 * vec.record_bytes)


def level_text(n: int) -> str:
    return Map(level=n).text


def build(config: int, n_envs: int | None = None, *, device=0, seed: int = 2026, env_id_base: int = 0, **kw) -> Workload:
    """The workload of BASELINE config `config` (1..5) with `n_envs` envs on `device`; env ids start at `env_id_base`
    (range sharding over GPUs keeps every env's stream independent of the GPU count)."""
    n = int(n_envs or DEFAULT_ENVS[config])
    dev_index = torch.device(device if not isinstance(device, int) else f"cuda:{device}").index or 0
    if config in (1, 2):
        m = Map(level=1 if config == 1 else 6)
        return Workload(config, [VecWorld(m, n, device=device, seed=seed, env_id_base=env_id_base, **kw)], [m.text], None, DESCRIPTION[config])
    if config == 3:
        texts = generated_maps(1024, seed=seed, device=dev_index)
        moe = ((env_id_base + np.arange(n, dtype=np.int64)) // 1024 % 1024).astype(np.int32)  # global env e plays map (e // 1,024) mod 1,024
        vec = VecWorld([Map(t) for t in texts], n, map_of_env=moe, device=device, seed=seed, env_id_base=env_id_base, **kw)
        return Workload(config, [vec], texts, moe, DESCRIPTION[config])
    if config == 4:
        specs = [(Map(level=l), n // 6 + (1 if l <= n % 6 else 0)) for l in range(1, 7)]
        grp = VecWorldGroup(specs, device=device, seed=seed, env_id_base=env_id_base, **kw)
        return Workload(config, grp.parts, [m.text for m, _ in specs], None, DESCRIPTION[config])
    if config == 5:
        text = synthetic_map(64, 64, 8, 16, seed=5)
        return Workload(config, [VecWorld(Map(text), n, device=device, seed=seed, env_id_base=env_id_base, **kw)], [text], None, DESCRIPTION[config])
    raise ValueError(f"unknown config {config}")
