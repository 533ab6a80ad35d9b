"""Procedural layout generation on the device: host mirror of `lle.generator` (python/lle/generator/__init__.py,
generator.py, builder.py) over the lle_gen_* entry points of include/lle_b200.h.

`WorldGenerator(...)` takes the reference's keyword arguments (generator.py:97-114).  One device thread runs one
*attempt* (`_try_generate(seed)`, generator.py:243-254) or one *chain* (`generate(max_attempts, seed)`, :268-284) with a
re-implementation of CPython's `random.Random`, so a seed gives the reference's layout bit for bit; `generate_n` follows
the reference's parallel path `_generate_n_multi` (:296-314: attempt i is seeded with the i-th
`rng.randrange(sys.maxsize)`), taking the accepted attempts in attempt order (the reference's `imap_unordered` leaves the
order to the scheduler).

Differences, all documented in include/lle_b200.h: the SAT-based `Constraint` is replaced by `require`, a mask of
breadth-first reachability labels (`WALKABLE`, `INDEPENDENT`, `NEEDS_BLOCKER`) that is a heuristic of this library, not
`Cooperative()` / `Independent()`; `cluster_shape` is explicit (the reference draws it from the global unseeded generator).
There is no CPU fallback: without the CUDA extension and a device these calls raise.
"""
from __future__ import annotations

import ctypes as C
import math
import random as _random
import sys
from typing import Iterator, Literal, Sequence

import numpy as np
import torch

from . import _native
from ._native import check, lib

WALKABLE, INDEPENDENT, NEEDS_BLOCKER = 1, 2, 4

_STARTS = {"random": 0, "edge": 1, "clustered": 2}
_EXITS = {"random": 0, "edge": 1, "cluster": 2, "opposite": 3}
_PLACEMENT = {"free": 0, "cross-agent": 1, "cross-cluster": 2}


def _default_cluster_shape(n_agents: int) -> tuple[int, int]:
    """The first alternative of placements.cluster_shape (placements.py:44-60); pass `cluster_shape` to choose another."""
    return {1: (1, 1), 2: (1, 2), 3: (1, 3), 4: (2, 2)}.get(n_agents, (1, n_agents))


def cells_to_text(cells: np.ndarray | torch.Tensor, height: int, width: int) -> str:
    """world_builder.py:83-88 via lle_gen_cells_to_text."""
    arr = np.ascontiguousarray(cells.cpu().numpy() if isinstance(cells, torch.Tensor) else cells, dtype=np.uint8).reshape(-1)
    n = C.c_size_t(0)
    check(lib().lle_gen_cells_to_text(arr.ctypes.data_as(C.c_void_p), height, width, None, 0, C.byref(n)))
    buf = C.create_string_buffer(n.value + 1)
    check(lib().lle_gen_cells_to_text(arr.ctypes.data_as(C.c_void_p), height, width, buf, n.value + 1, None))
    return buf.value.decode()


def is_geometry_valid(cells: np.ndarray | torch.Tensor, height: int, width: int) -> bool:
    """CandidateLayout.is_geometry_valid (candidates.py:27-41) of a cell grid, via lle_gen_geometry_valid."""
    arr = np.ascontiguousarray(cells.cpu().numpy() if isinstance(cells, torch.Tensor) else cells, dtype=np.uint8).reshape(-1)
    ok = C.c_int32(0)
    check(lib().lle_gen_geometry_valid(arr.ctypes.data_as(C.c_void_p), height, width, C.byref(ok)))
    return bool(ok.value)


def attempt_seeds(seed: int, n: int) -> np.ndarray:
    """generator.py:296-301: the seeds `_generate_n_multi` hands to its workers."""
    out = np.empty(n, dtype=np.uint64)
    check(lib().lle_gen_attempt_seeds(C.c_uint64(seed), n, out.ctypes.data_as(C.c_void_p)))
    return out


class WorldGenerator:
    """lle.generator.WorldGenerator (generator.py:60-186) with device batches."""

    def __init__(self, *, width: int, height: int, n_agents: int = 2, starts: str = "random", exits: str = "random", n_lasers: int = 0,
                 n_gems: int = 0, laser_placement: str = "free", laser_span: int | str = "any", n_walls: int | str = "auto",
                 walls_style: str = "individual", n_rooms_rows: int = 0, n_rooms_cols: int = 0, door_size: int = 1,
                 require: int = 0, cluster_shape: tuple[int, int] | None = None, device: int = 0, batch: int = 65536):
        for name, value, table in (("starts", starts, _STARTS), ("exits", exits, _EXITS), ("laser_placement", laser_placement, _PLACEMENT)):
            if value not in table:
                raise ValueError(f"Unknown {name} mode: {value!r}")
        o = _native.GenOptions()
        lib().lle_gen_default_options(C.byref(o))
        o.width, o.height, o.n_agents = width, height, n_agents
        o.starts, o.exits, o.laser_placement = _STARTS[starts], _EXITS[exits], _PLACEMENT[laser_placement]
        o.n_lasers, o.n_gems = n_lasers, n_gems
        o.laser_span = {"any": 0, "across": -1}[laser_span] if isinstance(laser_span, str) else int(laser_span)
        if not isinstance(laser_span, str) and laser_span < 2:
            raise ValueError(f"laser_span must be >= 2, got {laser_span}.")
        o.n_walls = -1 if n_walls == "auto" else int(n_walls)
        o.walls_shapes = {"individual": 0, "shapes": 1}[walls_style]
        o.n_rooms_rows, o.n_rooms_cols, o.door_size = n_rooms_rows, n_rooms_cols, door_size
        o.cluster_h, o.cluster_w = cluster_shape if cluster_shape is not None else _default_cluster_shape(n_agents)
        self.width, self.height, self.n_agents = width, height, n_agents
        self.require = int(require)
        self.device = torch.device("cuda", device)
        self.batch = int(batch)
        self._h = C.c_void_p()
        check(lib().lle_gen_create(C.byref(o), device, self.batch, C.byref(self._h)))
        b = _native.GenBuffers()
        check(lib().lle_gen_get_buffers(self._h, C.byref(b)))
        from .vec_world import _DevArray

        def wrap(ptr, shape, typestr):
            return torch.as_tensor(_DevArray(ptr, shape, typestr, self), device=self.device)

        self.cells = wrap(b.cells, (self.batch, height, width), "|u1")
        self.status = wrap(b.status, (self.batch,), "|u1")
        self.labels = wrap(b.labels, (self.batch,), "|u1")
        self.tries = wrap(b.tries, (self.batch,), "<i4")
        self._rng = _random.Random()

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().lle_gen_destroy(h)

    # -- device runs ---------------------------------------------------------------------------------------------------
    def run(self, seeds: Sequence[int] | np.ndarray | torch.Tensor | None = None, *, first_seed: int = 0, n: int | None = None,
            max_attempts: int = 1, require: int | None = None):
        """One chain per seed (include/lle_b200.h, lle_gen_run).  Returns views (cells u8[n,H,W], status, labels, tries)
        of the generator's device buffers, valid until the next run."""
        stream = torch.cuda.current_stream(self.device).cuda_stream
        ptr = None
        if seeds is not None:
            if not isinstance(seeds, torch.Tensor):
                # uint64 seeds travel as their int64 bit pattern
                seeds = torch.from_numpy(np.asarray(seeds, dtype=np.uint64).view(np.int64)).to(self.device)
            n = seeds.numel()
            ptr = C.c_void_p(seeds.data_ptr())
        assert n is not None and n <= self.batch, "n must be given and fit the generator's batch"
        check(lib().lle_gen_run(self._h, ptr, C.c_uint64(first_seed), n, max_attempts, self.require if require is None else require,
                                C.c_void_p(stream)))
        return self.cells[:n], self.status[:n], self.labels[:n], self.tries[:n]

    def try_generate(self, seed: int) -> str | None:
        """generator.py:243-254 `_try_generate(seed)`: the map text or None."""
        cells, status, _, _ = self.run([seed])
        return cells_to_text(cells[0], self.height, self.width) if int(status[0]) else None

    def generate(self, max_attempts: int | None, seed: int | None = None) -> str | None:
        """generator.py:268-284: attempts drawn from one stream until a layout is accepted."""
        if seed is None:
            seed = self._rng.randrange(sys.maxsize)
        # the reference searches without bound when max_attempts is None; a chain is one device thread (about 0.4 ms per
        # attempt at full occupancy, less alone), so an unbounded search stops after 20,000 attempts and returns None
        cells, status, _, _ = self.run([seed], max_attempts=20_000 if max_attempts is None else max_attempts)
        return cells_to_text(cells[0], self.height, self.width) if int(status[0]) else None

    def generate_n(self, n: int, seed: int | None = None, max_attempts: int | None = None, distinct: bool = False) -> Iterator[str]:
        """generator.py:296-341 (`generate_n` with n_jobs > 1): yields up to n accepted map texts in attempt order."""
        if seed is None:
            seed = self._rng.randrange(sys.maxsize)
        budget = sys.maxsize if max_attempts is None else max_attempts
        found, done, seen = 0, 0, set()
        # generator.py:296-301: the host draws one seed per attempt from its own generator, exactly as the reference does
        # (`self._rng.seed(seed)`, then `randrange(sys.maxsize)` per attempt); lle_gen_attempt_seeds is the same list for
        # hosts without a CPython
        self._rng.seed(seed)
        while found < n and done < budget:
            take = int(min(self.batch, budget - done))
            seeds = np.fromiter((self._rng.randrange(sys.maxsize) for _ in range(take)), dtype=np.uint64, count=take)
            cells, status, labels, _ = self.run(seeds)
            ok = torch.nonzero(status).flatten().cpu().numpy()
            grids = cells.cpu().numpy()
            for i in ok:
                text = cells_to_text(grids[i], self.height, self.width)
                if distinct and text in seen:
                    continue
                seen.add(text)
                found += 1
                yield text
                if found >= n:
                    return
            done += take


class GeneratorBuilder:
    """lle.generate(...) (builder.py:59-437): the fluent description of a generation request.  The behavioural methods of
    the reference (`solvable()`, `cooperative()`, `sequential()` ...) need its SAT characterizer and raise here: they are
    the reference's SAT semantics, whose encoding forbids agents following each other and swapping places
    (world_filter.py), which this engine allows.  `walkable()`, `independent_paths()` and `needs_blocker()` select this
    library's reachability labels instead, and `plannable(max_steps)` keeps the layouts the device planner can finish."""

    def __init__(self, *, width: int = 10, height: int = 10, n_agents: int = 3):
        self._kw = dict(width=width, height=height, n_agents=n_agents, starts="random", exits="random", n_gems=0, laser_placement="free",
                        laser_span="any", n_walls="auto", walls_style="individual", n_rooms_rows=0, n_rooms_cols=0, door_size=1)
        self._n_lasers: int | Literal["auto"] = "auto"
        self._require = 0
        self._cluster_shape = None
        self._plan: tuple[int, bool] | None = None

    def random(self):
        return self.starts("random").exits("random")

    def lanes(self):
        return self.starts("edge").exits("opposite")

    def clustered(self, shape: tuple[int, int] | None = None):
        self._cluster_shape = shape
        return self.starts("clustered").exits("opposite")

    def starts(self, mode: str):
        self._kw["starts"] = mode
        return self

    def exits(self, mode: str):
        self._kw["exits"] = mode
        return self

    def gems(self, n: int):
        self._kw["n_gems"] = n
        return self

    def lasers(self, n: int | Literal["auto"] = "auto", *, placement: str = "auto", span: int | str = "any"):
        self._n_lasers = n
        self._kw["laser_placement"] = "free" if placement == "auto" else placement  # builder.py:411-420
        self._kw["laser_span"] = span
        return self

    def walls(self, n: int | Literal["auto"] = "auto", *, style: str = "individual"):
        self._kw["n_walls"], self._kw["walls_style"] = n, style
        return self

    def rooms(self, n: int = 4, *, door_size: int = 1):
        """builder.py:196-242"""
        if n < 2:
            raise ValueError(f"rooms requires n >= 2, got {n}")
        if door_size < 1:
            raise ValueError(f"door_size must be >= 1, got {door_size}")
        rows = int(math.isqrt(n))
        while rows >= 1 and n % rows:
            rows -= 1
        cols = n // rows
        if self._kw["height"] < 2 * rows - 1:
            raise ValueError(f"{n} rooms ({rows}×{cols} layout) requires height >= {2 * rows - 1}, got {self._kw['height']}")
        if self._kw["width"] < 2 * cols - 1:
            raise ValueError(f"{n} rooms ({rows}×{cols} layout) requires width >= {2 * cols - 1}, got {self._kw['width']}")
        self._kw.update(n_rooms_rows=rows, n_rooms_cols=cols, door_size=door_size)
        return self

    def walkable(self):
        self._require = WALKABLE
        return self

    def independent_paths(self):
        self._require = WALKABLE | INDEPENDENT
        return self

    def needs_blocker(self):
        self._require = WALKABLE | NEEDS_BLOCKER
        return self

    def plannable(self, max_steps: int, *, all_gems: bool = False):
        """Keep only the layouts for which the device planner (lle_b200.planner.plan) finds a plan of at most `max_steps`
        joint steps in which nobody dies and every agent reaches an exit (and, with `all_gems`, every gem is collected).
        Applied after the other filters; `take` keeps the attempt order, and `build` returns the first such layout of the
        same attempt-ordered stream.  Layouts the map compiler refuses are dropped; a layout beyond the planner's limits
        (include/lle_b200.h: lle_plan) raises."""
        if not 1 <= int(max_steps) <= 1024:
            raise ValueError(f"max_steps must be in [1, 1024], got {max_steps}")
        self._plan = (int(max_steps), bool(all_gems))
        return self

    def _plannable(self, texts: Iterator[str], n: int, device: int) -> Iterator[str]:
        """The texts of `texts` that have a plan, in order, planned in batches of up to 1,024 maps, until n are found."""
        from .planner import plan
        from .types import ParsingError
        from .vec_world import Map

        max_steps, all_gems = self._plan
        found, batch = 0, []
        if n <= 0:
            return

        def flush():
            length = plan(batch, max_steps=max_steps, all_gems=all_gems, device=device).length
            return [m.text for m, k in zip(batch, length) if k >= 0]

        for text in texts:
            try:
                batch.append(Map(text))
            except ParsingError:
                continue
            if len(batch) < min(1024, 2 * (n - found)):
                continue
            for kept in flush():
                yield kept
                found += 1
                if found == n:
                    return
            batch = []
        for kept in flush()[: n - found] if batch else []:
            yield kept

    def _sat_only(self, *_a, **_k):
        raise NotImplementedError("this predicate needs the reference's SAT characterizer (world_filter.py), which is out of scope; "
                                  "use walkable() / independent_paths() / needs_blocker() (reachability labels) or plannable(max_steps) (device planner)")

    solvable = independent = cooperative = sequential = mutual = interdependent = convergent = divergent = asymmetric = require = _sat_only

    def _make_generator(self, device: int = 0, batch: int = 65536) -> WorldGenerator:
        n_lasers = self._n_lasers if self._n_lasers != "auto" else _random.randint(0, self._kw["n_agents"])  # builder.py:422-430
        return WorldGenerator(**self._kw, n_lasers=n_lasers, require=self._require, cluster_shape=self._cluster_shape, device=device, batch=batch)

    def build(self, *, seed: int | None = None, max_attempts: int | None = None, device: int = 0):
        """One `World` (builder.py:321-344, the n_jobs=1 path: one stream across the attempts; with `plannable`, the first
        plannable layout of `take`'s attempt-ordered stream)."""
        from .world import World

        if self._plan is not None:
            text = next(iter(self.take(1, seed=seed, max_attempts=max_attempts, device=device, texts=True)), None)
        else:
            text = self._make_generator(device, batch=1).generate(max_attempts, seed)
        return None if text is None else World(text)

    def take(self, n: int, *, seed: int | None = None, max_attempts: int | None = None, device: int = 0, distinct: bool = False,
             texts: bool = False) -> Iterator:
        """Up to n worlds (builder.py:346-371 with parallel workers).  Yields `World` objects like the reference; with
        `texts=True` the v1 map texts instead, which is what a batch wants (`VecWorld(list_of_texts, ...)`)."""
        from .world import World

        stream = self._make_generator(device).generate_n(n if self._plan is None else sys.maxsize, seed=seed, max_attempts=max_attempts,
                                                         distinct=distinct)
        if self._plan is not None:
            stream = self._plannable(stream, n, device)
        for text in stream:
            yield text if texts else World(text, device)


def generate(width: int = 10, height: int = 10, n_agents: int = 3) -> GeneratorBuilder:
    """lle.generate (python/lle/generator/__init__.py:67-93)."""
    return GeneratorBuilder(width=width, height=height, n_agents=n_agents)
