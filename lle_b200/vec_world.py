"""`VecWorld`: N independent worlds resident on one B200, stepped by one fused kernel launch.

Host-side mirror of the reference's `World` for a batch (src/bindings/world/pyworld.rs:144-626): the
same operations (`reset`, `step`, `available_actions`, `get_state`, `set_state`), but every result is a
zero-copy torch view of a device buffer owned by the C-ABI object (include/lle_b200.h).
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np
import torch

from . import _native
from ._native import MapInfo, RawState, VecBuffers, VecOptions, check, lib
from .types import OBS_STATE, Direction, InvalidLevelError, LaserSource, obs_spec


class Map:
    """A compiled map (lle_map).  Replaces `World::try_from(&str)` up to, but excluding, the dynamic state."""

    def __init__(self, text: str | None = None, *, level: int | None = None):
        h = C.c_void_p()
        if level is not None:
            if not isinstance(level, int) or not 1 <= level <= 6:
                raise InvalidLevelError(f"InvalidLevel {{ asked: {level}, min: 1, max: 6 }}")
            check(lib().lle_map_level(level, C.byref(h)))
        else:
            raw = text.encode()
            check(lib().lle_map_parse(raw, len(raw), C.byref(h)))
        self._h = h
        info = MapInfo()
        check(lib().lle_map_get_info(self._h, C.byref(info)))
        self.info = info
        self.height, self.width = info.height, info.width
        self.n_agents, self.n_gems, self.n_sources, self.n_channels = info.n_agents, info.n_gems, info.n_sources, info.n_channels
        self.obs_invalid = bool(info.obs_invalid)
        self.gem_toplevel = int(info.gem_toplevel)
        self.text = lib().lle_map_text(self._h).decode()

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            lib().lle_map_free(h)
            self._h = None

    def positions(self, kind: int) -> list[tuple[int, int]]:
        n = C.c_int32(0)
        check(lib().lle_map_positions(self._h, kind, None, 0, C.byref(n)))
        buf = (C.c_int32 * max(1, 2 * n.value))()
        check(lib().lle_map_positions(self._h, kind, buf, n.value, C.byref(n)))
        return [(buf[2 * k], buf[2 * k + 1]) for k in range(n.value)]

    walls = property(lambda self: self.positions(0))
    voids = property(lambda self: self.positions(1))
    exits = property(lambda self: self.positions(2))
    gems = property(lambda self: self.positions(3))
    starts = property(lambda self: self.positions(4))
    laser_cells = property(lambda self: self.positions(5))

    @property
    def random_starts(self) -> list[list[tuple[int, int]]]:
        """World.random_start_pos (world.rs:297-303): the start candidates of every agent."""
        out = []
        for a in range(self.n_agents):
            n = C.c_int32(0)
            check(lib().lle_map_start_candidates(self._h, a, None, 0, C.byref(n)))
            buf = (C.c_int32 * max(1, 2 * n.value))()
            check(lib().lle_map_start_candidates(self._h, a, buf, n.value, C.byref(n)))
            out.append([(buf[2 * k], buf[2 * k + 1]) for k in range(n.value)])
        return out

    def sources(self) -> list[LaserSource]:
        n = C.c_int32(0)
        check(lib().lle_map_sources(self._h, None, 0, C.byref(n)))
        buf = (C.c_int32 * max(1, 7 * n.value))()
        check(lib().lle_map_sources(self._h, buf, n.value, C.byref(n)))
        return [LaserSource((buf[7 * k], buf[7 * k + 1]), buf[7 * k + 2], Direction(buf[7 * k + 3]), bool(buf[7 * k + 4]),
                            buf[7 * k + 5], buf[7 * k + 6]) for k in range(n.value)]

    def laser_tiles(self) -> list[tuple[tuple[int, int], int, int, Direction, int, int]]:
        """(pos, laser_id, agent_id, direction, beam, offset) of every tile listed by World::lasers()."""
        n = C.c_int32(0)
        check(lib().lle_map_lasers(self._h, None, 0, C.byref(n)))
        buf = (C.c_int32 * max(1, 7 * n.value))()
        check(lib().lle_map_lasers(self._h, buf, n.value, C.byref(n)))
        return [((buf[7 * k], buf[7 * k + 1]), buf[7 * k + 2], buf[7 * k + 3], Direction(buf[7 * k + 4]), buf[7 * k + 5],
                 buf[7 * k + 6]) for k in range(n.value)]


def _obs_dtype(dtype) -> torch.dtype:
    """torch.float32 / torch.int8, or their names."""
    named = {"float32": torch.float32, "int8": torch.int8}
    dt = named.get(dtype, dtype) if isinstance(dtype, str) else dtype
    if dt not in (torch.float32, torch.int8):
        raise ValueError(f"obs_dtype must be torch.float32 or torch.int8 (or 'float32' / 'int8'), got {dtype!r}")
    return dt


class _DevArray:
    """Exposes a raw device pointer through __cuda_array_interface__ so torch can wrap it without a copy."""

    def __init__(self, ptr: int, shape: tuple[int, ...], typestr: str, owner):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (int(ptr), False), "version": 2}
        self._owner = owner


def _stream_ptr(device: torch.device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


class VecWorld:
    """N worlds on one CUDA device.

    Parameters mirror `lle_vec_options`.  `maps` is a list of `Map` / map strings / level numbers; all maps
    must share (height, width, n_agents, n_gems).  `map_of_env[e]` selects the map of env e.
    """

    def __init__(self, maps: Sequence[Map | str | int] | Map | str | int, n_envs: int, *, map_of_env: Sequence[int] | None = None,
                 device: int | str | torch.device = 0, reward_dim: int = 1, walkable_lasers: bool = True, auto_reset: bool = True,
                 lle_semantics: bool = True, write_obs: bool = True, seed: int = 0, env_id_base: int = 0,
                 extras: str | Sequence[int] | None = None, pbrs: dict | None = None, obs_type: str = "layered",
                 padding_size: int = 0, randomize_lasers: bool = False, state_type: str = "state", episode_stats: bool = False,
                 obs_dtype: torch.dtype | str = torch.float32):
        """obs_type: an ObservationType value (observations.py:37-60) other than "rgb-image"; padding_size for "layered-padded".
        obs_dtype: torch.float32 (default) or torch.int8 (also "float32" / "int8"): the element type of `obs`.  Every value of a
        layered, padded, flattened or perspective observation is -1, 0 or 1, so int8 holds the same observation in a quarter of the
        HBM bytes (`obs.to(torch.bfloat16)` and `obs.float()` are exact).  Partial and state observations are float32 only.
        state_type: the ObservationType whose first-agent observation is the state (Builder.state_type, builder.py:51-58).
        extras: None | "laser_subgoal" (all sources) | source indices (World::sources() order) — Builder.add_extras.
        pbrs: None | dict(gamma=0.99, reward_value=0.5, lasers_to_reward=None | indices, with_extras=True) — Builder.pbrs
        (python/lle/env/builder.py:77-150)."""
        if not torch.cuda.is_available():
            raise RuntimeError("lle_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        if isinstance(maps, (Map, str, int)):
            maps = [maps]
        self.maps = [m if isinstance(m, Map) else (Map(level=m) if isinstance(m, int) else Map(m)) for m in maps]
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        opts = VecOptions()
        lib().lle_vec_default_options(C.byref(opts))
        opts.device = self.device.index or 0
        opts.reward_dim, opts.walkable_lasers, opts.auto_reset = int(reward_dim), int(walkable_lasers), int(auto_reset)
        opts.lle_semantics, opts.write_obs = int(lle_semantics), int(write_obs)
        opts.seed, opts.env_id_base = int(seed), int(env_id_base)
        self.obs_type = obs_type
        opts.obs_type, opts.obs_param, self._flatten = obs_spec(obs_type, padding_size)
        opts.randomize_lasers = int(bool(randomize_lasers))
        opts.episode_stats = int(bool(episode_stats))
        self.obs_dtype = _obs_dtype(obs_dtype)
        opts.obs_dtype = _native.DTYPE_I8 if self.obs_dtype == torch.int8 else _native.DTYPE_F32
        self.state_type = getattr(state_type, "value", state_type)
        opts.state_type, opts.state_param, self._state_flatten = obs_spec(state_type, 0)  # the reference builds it with padding_size = 0 (env.py:86)
        extras_src = None if extras in (None, "laser_subgoal") else [int(x) for x in extras]
        want_extras = extras is not None
        if pbrs is not None:
            opts.pbrs = 1
            opts.pbrs_gamma = float(pbrs.get("gamma", 0.99))
            opts.pbrs_reward_value = float(pbrs.get("reward_value", 0.5))
            rewarded = pbrs.get("lasers_to_reward")
            opts.n_pbrs = -1 if rewarded is None else len(rewarded)
            for k, b in enumerate(rewarded or []):
                opts.pbrs_src[k] = int(b)
            if pbrs.get("with_extras", True) and not want_extras:
                want_extras, extras_src = True, (None if rewarded is None else [int(x) for x in rewarded])
        if want_extras:
            opts.n_extras = -1 if extras_src is None else len(extras_src)
            for k, b in enumerate(extras_src or []):
                opts.extras_src[k] = int(b)
        handles = (C.c_void_p * len(self.maps))(*[m._h for m in self.maps])
        moe = None
        if map_of_env is not None:
            arr = np.ascontiguousarray(map_of_env, dtype=np.int32)
            if arr.shape != (n_envs,):
                raise ValueError("map_of_env must have n_envs entries")
            moe = arr.ctypes.data_as(C.POINTER(C.c_int32))
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.cuda.current_stream().synchronize()  # make sure torch's primary context exists
            h = C.c_void_p()
            check(lib().lle_vec_create(handles, len(self.maps), moe, int(n_envs), C.byref(opts), C.byref(h)))
        self._h = h
        b = VecBuffers()
        check(lib().lle_vec_get_buffers(self._h, C.byref(b)))
        self.n_envs, self.n_agents, self.n_gems, self.n_channels = int(b.n_envs), b.n_agents, b.n_gems, b.n_channels
        self.height, self.width, self.reward_dim, self.state_dim, self.n_beams_max = b.height, b.width, b.reward_dim, b.state_dim, b.n_beams_max
        self.obs_stride = int(b.obs_stride)
        self.record_bytes = int(b.record_bytes)
        N, A = self.n_envs, self.n_agents
        dev = self.device

        def wrap(ptr, shape, typestr):
            return torch.as_tensor(_DevArray(ptr, shape, typestr, self), device=dev)

        #: one block per env, shaped by the observation type (include/lle_b200.h: lle_vec_buffers.obs):
        #: layered (C,H,W) [flattened: (C*H*W,)] / partial (A,2A+3,s,s) / perspective (A,C,H,W) / state (3A+G,)
        self.obs = None
        self.obs_kind, self.obs_view_agents = int(b.obs_type), int(b.obs_view_agents)
        #: a laser colour selects a channel past the last layer of this observation type (the reference raises IndexError)
        self.obs_invalid = bool(b.obs_invalid)
        self.obs_shape = (b.obs_c,) if self.obs_kind == OBS_STATE else (b.obs_c, b.obs_h, b.obs_w)  # one agent's observation
        if write_obs:
            rows = wrap(b.obs_i8, (N, self.obs_stride), "|i1") if int(b.obs_dtype) == _native.DTYPE_I8 else wrap(b.obs, (N, self.obs_stride), "<f4")
            block = self.obs_shape if self.obs_view_agents else (A, *self.obs_shape)
            n = int(np.prod(block))
            self.obs = rows[:, :n].unflatten(1, block)
            if self._flatten:
                self.obs = self.obs.flatten(1)
        self.state = wrap(b.state, (N, self.state_dim), "<f4")
        self.avail = wrap(b.avail, (N, A, 5), "|u1")
        self.reward = wrap(b.reward, (N, self.reward_dim), "<f4")
        self.done = wrap(b.done, (N,), "|u1")
        self.events = wrap(b.events, (N, A), "|u1")
        self.actions = wrap(b.actions, (N, A), "|i1")
        self.err = wrap(b.err, (N,), "|u1")
        #: with randomize_lasers: (N,) i32, map * n_variants + colouring (colour of source b = digit b in base n_agents)
        self.n_variants = int(b.n_variants)
        self.map_index = wrap(b.map_index, (N,), "<i4") if b.map_index else None
        #: LLE(state_type=...): the state observation, one block per env shaped like `obs` of that type; `state_of_type` is what
        #: the reference's get_state() returns per env (the first agent's observation, observations.py:118-119)
        self.state_obs = None
        if b.state_obs:
            shape = (b.state_c,) if int(b.state_type) == OBS_STATE else (b.state_c, b.state_h, b.state_w)
            rows = wrap(b.state_obs, (N, int(b.state_obs_stride)), "<f4")
            block = shape if b.state_view_agents or int(b.state_type) == OBS_STATE else (A, *shape)
            self.state_obs = rows[:, : int(np.prod(block))].unflatten(1, block)
            self._state_first = bool(not b.state_view_agents and int(b.state_type) != OBS_STATE)
        #: episode_stats: Step.info of every env (env.py:174-188) and episode return / length accumulators kept by the step kernel
        self.info_bytes = wrap(b.info, (N, 2 + A), "|u1") if b.info else None
        self.ep_return = wrap(b.ep_return, (N, self.reward_dim), "<f4") if b.ep_return else None
        self.ep_length = wrap(b.ep_length, (N,), "<i4") if b.ep_length else None
        self.last_return = wrap(b.last_return, (N, self.reward_dim), "<f4") if b.last_return else None
        self.last_length = wrap(b.last_length, (N,), "<i4") if b.last_length else None
        #: LaserSubgoal flags (N, A, n_sources); None when extras are off
        self.extras_dim = int(b.extras_dim)
        self.extras = wrap(b.extras, (N, A, self.extras_dim), "<f4") if self.extras_dim else None

    def destroy(self):
        """Release the device memory now (lle_vec_destroy; an open parts loop is aborted first).  The tensors handed out become
        dangling: only for callers that manage lifetimes explicitly — dropping the last reference does the same."""
        h = getattr(self, "_h", None)
        if h:
            self._h = None
            lib().lle_vec_destroy(h)

    def __del__(self):
        self.destroy()

    # ---- views
    @property
    def obs_per_agent(self) -> torch.Tensor:
        """(N, n_agents[+padding], *shape): what the reference's generator returns per env.  Where the reference tiles
        one block over the agents (np.tile: layered, flattened, state) the agent dimension is a stride-0 view."""
        if not self.obs_view_agents:
            return self.obs
        return self.obs.unsqueeze(1).expand(-1, self.obs_view_agents, *([-1] * (self.obs.dim() - 1)))

    @property
    def info(self) -> dict:
        """Step.info of LLE.step (env.py:174-188) for every env, as device tensors (needs episode_stats=True)."""
        if self.info_bytes is None:
            raise ValueError("create the batch with episode_stats=True")
        A, G = self.n_agents, self.n_gems
        out = {"gems_collected": self.info_bytes[:, 0], "exit_rate": self.info_bytes[:, 1].float() / A}
        for i in range(A):
            out[f"has-arrived-{i}"] = self.info_bytes[:, 2 + i].bool()
            out[f"is-alive-{i}"] = self.state[:, 2 * A + G + i] != 0
        return out

    @property
    def state_of_type(self) -> torch.Tensor:
        """(N, *state_shape): LLE.get_state() of every env for the configured state_type (env.py:205-206)."""
        if self.state_obs is None:
            return self.state
        st = self.state_obs[:, 0] if self._state_first else self.state_obs
        return st.flatten(1) if self._state_flatten else st

    @property
    def obs_flattened(self) -> torch.Tensor:
        """FlattenedLayered (observations.py:291-293)."""
        return self.obs.flatten(1)

    # ---- operations
    def reset(self, mask: torch.Tensor | None = None):
        ptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            ptr = mask.data_ptr()
        check(lib().lle_vec_reset(self._h, ptr, _stream_ptr(self.device)))

    def step(self, actions: torch.Tensor | None = None):
        """One lockstep step.  `actions`: int8 (N, A) device tensor, or None for on-device Philox sampling."""
        ptr = None
        if actions is not None:
            if actions.shape != (self.n_envs, self.n_agents):
                raise ValueError(f"InvalidNumberOfActions: expected shape {(self.n_envs, self.n_agents)}, got {tuple(actions.shape)}")
            actions = actions.to(device=self.device, dtype=torch.int8).contiguous()
            ptr = actions.data_ptr()
        check(lib().lle_vec_step(self._h, ptr, _stream_ptr(self.device)))

    def rollout(self, n_steps: int):
        """`n_steps` device-sampled lockstep steps in one launch (bit-identical to n_steps calls of step(None))."""
        check(lib().lle_vec_rollout(self._h, int(n_steps), _stream_ptr(self.device)))

    def step_host(self, actions: np.ndarray | torch.Tensor | None, reward_out: torch.Tensor, done_out: torch.Tensor):
        """Host-facing step: H2D actions, step, D2H reward/done, stream sync (lle_vec_step_host)."""
        ptr = None
        if actions is not None:
            t = actions if isinstance(actions, torch.Tensor) else torch.from_numpy(actions)
            assert t.dtype == torch.int8 and t.is_contiguous() and not t.is_cuda
            ptr = t.data_ptr()
        check(lib().lle_vec_step_host(self._h, ptr, reward_out.data_ptr(), done_out.data_ptr(), _stream_ptr(self.device)))

    def set_source(self, source_index: int, *, agent_id: int | None = None, enabled: bool | None = None, map_index: int = 0):
        """Recolour / switch one laser source in every env that uses map `map_index` (lle_vec_set_source;
        LaserBeam::set_agent_id / enable / disable, src/core/tiles/laser.rs:69-84)."""
        check(lib().lle_vec_set_source(self._h, int(map_index), int(source_index), -1 if agent_id is None else int(agent_id),
                                       -1 if enabled is None else int(bool(enabled)), _stream_ptr(self.device)))
        b = VecBuffers()
        check(lib().lle_vec_get_buffers(self._h, C.byref(b)))
        self.obs_invalid = bool(b.obs_invalid)

    def collect_gem(self, gem_index: int, map_index: int = 0):
        """PyGem.collect for gem `gem_index` in every env of a map (lle_vec_collect_gem); call refresh() afterwards."""
        check(lib().lle_vec_collect_gem(self._h, map_index, gem_index, _stream_ptr(self.device)))

    def set_exits(self, exits: Sequence[tuple[int, int]], map_index: int = 0):
        """World::set_exit_positions (world.rs:195-234) in every env that uses map `map_index` (lle_vec_set_exits)."""
        flat = (C.c_int32 * max(1, 2 * len(exits)))(*[int(x) for p in exits for x in p])
        check(lib().lle_vec_set_exits(self._h, int(map_index), flat, len(exits), _stream_ptr(self.device)))

    def source_colours(self) -> torch.Tensor:
        """(N, n_sources) current colour of every source of every env (they differ per env with randomize_lasers)."""
        nb = self.n_beams_max
        if self.n_variants == 1:
            per_map = torch.tensor([[c for c, _ in self.source_states(k)] + [0] * (nb - len(self.source_states(k)))
                                    for k in range(len(self.maps))], dtype=torch.int32, device=self.device).reshape(len(self.maps), nb)
            idx = self.map_index.long() if self.map_index is not None else torch.zeros(self.n_envs, dtype=torch.long, device=self.device)
            return per_map[idx]
        variant = self.map_index.long() % self.n_variants
        digits = [(variant // (self.n_agents ** k)) % self.n_agents for k in range(nb)]
        return torch.stack(digits, dim=1).to(torch.int32) if nb else torch.zeros((self.n_envs, 0), dtype=torch.int32, device=self.device)

    def source_states(self, map_index: int = 0) -> list[tuple[int, bool]]:
        """Current (agent_id, is_enabled) of the sources of map `map_index` (lle_vec_get_sources)."""
        n = C.c_int32(0)
        check(lib().lle_vec_get_sources(self._h, int(map_index), None, 0, C.byref(n)))
        buf = (C.c_int32 * max(1, 2 * n.value))()
        check(lib().lle_vec_get_sources(self._h, int(map_index), buf, n.value, C.byref(n)))
        return [(int(buf[2 * k]), bool(buf[2 * k + 1])) for k in range(n.value)]

    def seed(self, seed: int):
        """World::seed (world.rs:92-96): Philox key of the action sampler and of the start sampler."""
        check(lib().lle_vec_set_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF))

    def refresh(self):
        """Re-export observation / state / availability of every env from its current engine state, resetting none
        (lle_vec_refresh)."""
        check(lib().lle_vec_refresh(self._h, _stream_ptr(self.device)))

    def submit_host(self, actions: np.ndarray | torch.Tensor | None, reward_out: torch.Tensor, done_out: torch.Tensor,
                    after_current_stream: bool = True):
        """Pipelined host-facing step (lle_vec_pipeline_submit): H2D copy of the actions, the step (which writes reward / done
        straight into the pinned host buffers) on the vec's own streams; returns at once.  Buffers must be pinned and stay alive
        until the matching `wait_host()`.  after_current_stream=False: nothing the step depends on is pending on torch's stream
        (LLE_STREAM_NONE: a closed host loop that only talks to the env through these two calls)."""
        ptr = None
        if actions is not None:
            t = actions if isinstance(actions, torch.Tensor) else torch.from_numpy(actions)
            assert t.dtype == torch.int8 and t.is_contiguous() and not t.is_cuda
            ptr = t.data_ptr()
        check(lib().lle_vec_pipeline_submit(self._h, ptr, reward_out.data_ptr() if reward_out is not None else None,
                                            done_out.data_ptr() if done_out is not None else None,
                                            _stream_ptr(self.device) if after_current_stream else C.c_void_p(-1)))

    def wait_host(self) -> int:
        """Block until the oldest submitted step's reward / done are in their host buffers; returns the number of steps
        still outstanding (lle_vec_pipeline_wait)."""
        left = C.c_int32(0)
        check(lib().lle_vec_pipeline_wait(self._h, C.byref(left)))
        return left.value

    def parts_loop(self, n_parts: int, actions: torch.Tensor, reward_out: torch.Tensor | None, done_out: torch.Tensor | None,
                   after_current_stream: bool = True) -> "PartsLoop":
        """Open a closed loop over `n_parts` parts of this batch (lle_vec_parts_*, include/lle_b200.h): every step is one launch
        over the whole batch, and the step kernel waits part by part for the actions the host releases.  `actions` (int8 [N, A]),
        `reward_out` (float32 [N, reward_dim]) and `done_out` (uint8 [N]) are pinned host tensors the kernel reads / writes in
        place.  Use as a context manager."""
        return PartsLoop(self, n_parts, actions, reward_out, done_out, after_current_stream)

    def set_state(self, positions: torch.Tensor, gems_collected: torch.Tensor, agents_alive: torch.Tensor):
        pos = positions.to(device=self.device, dtype=torch.int32).contiguous()
        gems = gems_collected.to(device=self.device, dtype=torch.uint8).contiguous()
        alive = agents_alive.to(device=self.device, dtype=torch.uint8).contiguous()
        if pos.shape != (self.n_envs, self.n_agents, 2) or alive.shape != (self.n_envs, self.n_agents):
            raise ValueError("InvalidNumberOfAgents")
        if gems.shape != (self.n_envs, self.n_gems):
            raise ValueError("InvalidNumberOfGems")
        check(lib().lle_vec_set_state(self._h, pos.data_ptr(), gems.data_ptr() if self.n_gems else None, alive.data_ptr(),
                                      _stream_ptr(self.device)))

    # ---- the device expert (include/lle_b200.h: lle_vec_expert_*)
    def build_expert(self, all_gems: bool = False) -> np.ndarray:
        """Builds, on the device, the exact distance-to-goal table of every map as the batch holds it now: over every joint state
        reachable from reset without a death, the length of a shortest death-free way to a goal (every agent on an exit, and with
        `all_gems` every gem collected) and the smallest joint action that starts one.  Returns the size of each map's reached set
        (int64 [n_maps]).  Limits: those of `lle_b200.planner.plan`; the batch needs walkable_lasers and no randomize_lasers.
        `set_source` / `set_exits` drop the tables: build again after them."""
        n_states = np.zeros(len(self.maps), np.int64)
        check(lib().lle_vec_expert_build(self._h, 1 if all_gems else 0, n_states.ctypes.data_as(C.c_void_p), _stream_ptr(self.device)))
        return n_states

    def expert_actions(self, actions_out: torch.Tensor | None = None, dist_out: torch.Tensor | None = None):
        """(actions int8 [N, A], dist int32 [N]) of every env from its current state, on the batch's device and torch's current
        stream: the optimal joint action (all Stay where dist <= 0), directly usable as `step`'s actions, and the distance to a goal
        (-1: no death-free way there; -2: not in the table, an agent is dead or the state is not reachable from reset)."""
        N, A = self.n_envs, self.n_agents
        if actions_out is None:
            actions_out = torch.empty((N, A), dtype=torch.int8, device=self.device)
        if dist_out is None:
            dist_out = torch.empty((N,), dtype=torch.int32, device=self.device)
        for t, dt, shape in ((actions_out, torch.int8, (N, A)), (dist_out, torch.int32, (N,))):
            if t.dtype != dt or tuple(t.shape) != shape or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"expert_actions: expected a contiguous {dt} {shape} tensor on {self.device}")
        check(lib().lle_vec_expert_act(self._h, actions_out.data_ptr(), dist_out.data_ptr(), _stream_ptr(self.device)))
        return actions_out, dist_out

    def expert_table(self, map_index: int = 0) -> tuple[np.ndarray, np.ndarray]:
        """Host copy of map `map_index`'s table, indexed by state key (include/lle_b200.h: lle_vec_expert_build): dist int32 [K]
        (-2 not reached, -1 no way to a goal, else the distance) and joint int16 [K] (sum_a act[a] * 5^a; -1 where dist <= 0)."""
        K = C.c_int64(0)
        check(lib().lle_vec_expert_table(self._h, int(map_index), None, None, 0, C.byref(K)))
        dist, joint = np.zeros(K.value, np.int32), np.zeros(K.value, np.int16)
        check(lib().lle_vec_expert_table(self._h, int(map_index), dist.ctypes.data_as(C.c_void_p), joint.ctypes.data_as(C.c_void_p),
                                         K.value, C.byref(K)))
        return dist, joint

    def export_raw(self) -> dict[str, torch.Tensor]:
        N, A, NB = self.n_envs, self.n_agents, max(self.n_beams_max, 1)
        d = self.device
        out = dict(pos=torch.zeros((N, A, 2), dtype=torch.int16, device=d), alive=torch.zeros((N, A), dtype=torch.uint8, device=d),
                   arrived=torch.zeros((N, A), dtype=torch.uint8, device=d), slot=torch.zeros((N, A), dtype=torch.uint8, device=d),
                   beam_on=torch.zeros((N, NB), dtype=torch.int64, device=d), collected=torch.zeros((N,), dtype=torch.int64, device=d),
                   counters=torch.zeros((N, 3), dtype=torch.uint8, device=d))
        check(lib().lle_vec_export_raw(self._h, out["pos"].data_ptr(), out["alive"].data_ptr(), out["arrived"].data_ptr(),
                                       out["slot"].data_ptr(), out["beam_on"].data_ptr() if self.n_beams_max else None,
                                       out["collected"].data_ptr(), out["counters"].data_ptr(), _stream_ptr(self.device)))
        return out

    _RAW_FIELDS = (("pos", torch.int16, 2), ("alive", torch.uint8, 0), ("arrived", torch.uint8, 0), ("slot", torch.uint8, 0),
                   ("avail_cache", torch.uint8, 0), ("subgoals_extras", torch.int64, 0), ("subgoals_pbrs", torch.int64, 0))

    def checkpoint(self) -> dict:
        """Everything a bit-exact resume needs (lle_vec_export_raw_state + the counters of the random streams): device tensors."""
        N, A, NB = self.n_envs, self.n_agents, max(self.n_beams_max, 1)
        d = self.device
        t = {name: torch.zeros((N, A, extra) if extra else (N, A), dtype=dt, device=d) for name, dt, extra in self._RAW_FIELDS}
        t["beam_on"] = torch.zeros((N, NB), dtype=torch.int64, device=d)
        t["collected"] = torch.zeros((N,), dtype=torch.int64, device=d)
        t["counters"] = torch.zeros((N, 3), dtype=torch.uint8, device=d)
        raw = RawState(**{k: v.data_ptr() for k, v in t.items()})
        check(lib().lle_vec_export_raw_state(self._h, C.byref(raw), _stream_ptr(self.device)))
        rc = C.c_uint32(0)
        check(lib().lle_vec_get_reset_count(self._h, C.byref(rc)))
        t["step_count"], t["reset_count"] = self.step_count, rc.value
        if self.map_index is not None:
            t["map_index"] = self.map_index.clone()
        return t

    def restore(self, ckpt: dict):
        """Inverse of checkpoint() on a batch built from the same maps and options (lle_vec_import_raw_state)."""
        keep = {k: ckpt[k].to(self.device).contiguous() for k in ("pos", "alive", "arrived", "slot", "avail_cache", "subgoals_extras",
                                                                  "subgoals_pbrs", "beam_on", "collected", "counters")}
        if self.map_index is not None:
            self.map_index.copy_(ckpt["map_index"])
        raw = RawState(**{k: v.data_ptr() for k, v in keep.items()})
        check(lib().lle_vec_import_raw_state(self._h, C.byref(raw), _stream_ptr(self.device)))
        self.step_count = int(ckpt["step_count"])
        check(lib().lle_vec_set_reset_count(self._h, int(ckpt["reset_count"])))
        self.synchronize()  # `keep` may be freed once the import kernel has run

    @property
    def step_count(self) -> int:
        v = C.c_uint64(0)
        check(lib().lle_vec_get_step_count(self._h, C.byref(v)))
        return v.value

    @step_count.setter
    def step_count(self, value: int):
        check(lib().lle_vec_set_step_count(self._h, int(value)))

    @property
    def launch_count(self) -> int:
        v = C.c_uint64(0)
        check(lib().lle_vec_launch_count(self._h, C.byref(v)))
        return v.value

    def timing_begin(self):
        check(lib().lle_vec_timing_begin(self._h, _stream_ptr(self.device)))

    def timing_end(self) -> tuple[float, int]:
        ms, n = C.c_float(0), C.c_uint64(0)
        check(lib().lle_vec_timing_end(self._h, _stream_ptr(self.device), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def synchronize(self):
        torch.cuda.current_stream(self.device).synchronize()


class PartsLoop:
    """A closed host loop over parts of one VecWorld (lle_vec_parts_begin ... lle_vec_parts_end).

        with vec.parts_loop(8, actions, reward, done) as loop:
            loop.launch()                         # step 0 (waits on the device for its actions)
            for k in range(loop.n_parts):
                actions[loop.slice(k)] = ...      # the first actions
                loop.feed(k)
            loop.launch()                         # keep two steps in flight
            for step in range(steps):
                for k in range(loop.n_parts):
                    loop.wait(k)                  # reward / done of part k, step `step`, are in the host tensors
                    if step + 1 < steps:
                        actions[loop.slice(k)] = policy(reward[loop.slice(k)], done[loop.slice(k)])
                        loop.feed(k)
                if step + 2 < steps:
                    loop.launch()
    """

    def __init__(self, vec: VecWorld, n_parts: int, actions: torch.Tensor, reward_out, done_out, after_current_stream: bool = True):
        for t, dt, shape in ((actions, torch.int8, (vec.n_envs, vec.n_agents)), (reward_out, torch.float32, (vec.n_envs, vec.reward_dim)),
                             (done_out, torch.uint8, (vec.n_envs,))):
            if t is None:
                continue
            if t.dtype != dt or tuple(t.shape) != shape or not t.is_contiguous() or t.is_cuda or not t.is_pinned():
                raise ValueError(f"parts_loop needs pinned, contiguous host tensors; expected {dt} {shape}")
        if actions is None:
            raise ValueError("parts_loop needs an actions tensor")
        self._open = False
        self.vec, self._keep = vec, (actions, reward_out, done_out)
        check(lib().lle_vec_parts_begin(vec._h, int(n_parts), actions.data_ptr(), reward_out.data_ptr() if reward_out is not None else None,
                                        done_out.data_ptr() if done_out is not None else None,
                                        _stream_ptr(vec.device) if after_current_stream else C.c_void_p(-1)))
        n = C.c_int32(0)
        check(lib().lle_vec_parts_count(vec._h, C.byref(n)))
        self.n_parts = n.value
        self.ranges = []
        for k in range(self.n_parts):
            first, count = C.c_int64(0), C.c_int64(0)
            check(lib().lle_vec_parts_range(vec._h, k, C.byref(first), C.byref(count)))
            self.ranges.append((first.value, count.value))
        self._open = True

    def slice(self, part: int) -> slice:
        first, count = self.ranges[part]
        return slice(first, first + count)

    def launch(self):
        check(lib().lle_vec_parts_launch(self.vec._h))

    def feed(self, part: int):
        check(lib().lle_vec_parts_feed(self.vec._h, int(part)))

    def wait(self, part: int):
        check(lib().lle_vec_parts_wait(self.vec._h, int(part)))

    def close(self):
        if self._open:
            self._open = False
            check(lib().lle_vec_parts_end(self.vec._h))

    def abort(self):
        if self._open:
            self._open = False
            check(lib().lle_vec_parts_abort(self.vec._h))

    def __del__(self):  # a dropped loop must not leave a launched step waiting for actions on the device
        try:
            if self._open and self.vec._h:
                self.abort()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        else:
            self.abort()  # never leave a kernel waiting for actions
        return False
