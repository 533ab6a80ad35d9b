"""`VecLLE`: the batched counterpart of `lle.LLE` (python/lle/env/env.py) — what an RL loop uses.

`lle_b200.level(6).n_envs(65536).build()` mirrors the reference's fluent builder
(python/lle/env/builder.py:30-160) for the options that exist on the accelerated path.
All per-step results are device tensors (zero-copy views, DLPack-exportable); nothing is copied to the host.
"""
from __future__ import annotations

from typing import Sequence

import torch

from .types import obs_spec
from .vec_world import Map, VecWorld, _obs_dtype


class VecLLE:
    """N lock-stepped `LLE` environments on one GPU.

    step() semantics: reward / done / events describe the transition just taken; with auto_reset (default)
    obs / state / available_actions are those of the freshly reset world when done is set (SURVEY §8d).
    """

    def __init__(self, maps, n_envs: int, *, map_of_env: Sequence[int] | None = None, device=0, multi_objective: bool = False,
                 walkable_lasers: bool = True, auto_reset: bool = True, seed: int = 0, env_id_base: int = 0, write_obs: bool = True,
                 extras=None, pbrs: dict | None = None, obs_type: str = "layered", padding_size: int = 0,
                 randomize_lasers: bool = False, state_type: str = "state", episode_stats: bool = False, obs_dtype=torch.float32):
        self.world = VecWorld(maps, n_envs, map_of_env=map_of_env, device=device, reward_dim=4 if multi_objective else 1,
                              walkable_lasers=walkable_lasers, auto_reset=auto_reset, lle_semantics=True, write_obs=write_obs,
                              seed=seed, env_id_base=env_id_base, extras=extras, pbrs=pbrs, obs_type=obs_type,
                              padding_size=padding_size, randomize_lasers=randomize_lasers, state_type=state_type,
                              episode_stats=episode_stats, obs_dtype=obs_dtype)
        if self.world.obs_invalid and write_obs:
            raise IndexError("index out of bounds: a laser colour selects a channel past the last layer")
        w = self.world
        self.n_envs, self.n_agents, self.n_actions = w.n_envs, w.n_agents, 5
        self.width, self.height = w.width, w.height  # env.py:120-126
        self.observation_shape = tuple(w.obs.shape[1:]) if self._flat(w) else w.obs_shape  # one agent's observation
        self.state_shape = tuple(w.state_of_type.shape[1:])  # env.py:100: the shape of get_state()
        self.reward_dim = w.reward_dim

    @staticmethod
    def _flat(w) -> bool:
        return w.obs is not None and w._flatten

    # tensors (views on device buffers)
    obs = property(lambda self: self.world.obs)                      # (N, C, H, W)
    obs_per_agent = property(lambda self: self.world.obs_per_agent)  # (N, A, C, H, W), stride-0 agent dim
    state = property(lambda self: self.world.state_of_type)          # (N, 3A+G), or (N, *shape) of Builder.state_type
    state_vector = property(lambda self: self.world.state)           # (N, 3A+G) always: PyWorldState::as_array
    available_actions = property(lambda self: self.world.avail)      # (N, A, 5) u8
    reward = property(lambda self: self.world.reward)                # (N, reward_dim)
    done = property(lambda self: self.world.done)                    # (N,) u8
    events = property(lambda self: self.world.events)                # (N, A) u8
    actions = property(lambda self: self.world.actions)              # (N, A) i8
    err = property(lambda self: self.world.err)                      # (N,) u8
    extras = property(lambda self: self.world.extras)                # (N, A, n_sources) f32 or None
    info = property(lambda self: self.world.info)                    # Step.info per env (episode_stats=True)
    ep_return = property(lambda self: self.world.ep_return)          # (N, reward_dim) running episode return
    ep_length = property(lambda self: self.world.ep_length)          # (N,) running episode length
    last_return = property(lambda self: self.world.last_return)      # (N, reward_dim) return of the last finished episode
    last_length = property(lambda self: self.world.last_length)      # (N,)

    def reset(self, mask: torch.Tensor | None = None):
        self.world.reset(mask)
        return self.obs, self.state

    def step(self, actions: torch.Tensor | None = None):
        """actions: int8 (N, A) on the device, or None to sample uniformly among available actions on the GPU."""
        self.world.step(actions)
        return self.obs, self.state, self.reward, self.done

    def dlpack(self, name: str):
        return getattr(self, name).__dlpack__()

    def run_host_policy(self, policy, steps: int, n_parts: int = 8, first_actions=None):
        """Closed loop with a policy that runs ON THE HOST between steps (the reference's `while not done: env.step(policy(obs))`,
        python/lle/env/env.py:165-189, over N envs): `policy(part_slice, reward, done)` gets numpy views of one part's results in
        pinned host memory and returns that part's next actions (int8 array (n, A), or None to keep everybody on STAY).  Every
        step is one launch over the whole batch; the step kernel waits part by part for the actions (lle_vec_parts_*), so the
        device keeps stepping the other parts while the policy thinks.  Returns (reward, done) of the last step (host tensors).
        Observations stay on the device (`obs`): a host policy that needs them copies the slices it wants."""
        w = self.world
        act = torch.full((w.n_envs, w.n_agents), 4, dtype=torch.int8).pin_memory()
        rew = torch.zeros((w.n_envs, w.reward_dim), dtype=torch.float32).pin_memory()
        done = torch.zeros((w.n_envs,), dtype=torch.uint8).pin_memory()
        act_np, rew_np, done_np = act.numpy(), rew.numpy(), done.numpy()
        if first_actions is not None:
            act_np[...] = first_actions
        with w.parts_loop(n_parts, act, rew, done) as loop:
            slices = [loop.slice(k) for k in range(loop.n_parts)]
            loop.launch()
            for k in range(loop.n_parts):
                loop.feed(k)
            if steps > 1:
                loop.launch()
            for s in range(steps):
                for k, sl in enumerate(slices):
                    loop.wait(k)
                    if s + 1 < steps:
                        nxt = policy(sl, rew_np[sl], done_np[sl])
                        act_np[sl] = 4 if nxt is None else nxt
                        loop.feed(k)
                if s + 2 < steps:
                    loop.launch()
        return rew, done


class VecWorldGroup:
    """Several `VecWorld`s stepped together — for batches whose maps do not share one tensor shape, e.g. the six
    built-in levels mixed (BASELINE.json configs[3]: channel counts 6/8/8/8/12/12 => one sub-batch per level)."""

    def __init__(self, specs: Sequence[tuple], **kw):
        """specs: (maps, n_envs) pairs; kw: VecWorld options.  env ids are assigned contiguously across sub-batches."""
        base = int(kw.pop("env_id_base", 0))
        self.parts = []
        for maps, n in specs:
            self.parts.append(VecWorld(maps, n, env_id_base=base, **kw))
            base += n
        self.n_envs = sum(p.n_envs for p in self.parts)

    def reset(self):
        for p in self.parts:
            p.reset()

    def step(self):
        """Device-sampled actions for every sub-batch; the launches are adjacent on the stream and overlap (PDL)."""
        for p in self.parts:
            p.step(None)

    def rollout(self, n_steps: int):
        for p in self.parts:
            p.rollout(n_steps)

    def synchronize(self):
        for p in self.parts:
            p.synchronize()


class Builder:
    """Subset of python/lle/env/builder.py that exists on the accelerated path."""

    def __init__(self, maps, name: str = "LLE"):
        self._maps = maps
        self._kw = {}
        self._n = 1
        self._name = name  # builder.py:25

    def n_envs(self, n: int):
        self._n = int(n)
        return self

    def name(self, name: str):
        """builder.py:117-119"""
        self._name = name
        return self

    def device(self, device):
        self._kw["device"] = device
        return self

    def seed(self, seed: int):
        self._kw["seed"] = int(seed)
        return self

    def multi_objective(self, enabled: bool = True):
        if enabled and "pbrs" in self._kw:  # builder.py:66-73
            raise ValueError("Cannot set multi-objective after setting a reward shaping strategy. Call `multi_objective()` first.")
        if enabled and not self._kw.get("multi_objective"):
            self._name = f"{self._name}-MO"  # builder.py:75
        self._kw["multi_objective"] = enabled
        return self

    def pbrs(self, gamma: float = 0.99, reward_value: float = 0.5, lasers_to_reward=None, with_extras: bool = True):
        """Potential-based reward shaping on laser crossings (builder.py:77-110).  `lasers_to_reward`: source positions
        (i, j) or source indices; None = all sources."""
        rewarded = None
        if lasers_to_reward is not None:
            src_pos = [s.pos for s in self._maps.sources()] if isinstance(self._maps, Map) else None
            rewarded = []
            for item in lasers_to_reward:
                if isinstance(item, tuple):
                    if src_pos is None or item not in src_pos:
                        raise ValueError(f"Invalid laser source: {item}")
                    rewarded.append(src_pos.index(item))
                else:
                    rewarded.append(int(item))
        self._kw["pbrs"] = dict(gamma=gamma, reward_value=reward_value, lasers_to_reward=rewarded, with_extras=with_extras)
        self._name = f"{self._name}-PBRS"  # builder.py:102
        return self

    def add_extras(self, *extras):
        """Only "laser_subgoal" exists on the accelerated path (builder.py:124-150)."""
        for e in extras:
            if e != "laser_subgoal":
                raise ValueError(f"Invalid extra type: {e}")
            self._kw["extras"] = "laser_subgoal"
        return self

    def randomize_lasers(self, enabled: bool = True):
        """Randomize the colour of the lasers at each reset (builder.py:112-115, env.py:198-200)."""
        self._kw["randomize_lasers"] = bool(enabled)
        return self

    def walkable_lasers(self, walkable: bool = True):
        self._kw["walkable_lasers"] = walkable
        return self

    def auto_reset(self, enabled: bool = True):
        self._kw["auto_reset"] = enabled
        return self

    def obs_type(self, obs_type: str, padding_size: int = 0):
        """Builder.obs_type (builder.py:42-49): any ObservationType value but "rgb-image"."""
        obs_spec(obs_type, padding_size)  # ValueError / NotImplementedError
        self._kw["obs_type"], self._kw["padding_size"] = obs_type, int(padding_size)
        return self

    def obs_dtype(self, dtype=torch.float32):
        """Element type of the observation: torch.float32 (default) or torch.int8 (also "float32" / "int8"), a quarter of the
        bytes for layered and perspective observations (VecWorld's obs_dtype)."""
        self._kw["obs_dtype"] = _obs_dtype(dtype)  # ValueError
        return self

    def episode_stats(self, enabled: bool = True):
        """Step.info (env.py:174-188) and episode return / length per env, kept by the step kernel."""
        self._kw["episode_stats"] = bool(enabled)
        return self

    def state_type(self, state_type: str):
        """Builder.state_type (builder.py:51-58): any ObservationType value but "rgb-image"."""
        obs_spec(state_type)  # ValueError / NotImplementedError
        self._kw["state_type"] = getattr(state_type, "value", state_type)
        return self

    def death_strategy(self, strategy: str):
        if strategy == "respawn":
            raise NotImplementedError("Respawn strategy is not implemented yet")  # env.py:106-108
        if strategy != "end":
            raise ValueError(f"Unknown death strategy: {strategy}")
        return self

    def build(self) -> VecLLE:
        env = VecLLE(self._maps, self._n, **self._kw)
        env.name = self._name
        return env


def level(n: int) -> Builder:
    return Builder(Map(level=n), f"LLE-lvl{n}")  # env.py:238-242


def from_str(world_string: str) -> Builder:
    return Builder(Map(world_string))


def from_file(path: str) -> Builder:
    import os

    with open(path) as f:
        return Builder(Map(f.read()), f"LLE-{os.path.basename(path)}")  # env.py:226-232
