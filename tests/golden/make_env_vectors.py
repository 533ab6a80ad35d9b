"""Generates tests/golden/env_vectors.npz by running the REFERENCE's own Python environment layer, unmodified:

    python/lle/observations.py          every ObservationGenerator  (:145-395)
    python/lle/env/reward_strategy.py   SingleObjective / MultiObjective / PotentialShapedLLE  (:58-181)
    python/lle/env/extras_generators.py LaserSubgoal  (:75-101)
    python/lle/env/env.py               LLE.step / reset / set_state / available_actions / compute_done  (:146-254)
    python/lle/env/builder.py           Builder  (the environments below are built through it)

imported from /root/reference with two stubs: the native module (`lle.world`, `lle.tiles` — served by the oracle's
`World`, oracle/lle_oracle.py, because the Rust crate cannot be built in this image) and `marlenv` (absent; only its
containers are used on this path: spaces, Observation, State, Step).  So every number in the fixture except the engine
transition itself (positions, beams, events — pinned by the transcribed engine KATs) is an OUTPUT OF REFERENCE CODE:
observations of every type, availability masks incl. walkable_lasers=False, rewards of every strategy, done, the
Step.info metrics, LaserSubgoal extras, and the effect of LLE.set_state on the strategy's counters.

A case = (map, options).  Its script is a list of operations replayed by tests/test_env_vectors.py against the oracle
(CPU suite) and the CUDA path (-m gpu): step(actions) / reset() / set_state(state).  Actions are drawn with a seeded
numpy generator among the actions the reference's own `available_actions()` allows.

Usage (build container only; /root/reference does not exist on the GPU box):
    python tests/golden/make_env_vectors.py [/root/reference]
"""
import importlib
import json
import os
import sys
import types

import numpy as np

REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import lle_oracle as lo  # noqa: E402  (the engine under the reference's Python layer)

OBS_TYPES = ["layered", "flattened", "partial3x3", "partial5x5", "partial7x7", "state", "normalized-state", "perspective",
             "layered-padded-1", "layered-padded-2", "layered-padded-3"]
STEPS = 64


# ---------------------------------------------------------------------------------------------- stubs
def stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


class _Space:
    def __init__(self, shape):
        self.shape = shape

    def repeat(self, n):
        return self


class DiscreteSpace(_Space):
    @staticmethod
    def action(n, labels=None):
        s = DiscreteSpace((n,))
        s.n = n
        return s


class ContinuousSpace(_Space):
    @staticmethod
    def from_shape(n):
        return ContinuousSpace((n,) if isinstance(n, int) else tuple(n))


class DiscreteMARLEnv:
    """What LLE.__init__ hands to marlenv (env.py:96-104); `n_actions` is read back by LLE.available_actions (:147)."""

    def __init__(self, n_agents, action_space, observation_shape, state_shape, reward_space, extras_shape, extras_meanings):
        self.n_agents, self.n_actions = n_agents, action_space.n
        self.observation_shape, self.state_shape, self.reward_space = observation_shape, state_shape, reward_space
        self.extras_shape, self.extras_meanings = extras_shape, extras_meanings

    @property
    def name(self):
        return type(self).__name__


class Observation:
    def __init__(self, data, available_actions, extras):
        self.data, self.available_actions, self.extras = data, available_actions, extras


class State:
    def __class_getitem__(cls, item):  # annotated as State[npt.NDArray[np.float32]] (env.py:208)
        return cls

    def __init__(self, data):
        self.data = data
        self.shape = data.shape


class Step:
    def __init__(self, actions, obs, state, reward, done, info):
        self.actions, self.obs, self.state, self.reward, self.done, self.info = actions, obs, state, reward, done, info


stub("marlenv", models=stub("marlenv.models", DiscreteMARLEnv=DiscreteMARLEnv, DiscreteSpace=DiscreteSpace, ContinuousSpace=ContinuousSpace,
                            Observation=Observation, State=State, Step=Step))


class Action(int):
    """The native lle.world.Action as the Python layer uses it (src/bindings/world/pyaction.rs:26-160): `Action(value)`,
    `.value`, `.delta`, `.name`, `Action.cardinality()`, `Action.variants()`; handed to the oracle's World.step as an int."""
    _NAMES = ("NORTH", "SOUTH", "EAST", "WEST", "STAY")

    def __new__(cls, value):
        value = int(value)
        if not 0 <= value < 5:
            raise ValueError(f"Invalid action value: {value}")
        return super().__new__(cls, value)

    value = property(lambda self: int(self))
    name = property(lambda self: Action._NAMES[int(self)])
    delta = property(lambda self: lo.Action(int(self)).delta)

    @staticmethod
    def cardinality():
        return 5

    @staticmethod
    def variants():
        return [Action(k) for k in range(5)]


class World(lo.World):
    def available_actions(self):
        return [[Action(int(a)) for a in row] for row in super().available_actions()]

    def step(self, actions):
        return super().step([lo.Action(int(a)) for a in actions])


pkg = stub("lle")
pkg.__path__ = [os.path.join(REF, "python", "lle")]
stub("lle.world", World=World, WorldState=lo.WorldState, Action=Action, EventType=lo.EventType, WorldEvent=lo.WorldEvent)
pkg.tiles = stub("lle.tiles", LaserSource=lo.LaserSource, Laser=lo.Laser, Gem=lo.Gem, Direction=lo.Direction)
# everything below is the reference's own source, imported through the normal machinery from REF/python/lle
observations = importlib.import_module("lle.observations")
env_pkg = importlib.import_module("lle.env")
Builder = env_pkg.Builder
for mod in ("lle.observations", "lle.env.env", "lle.env.builder", "lle.env.reward_strategy", "lle.env.extras_generators", "lle.env.utils"):
    assert sys.modules[mod].__file__.startswith(REF), mod


# ---------------------------------------------------------------------------------------------- cases
EXTRA_MAPS = {
    # python/tests/test_observations.py::test_layered_observation_laser_source_agent_id_above_n_agents: colour 1 with one agent
    # lands in the WALL channel; colour 7 indexes past the last channel and the generator raises IndexError
    "colour-spills-into-wall-channel": "S0 . . .\n.  . . L1W\nX  . G .",
    "colour-out-of-range": "S0 . . .\n.  . . L7W\nX  . G .",
    "gems-and-void": "S0 G . V S1\n.  . G . .\nX  . . G X",
}


def maps():
    out = dict(EXTRA_MAPS)
    for n in range(1, 7):
        with open(os.path.join(HERE, "levels", f"lvl{n}")) as f:
            out[f"lvl{n}"] = f.read()
    with open(os.path.join(HERE, "layouts.json")) as f:
        for name, text in json.load(f).items():
            out[name] = text
    return out


CONFIGS = {
    # name: (multi_objective, walkable_lasers, extras, pbrs kwargs | None)
    "single": (False, True, False, None),
    "multi-nowalk-extras": (True, False, True, None),
    "pbrs": (False, True, False, dict(gamma=0.99, reward_value=0.5, lasers_to_reward=None, with_extras=True)),
    "multi-pbrs-first-source": (True, True, False, dict(gamma=0.9, reward_value=1.0, lasers_to_reward=[0], with_extras=False)),
}


def build_env(text, cfg):
    multi, walkable, extras, pbrs = CONFIGS[cfg]
    world = World(text)
    b = Builder(world).walkable_lasers(walkable)
    if multi:
        b = b.multi_objective()
    if extras:
        b = b.add_extras("laser_subgoal")
    if pbrs is not None:
        kw = dict(pbrs)
        if kw["lasers_to_reward"] is not None:
            if not world.laser_sources:
                return None, None
            kw["lasers_to_reward"] = [world.laser_sources[k] for k in kw["lasers_to_reward"]]
        b = b.pbrs(**kw)
    return world, b.build()


def to_i8(a):
    a = np.asarray(a)
    r = a.astype(np.int8)
    assert np.array_equal(r.astype(a.dtype), a), "value not representable as int8"
    return r


class Recorder:
    """One case: the script and, after every operation, what the reference's code returns."""

    def __init__(self, world, env, with_obs_types):
        self.world, self.env = world, env
        self.gens = {}
        if with_obs_types:
            for t in OBS_TYPES:
                try:
                    self.gens[t] = observations.ObservationType.from_str(t).get_observation_generator(world)
                except IndexError:  # a laser colour >= the channel count of this type: the reference raises
                    self.gens[t] = None
        self.ops, self.rows = [], []

    def snapshot(self, op, actions=None, state=None, step=None):
        env, world = self.env, self.world
        A = world.n_agents
        row = {"op": op}
        if actions is not None:
            row["actions"] = [int(a) for a in actions]
        if state is not None:
            row["set_state"] = [[list(p) for p in state.agents_positions], [bool(g) for g in state.gems_collected],
                                [bool(a) for a in state.agents_alive]]
        ob = step.obs if step is not None else env.get_observation()
        row["avail"] = np.asarray(ob.available_actions, dtype=bool)
        row["extras"] = np.asarray(ob.extras, dtype=np.float32)
        row["state"] = np.asarray(env.get_state().data, dtype=np.float32)
        row["done"] = bool(env.done)
        row["n_arrived"] = int(env.n_arrived)
        if step is not None:
            row["reward"] = np.asarray(step.reward, dtype=np.float64)  # PBRS adds a python float: keep what numpy returned
            row["reward_dtype"] = str(np.asarray(step.reward).dtype)
            info = step.info
            row["info"] = [int(info["gems_collected"]), float(info["exit_rate"])] + [int(bool(info[f"has-arrived-{i}"])) for i in range(A)] + \
                          [int(bool(info[f"is-alive-{i}"])) for i in range(A)]
        obs = {"layered": np.asarray(ob.data)} if not self.gens else {}
        for t, g in self.gens.items():
            if g is not None:
                obs[t] = np.asarray(g.observe())
        row["obs"] = obs
        self.rows.append(row)


def careful(world, mask, rng):
    """Drops (most of the time) the moves that end on a lit laser of another colour or in a void, so that some episodes
    live long enough to collect gems and reach the exits.  Only the CHOICE of actions: every action stays available."""
    lasers, voids = world.lasers, set(world.void_pos)
    out = mask.copy()
    for a, pos in enumerate(world.agents_positions):
        for act in np.flatnonzero(mask[a]):
            d = Action(int(act)).delta
            new = (pos[0] + d[0], pos[1] + d[1])
            if (new in voids or any(l.pos == new and l.agent_id != a and l.is_on for l in lasers)) and rng.random() < 0.95:
                out[a, act] = False
        if not out[a].any():
            out[a] = mask[a]
    return out


def run_case(text, cfg, seed, with_obs_types, policy="random"):
    world, env = build_env(text, cfg)
    if env is None:
        return None
    rng = np.random.default_rng(seed)
    rec = Recorder(world, env, with_obs_types)
    env.reset()
    for g in rec.gens.values():
        if g is not None:
            g.reset()
    rec.snapshot("reset")
    saved = []
    for t in range(STEPS):
        if env.done:
            env.reset()
            for g in rec.gens.values():
                if g is not None:
                    g.reset()
            rec.snapshot("reset")
            saved = []
            continue
        if saved and rng.random() < 0.08:  # LLE.set_state (env.py:208-216) with a state seen earlier in this episode
            st = saved[int(rng.integers(len(saved)))]
            env.set_state(st)
            rec.snapshot("set_state", state=st)
            continue
        mask = env.available_actions()
        if policy == "careful":
            mask = careful(world, mask, rng)
        acts = [int(rng.choice(np.flatnonzero(mask[a]))) for a in range(world.n_agents)]
        step = env.step(acts)
        rec.snapshot("step", actions=acts, step=step)
        if not env.done:
            saved.append(world.get_state())
    return rec


def store(arrays, index, name, text, cfg, policy, rec):
    key = f"{name}|{cfg}|{policy}"
    rows = rec.rows
    script = []
    for r in rows:
        e = {"op": r["op"], "done": r["done"], "n_arrived": r["n_arrived"]}
        for k in ("actions", "set_state", "info", "reward_dtype"):
            if k in r:
                e[k] = r[k]
        script.append(e)
    entry = dict(map=name, text=text, config=cfg, policy=policy, key=key, n_agents=rec.world.n_agents, script=script,
                 obs_types=sorted(rows[0]["obs"]), obs_raises=sorted(t for t, g in rec.gens.items() if g is None),
                 obs_agents={}, obs_tiled={})
    arrays[f"{key}|avail"] = np.stack([r["avail"] for r in rows]).astype(np.uint8)
    arrays[f"{key}|extras"] = to_i8(np.stack([r["extras"] for r in rows]))
    arrays[f"{key}|state"] = to_i8(np.stack([r["state"] for r in rows]))
    rw = [r["reward"] for r in rows if "reward" in r]
    if rw:
        arrays[f"{key}|reward"] = np.stack(rw)  # float64 holding the float32 (or python-float-added) values exactly
    for t in entry["obs_types"]:
        data = np.stack([r["obs"][t] for r in rows])
        entry["obs_agents"][t] = int(data.shape[1])
        tiled = t in ("layered", "flattened", "state", "normalized-state") or t.startswith("layered-padded")
        if tiled:  # np.tile over the agent dimension (observations.py:158, :266): keep one copy, after checking
            assert all(np.array_equal(data[:, 0], data[:, k]) for k in range(data.shape[1]))
            data = data[:, 0]
        entry["obs_tiled"][t] = bool(tiled)
        arrays[f"{key}|obs|{t}"] = data.astype(np.float32) if t == "normalized-state" else to_i8(data)
    index.append(entry)


def main():
    arrays, index = {}, []
    for m_idx, (name, text) in enumerate(maps().items()):
        for c_idx, cfg in enumerate(CONFIGS):
            for policy in ("random", "careful"):
                try:
                    rec = run_case(text, cfg, seed=1000 * m_idx + 10 * c_idx + (policy == "careful"), with_obs_types=cfg == "single",
                                   policy=policy)
                except IndexError:
                    # Layered(world) raises in its constructor when a laser colour indexes past the channels (observations.py:235)
                    index.append(dict(map=name, text=text, config=cfg, raises="IndexError"))
                    break
                if rec is None:  # the configuration names a laser source and the map has none
                    break
                store(arrays, index, name, text, cfg, policy, rec)
        print(name, "done", file=sys.stderr)
    out = os.path.join(HERE, "env_vectors.npz")
    save(arrays, index, out)
    print(f"{out}: {len(index)} cases, {os.path.getsize(out) / 1e6:.2f} MB")


def save(arrays: dict, index: list, out: str) -> None:
    """One flat array per dtype, a JSON layout (key -> dtype, offset, shape) and the JSON index, in an .npz whose entries are
    LZMA-compressed: two thousand small entries cost more in zip headers than in data, and LZMA packs the observations several
    times tighter than deflate.  tests/test_env_vectors.py cuts the arrays back out of the flat ones."""
    import zipfile

    flat, layout = {}, {}
    for key, a in arrays.items():
        parts = flat.setdefault(a.dtype.name, [])
        layout[key] = [a.dtype.name, sum(p.size for p in parts), list(a.shape)]
        parts.append(a.ravel())
    entries = {name: np.concatenate(parts) for name, parts in flat.items()}
    entries["layout"] = np.frombuffer(json.dumps(layout).encode(), dtype=np.uint8)
    entries["index"] = np.frombuffer(json.dumps(index).encode(), dtype=np.uint8)
    with zipfile.ZipFile(out, "w", compression=zipfile.ZIP_LZMA) as zf:
        for name, a in entries.items():
            with zf.open(name + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, a)


if __name__ == "__main__":
    main()
