"""Replays tests/golden/env_vectors.npz — outputs of the REFERENCE's own, unmodified Python environment layer
(python/lle/observations.py, env/reward_strategy.py, env/extras_generators.py, env/env.py, env/builder.py, run by
tests/golden/make_env_vectors.py in the build container) — against the oracle (CPU suite) and the CUDA path (-m gpu).

Every case is a script of LLE.step / LLE.reset / LLE.set_state calls on one map with one set of options; after every call the
fixture holds what the reference returned: the observation of every ObservationType, the availability mask (both
walkable_lasers settings), the LaserSubgoal extras, the state vector, the reward of every strategy (SingleObjective,
MultiObjective, PotentialShapedLLE over either), done, n_arrived and the Step.info metrics.  Bit-exact comparison.
"""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

_DATA = None


def data():
    global _DATA
    if _DATA is None:
        z = np.load(os.path.join(GOLDEN, "env_vectors.npz"))
        # the file holds one flat array per dtype (tests/golden/make_env_vectors.py: save); the layout cuts the recorded arrays out
        layout = json.loads(bytes(z["layout"]).decode())
        flat = {dt: z[dt] for dt in {dt for dt, _, _ in layout.values()}}
        arrays = {key: flat[dt][off:off + int(np.prod(shape))].reshape(shape) for key, (dt, off, shape) in layout.items()}
        _DATA = (arrays, json.loads(bytes(z["index"]).decode()))
    return _DATA


CONFIG_KW = {
    "single": {},
    "multi-nowalk-extras": dict(multi_objective=True, walkable_lasers=False, extras="laser_subgoal"),
    "pbrs": dict(pbrs=dict(gamma=0.99, reward_value=0.5, lasers_to_reward=None, with_extras=True)),
    "multi-pbrs-first-source": dict(multi_objective=True, pbrs=dict(gamma=0.9, reward_value=1.0, lasers_to_reward=[0], with_extras=False)),
}


def cases():
    return [e for e in data()[1] if "raises" not in e]


def map_names():
    return sorted({e["map"] for e in cases()})


def replay(api, entry, obs_type, check_env=True):
    """Runs the case's script on `api.LLE` with the given observation type; compares after every operation."""
    z, _ = data()
    key = entry["key"]
    A = entry["n_agents"]
    env = api.LLE(entry["text"], obs_type=obs_type, **CONFIG_KW[entry["config"]])
    want_obs = z[f"{key}|obs|{obs_type}"]
    tiled = entry["obs_tiled"][obs_type]
    avail, extras, state = z[f"{key}|avail"], z[f"{key}|extras"], z[f"{key}|state"]
    reward = z[f"{key}|reward"] if f"{key}|reward" in z else None
    n_step = 0
    for row, op in enumerate(entry["script"]):
        where = f"{key} [{obs_type}] op {row} ({op['op']})"
        step = None
        if op["op"] == "reset":
            env.reset()
        elif op["op"] == "set_state":
            pos, gems, alive = op["set_state"]
            env.set_state(api.WorldState([tuple(p) for p in pos], gems, alive))
        else:
            step = env.step(op["actions"])
        obs = np.asarray(env.observe())
        assert obs.dtype == np.float32, where
        assert obs.shape[0] == entry["obs_agents"][obs_type], where
        if tiled:  # the reference returns np.tile(block, (A, ...)): every agent's copy must equal the recorded block
            assert obs.shape[1:] == want_obs[row].shape, where
            for k in range(obs.shape[0]):
                assert np.array_equal(obs[k], want_obs[row].astype(np.float32)), f"{where}: observation (agent copy {k})"
        else:
            assert obs.shape == want_obs[row].shape and np.array_equal(obs, want_obs[row].astype(np.float32)), f"{where}: observation"
        if not check_env:
            if step is not None:
                n_step += 1
            continue
        assert np.array_equal(np.asarray(env.available_actions(), dtype=np.uint8), avail[row]), f"{where}: available actions"
        assert np.array_equal(np.asarray(env.get_state()), state[row].astype(np.float32)), f"{where}: state"
        got_extras = np.asarray(env.extras())
        assert got_extras.shape == extras[row].shape and np.array_equal(got_extras, extras[row].astype(np.float32)), f"{where}: extras"
        assert bool(env.done) == op["done"], f"{where}: done"
        assert int(env.n_arrived) == op["n_arrived"], f"{where}: n_arrived"
        if step is not None:
            # the reference's reward is float32, except MultiObjective + PBRS whose np.concat with a python float gives float64:
            # the device stores float32, i.e. the rounded value
            want = reward[n_step].astype(np.float32)
            got = np.asarray(step.reward, dtype=np.float32)
            assert got.shape == want.shape and np.array_equal(got, want), f"{where}: reward {got} != {want}"
            assert bool(step.done) == op["done"], where
            assert np.array_equal(np.asarray(step.available_actions, dtype=np.uint8), avail[row]), where
            info = step.info
            want_info = op["info"]
            got_info = [int(info["gems_collected"]), float(info["exit_rate"])] + [int(info[f"has-arrived-{i}"]) for i in range(A)] + \
                       [int(info[f"is-alive-{i}"]) for i in range(A)]
            assert got_info == want_info, f"{where}: Step.info {got_info} != {want_info}"
            n_step += 1


@pytest.mark.parametrize("name", map_names())
def test_env_layer_matches_reference_python(api, name):
    """Rewards, done, availability, extras, state, info and the layered observation for every option set."""
    for entry in cases():
        if entry["map"] == name:
            replay(api, entry, "layered")


@pytest.mark.parametrize("obs_type", ["flattened", "partial3x3", "partial5x5", "partial7x7", "state", "normalized-state", "perspective",
                                      "layered-padded-1", "layered-padded-2", "layered-padded-3"])
def test_observation_types_match_reference_python(api, obs_type):
    """Every other ObservationType.get_observation_generator(world).observe() along the same rollouts."""
    n = 0
    for entry in cases():
        if entry["config"] == "single" and obs_type in entry["obs_types"]:
            replay(api, entry, obs_type, check_env=False)
            n += 1
    assert n >= 60


@pytest.mark.parametrize("state_type", ["layered", "flattened", "partial3x3", "partial7x7", "normalized-state", "perspective", "layered-padded-2"])
def test_state_types_match_reference_python(api, state_type):
    """Builder.state_type (builder.py:51-58): LLE.get_state() is the FIRST agent's observation of that generator
    (`_state_generator.get_state()`, observations.py:118-119, env.py:205-206) after every step / reset / set_state."""
    z, _ = data()
    n = 0
    for entry in cases():
        if entry["config"] != "single" or entry["policy"] != "careful" or state_type not in entry["obs_types"]:
            continue
        key = entry["key"]
        want = z[f"{key}|obs|{state_type}"]
        tiled = entry["obs_tiled"][state_type]
        env = api.LLE(entry["text"], state_type=state_type)
        for row, op in enumerate(entry["script"]):
            if op["op"] == "reset":
                env.reset()
            elif op["op"] == "set_state":
                pos, gems, alive = op["set_state"]
                env.set_state(api.WorldState([tuple(p) for p in pos], gems, alive))
            else:
                env.step(op["actions"])
            expect = (want[row] if tiled else want[row][0]).astype(np.float32)
            got = np.asarray(env.get_state())
            assert got.shape == expect.shape and np.array_equal(got, expect), f"{key} [state_type {state_type}] op {row}"
        n += 1
    assert n >= 30


def test_colour_past_the_last_channel_raises_like_the_reference(api):
    """Layered(world) raises IndexError in its constructor (observations.py:235) for every option set of that map."""
    raising = [e for e in data()[1] if "raises" in e]
    assert raising
    for e in raising:
        with pytest.raises(IndexError):
            env = api.LLE(e["text"], **CONFIG_KW[e["config"]])
            env.observe()
