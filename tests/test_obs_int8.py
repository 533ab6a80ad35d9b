"""int8 observations (lle_vec_options.obs_dtype = LLE_DTYPE_I8, VecWorld(obs_dtype=torch.int8)).

Every value of a layered, padded, flattened or perspective observation is -1, 0 or 1, so the int8 observation must be the f32
one exactly.  The GPU tests run twins: an f32 vec and an int8 vec with the same maps, seed and options, stepped alike, and after
every operation `obs_i8.float()` equals `obs_f32` bit for bit and every other output and the raw engine state are identical.
The CPU tests check the C ABI mirrors and the argument validation.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from _util import level_text

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _native():
    from lle_b200 import _native as N

    return N


# ----------------------------------------------------------------------------------------------------------------- CPU
def test_abi_struct_layout_matches_ctypes(tmp_path):
    """sizeof / offsetof of lle_vec_options and lle_vec_buffers as a C compiler lays them out equal the ctypes mirrors."""
    N = _native()
    fields = {"lle_vec_options": N.VecOptions, "lle_vec_buffers": N.VecBuffers}
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "lle_b200.h"', "int main(void) {"]
    for name, cls in fields.items():
        lines.append(f'    printf("{name} sizeof %zu\\n", sizeof({name}));')
        for f, _ in cls._fields_:
            lines.append(f'    printf("{name} {f} %zu\\n", offsetof({name}, {f}));')
    lines += ["    return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-std=c99", "-I", os.path.join(_REPO, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    seen = 0
    for line in filter(None, out):
        name, field, value = line.split()
        cls = fields[name]
        want = C.sizeof(cls) if field == "sizeof" else getattr(cls, field).offset
        assert int(value) == want, (name, field)
        seen += 1
    assert seen == 2 + len(N.VecOptions._fields_) + len(N.VecBuffers._fields_)
    assert N.VecOptions.obs_dtype.offset > N.VecOptions.episode_stats.offset
    assert N.VecBuffers.obs_i8.offset > N.VecBuffers.last_length.offset


def test_default_options_are_float32():
    N = _native()
    opts = N.VecOptions()
    opts.obs_dtype = 7
    N.lib().lle_vec_default_options(C.byref(opts))
    assert opts.obs_dtype == N.DTYPE_F32 == 0 and N.DTYPE_I8 == 1


def test_int8_argument_validation_precedes_any_device_call():
    """An unknown obs_dtype, or int8 with partial or state observations, is refused with LLE_INVALID_ARGUMENT (202) before a device
    is touched (this runs without a GPU)."""
    N = _native()
    L = N.lib()
    m6 = C.c_void_p()
    assert L.lle_map_level(6, C.byref(m6)) == 0
    one = (C.c_void_p * 1)(m6)
    out = C.c_void_p()

    def create(**fields):
        o = N.VecOptions()
        L.lle_vec_default_options(C.byref(o))
        for k, v in fields.items():
            setattr(o, k, v)
        return L.lle_vec_create(one, 1, None, 16, C.byref(o), C.byref(out))

    for bad in (2, -1, 255):
        assert create(obs_dtype=bad) == 202 and b"obs_dtype" in L.lle_last_error()
    assert create(obs_dtype=N.DTYPE_I8, obs_type=1, obs_param=3) == 202 and b"int8" in L.lle_last_error()   # partial3x3
    assert create(obs_dtype=N.DTYPE_I8, obs_type=3, obs_param=0) == 202 and b"int8" in L.lle_last_error()   # state
    assert create(obs_dtype=N.DTYPE_I8, obs_type=3, obs_param=1) == 202                                       # normalized-state
    assert not out.value
    L.lle_map_free(m6)


def test_python_dtype_argument():
    from lle_b200.vec_world import _obs_dtype

    assert _obs_dtype("int8") is torch.int8 and _obs_dtype(torch.int8) is torch.int8
    assert _obs_dtype("float32") is torch.float32 and _obs_dtype(torch.float32) is torch.float32
    for bad in ("float16", torch.bfloat16, torch.uint8, None):
        with pytest.raises(ValueError):
            _obs_dtype(bad)
    import lle_b200

    with pytest.raises(ValueError):
        lle_b200.level(1).obs_dtype("int4")
    assert lle_b200.level(1).obs_dtype("int8")._kw["obs_dtype"] is torch.int8


# ----------------------------------------------------------------------------------------------------------------- GPU
_OUTPUTS = ("state", "avail", "reward", "done", "events", "actions", "err", "extras", "info_bytes", "ep_return", "ep_length",
            "last_return", "last_length", "map_index", "state_obs")


def twins(maps, n, **kw):
    import lle_b200

    f = lle_b200.VecWorld(maps, n, **kw)
    i = lle_b200.VecWorld(maps, n, obs_dtype=torch.int8, **kw)
    assert f.obs.dtype == torch.float32 and i.obs.dtype == torch.int8
    assert i.obs.shape == f.obs.shape
    return f, i


def assert_twins(f, i, where=""):
    torch.cuda.synchronize()
    assert i.obs.dtype == torch.int8, where
    assert torch.equal(i.obs.float(), f.obs), f"{where}: observation"
    for name in _OUTPUTS:
        a, b = getattr(f, name), getattr(i, name)
        assert (a is None) == (b is None), f"{where}: {name}"
        if a is not None:
            assert torch.equal(a, b), f"{where}: {name}"
    ra, rb = f.export_raw(), i.export_raw()
    for name in ra:
        assert torch.equal(ra[name], rb[name]), f"{where}: raw {name}"


def run_twins(maps, n, steps, check_every=1, **kw):
    f, i = twins(maps, n, **kw)
    assert_twins(f, i, "after creation")
    for t in range(steps):
        f.step(None)
        i.step(None)
        if t % check_every == 0 or t == steps - 1:
            assert_twins(f, i, f"step {t}")
    return f, i


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 2, 3, 4, 5, 6])
def test_levels(level):
    """Levels 1-6: the fast kernel and the thread-per-world kernel; supplied actions too."""
    f, i = run_twins([level_text(level)], 1000, 60, seed=level)
    gen = torch.Generator(device="cpu").manual_seed(level)
    for t in range(20):
        acts = torch.randint(0, 5, (1000, f.n_agents), generator=gen, dtype=torch.int8).cuda()
        f.step(acts)
        i.step(acts)
        assert_twins(f, i, f"supplied actions, step {t}")


@pytest.mark.gpu
def test_layout_corpus(layouts):
    for name, text in layouts.items():
        import lle_b200

        try:
            lle_b200.Map(text)
        except Exception:
            continue
        run_twins([text], 64, 25, check_every=4, seed=11)


def _generated_maps():
    import json

    from _util import GOLDEN

    with open(os.path.join(GOLDEN, "generated_5x5.json")) as f:
        return json.load(f)["maps"]


@pytest.mark.gpu
def test_generated_maps_heterogeneous_batch():
    """1,024 generated 5x5 maps in one batch: config 3's thread-per-world path, maps blocked and interleaved."""
    maps = _generated_maps()
    run_twins(maps, 8192, 30, check_every=3, map_of_env=[m for m in range(1024) for _ in range(8)], seed=21)
    run_twins(maps, 4096, 20, check_every=4, map_of_env=[(e * 37) % 1024 for e in range(4096)], seed=22)


@pytest.mark.gpu
def test_levels_2_to_4_mixed():
    maps = [level_text(2), level_text(3), level_text(4)]
    run_twins(maps, 999, 50, check_every=2, map_of_env=[e % 3 for e in range(999)], seed=23)
    run_twins(maps, 960, 30, check_every=3, map_of_env=[e // 320 for e in range(960)], seed=24)


@pytest.mark.gpu
def test_large_map_chunked_general_path():
    """A 64x64 map with 8 agents: 80 KB per int8 row, streamed in chunks by the general kernel."""
    from _util import synthetic_map

    text = synthetic_map(64, 64, 8, 16, seed=5)
    run_twins([text], 96, 12, check_every=3, seed=25)
    run_twins([text], 40, 6, check_every=2, seed=26, obs_type="perspective")


@pytest.mark.gpu
def test_random_starts_and_randomize_lasers():
    from test_toml_maps import ANYWHERE, TEST_OK

    run_twins([TEST_OK], 300, 80, check_every=2, seed=81)
    run_twins([ANYWHERE], 128, 40, check_every=2, seed=84, auto_reset=False)
    run_twins([level_text(4), level_text(3)], 200, 80, check_every=2, seed=95, randomize_lasers=True,
              map_of_env=[e % 2 for e in range(200)])


@pytest.mark.gpu
def test_extras_pbrs_and_episode_stats():
    run_twins([level_text(6)], 500, 60, check_every=2, seed=31, extras="laser_subgoal", pbrs=dict(), episode_stats=True)
    run_twins([level_text(5)], 300, 40, check_every=2, seed=32, reward_dim=4, pbrs=dict(lasers_to_reward=[0]), walkable_lasers=False)


@pytest.mark.gpu
@pytest.mark.parametrize("obs_type", ["layered-padded-1", "layered-padded-2", "layered-padded-3", "flattened", "perspective"])
def test_observation_types(obs_type):
    for level in (3, 6):
        run_twins([level_text(level)], 300, 40, check_every=2, seed=41 + level, obs_type=obs_type)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 33, 100])
def test_ragged_sizes_and_no_auto_reset(n):
    for level in (1, 5, 6):
        run_twins([level_text(level)], n, 40, seed=50 + n)
        f, i = run_twins([level_text(level)], n, 30, check_every=3, seed=60 + n, auto_reset=False)
        f.reset()
        i.reset()
        assert_twins(f, i, "explicit reset")


@pytest.mark.gpu
def test_rollout():
    for level, n in ((6, 4096), (1, 2000)):
        f, i = twins([level_text(level)], n, seed=70)
        for k in (1, 7, 33):
            f.rollout(k)
            i.rollout(k)
            assert_twins(f, i, f"rollout({k})")
    maps = _generated_maps()
    f, i = twins(maps, 4096, map_of_env=[e // 4 for e in range(4096)], seed=71)
    f.rollout(25)
    i.rollout(25)
    assert_twins(f, i, "rollout on generated maps")


@pytest.mark.gpu
@pytest.mark.parametrize("level,n,n_parts", [(6, 4096, 8), (3, 1000, 3), (1, 333, 5)])
def test_parts_loop(level, n, n_parts):
    """A closed loop over parts: the host reward / done of every part at every step are the same for the twins.  (Parts are cut
    over each vec's own tickets, whose size depends on the row bytes, so the twins' part ranges may differ: the host buffers are
    compared whole, once every part of a step has been waited for.)"""
    f, i = twins([level_text(level)], n, seed=80 + level)
    steps = 12
    bufs = {}
    for name, vec in (("f", f), ("i", i)):
        bufs[name] = (torch.zeros((n, vec.n_agents), dtype=torch.int8).pin_memory(),
                      torch.zeros((n, vec.reward_dim), dtype=torch.float32).pin_memory(), torch.zeros(n, dtype=torch.uint8).pin_memory())
    gen = torch.Generator().manual_seed(level)
    plan = [torch.randint(0, 5, (n, f.n_agents), generator=gen, dtype=torch.int8) for _ in range(steps)]
    seen = {"f": [], "i": []}
    for name, vec in (("f", f), ("i", i)):
        acts, rew, done = bufs[name]
        with vec.parts_loop(n_parts, acts, rew, done) as loop:
            for step in range(steps):
                loop.launch()
                for k in range(loop.n_parts):
                    acts[loop.slice(k)] = plan[step][loop.slice(k)]
                    loop.feed(k)
                for k in range(loop.n_parts):
                    loop.wait(k)
                seen[name].append((rew.clone(), done.clone()))
    for step, ((r1, d1), (r2, d2)) in enumerate(zip(seen["f"], seen["i"], strict=True)):
        assert torch.equal(r1, r2) and torch.equal(d1, d2), step
    assert_twins(f, i, "after the parts loop")


@pytest.mark.gpu
def test_step_host_and_pipeline():
    n = 2048
    f, i = twins([level_text(6)], n, seed=90)
    gen = torch.Generator().manual_seed(90)
    out = {k: (torch.zeros((n, 1), dtype=torch.float32), torch.zeros(n, dtype=torch.uint8)) for k in "fi"}
    for t in range(10):  # pageable buffers: staged copies
        acts = torch.randint(0, 5, (n, 4), generator=gen, dtype=torch.int8)
        f.step_host(acts, *out["f"])
        i.step_host(acts, *out["i"])
        assert torch.equal(out["f"][0], out["i"][0]) and torch.equal(out["f"][1], out["i"][1])
        assert_twins(f, i, f"step_host {t}")
    pinned = {k: (torch.zeros((n, 4), dtype=torch.int8).pin_memory(), torch.zeros((n, 1), dtype=torch.float32).pin_memory(),
                  torch.zeros(n, dtype=torch.uint8).pin_memory()) for k in "fi"}
    for t in range(10):  # pinned buffers: submit / wait with two steps in flight
        acts = torch.randint(0, 5, (n, 4), generator=gen, dtype=torch.int8)
        for k, vec in (("f", f), ("i", i)):
            a, r, d = pinned[k]
            a.copy_(acts)
            vec.submit_host(a, r, d)
            vec.wait_host()
        assert torch.equal(pinned["f"][1], pinned["i"][1]) and torch.equal(pinned["f"][2], pinned["i"][2])
        assert_twins(f, i, f"pipeline {t}")
    for k, vec in (("f", f), ("i", i)):  # device sampling, several outstanding
        a, r, d = pinned[k]
        for _ in range(3):
            vec.submit_host(None, r, d)
        while vec.wait_host():
            pass
    assert_twins(f, i, "pipelined device sampling")


@pytest.mark.gpu
def test_mutators_reset_set_state_and_checkpoint():
    maps = [level_text(4), level_text(3), level_text(4)]
    moe = [e % 3 for e in range(300)]
    for kw in (dict(), dict(obs_type="perspective", auto_reset=False)):
        f, i = twins(maps, 300, map_of_env=moe, seed=100, **kw)
        for t in range(20):
            f.step(None); i.step(None)
        mask = (torch.arange(300) % 4 == 1).to(torch.uint8)
        f.reset(mask); i.reset(mask)
        assert_twins(f, i, "masked reset")
        for vec in (f, i):
            vec.set_source(1, enabled=False, map_index=0)
            vec.set_source(0, agent_id=1, map_index=1)
            vec.refresh()
        assert_twins(f, i, "set_source + refresh")
        for vec in (f, i):
            vec.collect_gem(0, map_index=2)
            vec.refresh()
        assert_twins(f, i, "collect_gem + refresh")
        for vec in (f, i):
            vec.set_exits([(11, 0), (10, 3), (5, 5)], map_index=1)
            vec.reset()
        assert_twins(f, i, "set_exits + reset")
        for t in range(30):
            f.step(None); i.step(None)
            assert_twins(f, i, f"step {t} after the mutators")
        pos = f.state[:, :4].reshape(300, 2, 2).to(torch.int32)
        pos[::5] = torch.flip(pos[::5], dims=(1,))
        gems = torch.zeros((300, 1), dtype=torch.uint8, device=f.device)
        alive = torch.ones((300, 2), dtype=torch.uint8, device=f.device)
        f.set_state(pos, gems, alive); i.set_state(pos, gems, alive)
        assert_twins(f, i, "set_state")
        ck_f, ck_i = f.checkpoint(), i.checkpoint()
        for t in range(15):
            f.step(None); i.step(None)
        f.restore(ck_f); i.restore(ck_i)
        assert_twins(f, i, "restore")
        for t in range(15):
            f.step(None); i.step(None)
        assert_twins(f, i, "after restore")


@pytest.mark.gpu
def test_state_type_fetch_and_dlpack():
    """state_type keeps its state observation in float32 (and equal); lle_vec_fetch(LLE_BUF_OBS) returns int8 bytes; DLPack
    exports the int8 tensor."""
    import lle_b200

    N = _native()
    f, i = run_twins([level_text(6)], 256, 20, check_every=5, seed=110, state_type="layered")
    assert i.state_obs.dtype == torch.float32 and torch.equal(i.state_of_type, f.state_of_type)
    b = N.VecBuffers()
    N.check(N.lib().lle_vec_get_buffers(i._h, C.byref(b)))
    assert b.obs_dtype == N.DTYPE_I8 and b.obs is None and b.obs_i8 and b.obs_stride % 16 == 0 and b.state_obs
    fb = N.VecBuffers()
    N.check(N.lib().lle_vec_get_buffers(f._h, C.byref(fb)))
    assert fb.obs_dtype == N.DTYPE_F32 and fb.obs and fb.obs_i8 is None
    n = 256 * b.obs_stride
    host = (C.c_int8 * n)()
    N.check(N.lib().lle_vec_fetch(i._h, 0, 0, n, host, None))
    rows = np.frombuffer(host, dtype=np.int8).reshape(256, b.obs_stride)
    assert np.array_equal(rows[:, :1872].reshape(256, 12, 12, 13), i.obs.cpu().numpy())
    assert not rows[:, 1872:].any()  # the pad bytes of a row stay zero
    assert N.lib().lle_vec_fetch(i._h, 0, 0, n + 1, host, None) == 201  # sized by element: one byte past the buffer
    env = lle_b200.level(6).n_envs(128).seed(5).obs_dtype(torch.int8).build()
    env.reset()
    t = torch.from_dlpack(env.dlpack("obs"))
    assert t.dtype == torch.int8 and t.data_ptr() == env.obs.data_ptr() and torch.equal(t, env.obs)
    assert torch.equal(env.obs.to(torch.bfloat16).float(), env.obs.float())
    ref = lle_b200.level(6).n_envs(128).seed(5).build()
    ref.reset()
    assert torch.equal(env.obs.float(), ref.obs)


@pytest.mark.gpu
def test_full_size_level6_and_config3():
    """Level 6 x 65,536 (the headline workload) and config 3 (1,024 maps x 1,024) for a few dozen steps."""
    f, i = run_twins([level_text(6)], 65536, 30, check_every=3, seed=2026)
    del f, i
    torch.cuda.empty_cache()
    maps = _generated_maps()
    moe = (np.arange(1 << 20) // 1024 % 1024).astype(np.int32)
    run_twins(maps, 1 << 20, 24, check_every=4, map_of_env=moe, seed=2026)


@pytest.mark.gpu
def test_env_vectors_through_an_int8_vec():
    """The reference's own recorded observations (tests/golden/env_vectors.npz) through a one-env int8 VecWorld: reset, step and
    set_state, obs.float() equal to the recorded observation after every operation."""
    import lle_b200
    from test_env_vectors import CONFIG_KW, cases, data

    z, _ = data()
    n_checked = 0
    for entry in cases():
        for obs_type in ("layered", "flattened", "layered-padded-1", "layered-padded-2", "layered-padded-3", "perspective"):
            key = f"{entry['key']}|obs|{obs_type}"
            if key not in z:
                continue
            want = z[key]
            ckw = CONFIG_KW[entry["config"]]
            kw = dict(reward_dim=4 if ckw.get("multi_objective") else 1, walkable_lasers=ckw.get("walkable_lasers", True),
                      extras=ckw.get("extras"), pbrs=ckw.get("pbrs"), auto_reset=False)
            try:
                vec = lle_b200.VecWorld(entry["text"], 1, obs_type=obs_type, obs_dtype=torch.int8, **kw)
            except IndexError:
                continue
            if vec.obs_invalid:
                continue
            tiled = entry["obs_tiled"][obs_type]
            for row, op in enumerate(entry["script"]):
                if op["op"] == "reset":
                    vec.reset()
                elif op["op"] == "set_state":
                    pos, gems, alive = op["set_state"]
                    vec.set_state(torch.tensor([pos], dtype=torch.int32), torch.tensor([gems], dtype=torch.uint8).reshape(1, -1),
                                  torch.tensor([alive], dtype=torch.uint8))
                else:
                    vec.step(torch.tensor([op["actions"]], dtype=torch.int8))
                torch.cuda.synchronize()
                got = (vec.obs[0] if tiled else vec.obs_per_agent[0]).float().cpu().numpy()
                assert np.array_equal(got, want[row].astype(np.float32)), f"{entry['key']} [{obs_type}] op {row} ({op['op']})"
                n_checked += 1
    assert n_checked > 1000
