"""Cost of the device expert (lle_vec_expert_build / lle_vec_expert_act): table builds, queries, and an expert-driven rollout.

  build   VecWorld.build_expert() on config 3's 1,024 generated 5x5 maps, on each of levels 1-4 alone, and on 1,024 generated 8x7
          three-agent maps (edge starts, opposite exits, 2 cross-agent lasers, wall shapes, 3 gems): a host clock around the
          synchronous call (upload, forward depths, backward levels, read-back), best of --repeats.
  act     VecWorld.expert_actions() on config 3 (2^20 worlds: 1,024 maps x 1,024) and on level 3 x 65,536: CUDA events around
          --iters back-to-back queries.
  loop    microseconds per step of `step(expert_actions()[0])` against device-sampled `step(None)` on the same vec, --iters steps
          each, CUDA events.
The card's name and power limit are read in the same run.  One JSON line per measurement goes to stdout and to --out.

    python tools/expert_bench.py --out profiles/expert_r03.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def main():
    import torch

    import lle_b200
    from lle_b200.generator import WorldGenerator
    from lle_b200.workloads import generated_maps

    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--maps-8x7", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "expert_bench measures the device expert: it needs a CUDA device"
    info = card()
    lines = []

    def emit(**kw):
        line = dict(**kw, **info)
        print(json.dumps(line), flush=True)
        lines.append(line)

    def vec_of(maps, n_envs, **kw):
        return lle_b200.VecWorld(maps, n_envs, map_of_env=[e % len(maps) for e in range(n_envs)], device=0, **kw)

    cfg3 = generated_maps(1024)
    g = WorldGenerator(width=8, height=7, n_agents=3, starts="edge", exits="opposite", n_lasers=2, laser_placement="cross-agent", n_walls=5,
                       walls_style="shapes", n_gems=3, batch=8192)
    gen8x7 = list(g.generate_n(args.maps_8x7, seed=21, distinct=True))
    builds = [("config3_5x5_2agents", cfg3)] + [(f"level{n}", [n]) for n in (1, 2, 3, 4)] + [("gen_8x7_3agents", gen8x7)]
    for name, maps in builds:
        vec = vec_of(maps, len(maps))
        times = []
        for _ in range(args.repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_states = vec.build_expert()
            times.append(time.perf_counter() - t0)
        dist = [vec.expert_table(m)[0] for m in range(len(maps))]
        reset = vec.expert_actions()[1].cpu().numpy()
        emit(kind="build", set=name, n_maps=len(maps), states=int(n_states.sum()), max_dist=int(max(d.max() for d in dist)),
             solvable=int((reset >= 0).sum()), seconds_best=min(times), seconds_all=times, states_per_s=float(n_states.sum()) / min(times))
        del vec

    def events(fn, iters):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / iters  # us per iteration

    for name, maps, n_envs in (("config3_5x5_2agents", cfg3, 1 << 20), ("level3", [3], 65536)):
        vec = vec_of(maps, n_envs)
        vec.build_expert()
        act, dist = vec.expert_actions()
        emit(kind="act", set=name, n_envs=n_envs, us_per_call=events(lambda: vec.expert_actions(act, dist), args.iters))

        def expert_step():
            vec.expert_actions(act, dist)
            vec.step(act)

        sampled = events(lambda: vec.step(None), args.iters)
        expert = events(expert_step, args.iters)
        emit(kind="loop", set=name, n_envs=n_envs, us_per_step_expert=expert, us_per_step_sampled=sampled)
        del vec
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
