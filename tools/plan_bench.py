"""Throughput of the device planner (lle_plan): maps per second and expanded states per second.

Two sets: the 1,024 generated 5x5 maps of BASELINE config 3 (2 agents, 2 lasers; claim tables in shared memory) and a set of
generated 8x7 maps with 3 agents (edge starts, opposite exits, 2 cross-agent lasers, wall shapes, 3 gems; claim tables in
global memory).  Each lle_plan call is timed with CUDA events on the current stream around the synchronous call (upload, search,
read-back); the card's name and power limit are read in the same run.  One JSON line per set goes to stdout and to --out.

    python tools/plan_bench.py --out profiles/plan_r03.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def main():
    import numpy as np
    import torch

    from lle_b200.generator import WorldGenerator
    from lle_b200.planner import plan
    from lle_b200.vec_world import Map
    from lle_b200.workloads import generated_maps

    ap = argparse.ArgumentParser()
    ap.add_argument("--max-steps", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--maps-8x7", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "plan_bench measures the device planner: it needs a CUDA device"
    info = card()
    sets = {"config3_5x5_2agents": generated_maps(1024)}
    g = WorldGenerator(width=8, height=7, n_agents=3, starts="edge", exits="opposite", n_lasers=2, laser_placement="cross-agent", n_walls=5,
                       walls_style="shapes", n_gems=3, batch=8192)
    sets["gen_8x7_3agents"] = list(g.generate_n(args.maps_8x7, seed=21, distinct=True))
    lines = []
    for name, texts in sets.items():
        maps = [Map(t) for t in texts]
        plan(maps, max_steps=args.max_steps)  # warm-up: module load, first allocations
        times = []
        for _ in range(args.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            res = plan(maps, max_steps=args.max_steps)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
        best = min(times)
        states = int(res.n_states.sum())
        line = dict(set=name, n_maps=len(maps), max_steps=args.max_steps, solvable=int((res.length >= 0).sum()),
                    mean_length=float(res.length[res.length > 0].mean()) if (res.length > 0).any() else None,
                    states=states, seconds_best=best, seconds_all=times, maps_per_s=len(maps) / best, states_per_s=states / best, **info)
        print(json.dumps(line))
        lines.append(line)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
