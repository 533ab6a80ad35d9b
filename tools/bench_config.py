"""Device-timed throughput + HBM roofline of one BASELINE.json workload (lle_b200/workloads.py); bench.py reports all of them
in its `configs` key, this is the single-config tool for sweeps and profiler captures.
    python tools/bench_config.py --config 1|2|3|4|5 [--envs N] [--steps K] [--warmup W] [--obs-type T] [--obs-dtype float32|int8]
One JSON line.  Tuning knobs are read by the library from the environment (LLE_B200_*: see lle_b200/csrc/vec_world.cu)."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from bench import measured_peak
from lle_b200 import workloads

ap = argparse.ArgumentParser()
ap.add_argument("--config", type=int, required=True)
ap.add_argument("--envs", type=int, default=0)
ap.add_argument("--steps", type=int, default=0)
ap.add_argument("--warmup", type=int, default=20)
ap.add_argument("--obs-type", default="layered")
ap.add_argument("--obs-dtype", default="float32", choices=["float32", "int8"])
ap.add_argument("--repeat", type=int, default=1)
args = ap.parse_args()
steps = args.steps or {1: 4000, 2: 2000, 3: 500, 4: 200, 5: 30}[args.config]
kw = {} if args.obs_type == "layered" else {"obs_type": args.obs_type}
if args.obs_dtype != "float32":
    kw["obs_dtype"] = args.obs_dtype
wl = workloads.build(args.config, args.envs or None, **kw)
ms = min(wl.measure(steps, args.warmup) for _ in range(args.repeat))
peak, src = measured_peak()
ach = wl.algorithmic_bytes() / (ms / 1e3) / 1e9
knobs = {k: v for k, v in os.environ.items() if k.startswith("LLE_B200_")}
print(json.dumps({"config": args.config, "workload": wl.description, "obs_type": args.obs_type, "obs_dtype": args.obs_dtype, "envs": wl.n_envs, "steps": steps,
                  "ms_per_step": ms, "env_steps_per_s": wl.n_envs / (ms / 1e3), "agent_env_steps_per_s": wl.agent_envs / (ms / 1e3),
                  "algorithmic_bytes_per_step": wl.algorithmic_bytes(), "knobs": knobs,
                  "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": src}}))
