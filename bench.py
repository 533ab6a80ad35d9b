#!/usr/bin/env python
"""bench.py — env-steps/s of the batched `World` step with layered observations (BASELINE.json metric).

A "step" is one lockstep step of the hot path over one batch: 65,536 x `World.level(6)` (4 agents, 3 laser
sources, 4 gems) per GPU with device-sampled (Philox) random actions, auto-reset, and every per-step output
of `LLE.step` written: layered observation, state vector, availability mask, reward, done, events.

  python bench.py [--gpus N] [--steps K] [--warmup W]             our arm (CUDA, through the C ABI)
  python bench.py --impl reference [--gpus N] [--steps K] ...     the CPU arm: the oracle's restatement of the
        reference engine on all host cores (the Rust crate cannot be built in this image: no cargo/rustc)

For N > 1 launch with torchrun (one rank per GPU); envs are range-sharded over ranks (weak scaling, no
collective on the step path; NCCL carries only the reductions of the timings and of three counters).
Prints ONE JSON line on rank 0.  Keys beyond the contract:
  configs    the other BASELINE.json workloads (1, 3, 4, 5 of SURVEY §8d) at their stated per-GPU sizes, bounded steps
  e2e        value = closed loop (the host reads step t's results before it chooses step t+1's actions), eight sub-batches
             in flight; pipelined_value = open loop, 8 recorded steps in flight; sync_value = one blocking call per step
  ranks      per-rank ms per step of the headline window (min / max / all)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LEVEL = 6
ENVS_PER_GPU = 65536
SEED = 2026
METRIC = "env-steps/s (layered obs, device-timed)"
UNIT = "env-steps/s"
# bounded timed steps of the other configs: (steps, warm-up) — about 0.1-0.2 s of device time each
CONFIG_STEPS = {1: (512, 16), 3: (96, 8), 4: (32, 4), 5: (8, 3)}
# steps from the reset at creation to the state the timed steps start from: an episode of level 6 under random actions lasts
# about 20 steps, so by then the batch has the mix of running and resetting envs of a long-running job
SETTLE_STEPS = 256
# --dump-outputs: at most this many bytes of float32 rows; above it, a fixed seeded sample of the envs is written
DUMP_BYTES = 64 << 20
DUMP_SEED = 7
OUTPUTS = ("obs", "state", "avail", "reward", "done", "events", "actions", "err")


def level_text(n: int) -> str:
    with open(os.path.join(ROOT, "lle_b200", "resources", "levels", f"lvl{n}")) as f:
        return f.read()


def measured_peak() -> tuple[float, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic() -> dict:
    """dram bytes per launch of the step kernel from the committed `ncu --set full` capture (profiles/traffic.json names the
    capture and the commit it was taken at; it is a profile reading, not something this run measures)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return {}


class ClockSampler:
    """`nvidia-smi -lms 20` in the background, its lines collected by a reader thread.  nvidia-smi needs 50-150 ms to print its first
    line and the timed window of the default run is 1.6 ms, so the sampler is started BEFORE the untimed preheat (the same
    kernel, back to back): the preheat runs until samples arrive, and the samples kept are those taken under that continuous
    load up to the end of the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.proc = None
        self.lines: list[str] = []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(device_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        try:
            for line in self.proc.stdout:
                self.lines.append(line)
        except Exception:
            pass

    def n_samples(self) -> int:
        return len(self.lines)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        lines = list(self.lines)  # what was sampled up to now: under load
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(power), "samples": len(sm),
                "window": "preheat + warm-up + timed steps + rollout: the step kernel back to back", "reasons": sorted(reasons)}


def cpu_baseline(sample_seconds: float = 12.0, n_envs: int = 4096, threads: int = 0) -> dict:
    """The oracle (CPU restatement of the reference engine + layered observation) on the host cores:
    one World per thread at a time, all outputs written each step, Philox actions, auto-reset."""
    from oracle import lle_oracle as lo

    vec = lo.OracleVec([level_text(LEVEL)], None, n_envs, seed=SEED, auto_reset=True)
    secs, used = vec.rollout(8, threads)  # warm-up + calibration
    rate = n_envs * 8 / max(secs, 1e-9)
    steps = max(8, int(sample_seconds * rate / n_envs))
    secs, used = vec.rollout(steps, threads)
    value = n_envs * steps / secs
    return {"value": value, "unit": UNIT, "cores": used, "kind": "port",
            "sample": f"{n_envs} envs x {steps} steps of level {LEVEL} in {secs:.2f} s, C++ restatement of the reference engine "
                      f"(Rust toolchain unavailable) with the reference's own allocation pattern (a fresh observation array and "
                      f"laser / gem lists per step, as python/lle/observations.py:254-266 does), one World per thread, {used} threads, "
                      f"layered obs + state + avail written each step",
            "seconds": secs}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each "step" of this arm is a bounded sample of the same workload; K samples are timed
    k = max(1, min(args.steps, 5))
    w = 1 if args.warmup > 0 else 0
    t0 = time.time()
    for _ in range(w):
        cpu_baseline(sample_seconds=2.0)
    res = [cpu_baseline(sample_seconds=6.0) for _ in range(k)]
    value = statistics.mean(r["value"] for r in res)
    ms = 1000.0 * statistics.mean(r["seconds"] for r in res)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": k, "warmup": w,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u64 bitmasks, f32 encodings",
        "data": "synthetic",
        "config": {"workload": f"World.level({LEVEL}) 4 agents, 3 laser sources (BASELINE.json says 4), layered observations, "
                               f"random Philox actions, auto-reset; CPU arm: bounded samples of 4096 envs"},
        "cpu_baseline": {**{k2: v for k2, v in res[-1].items() if k2 != "seconds"}, "value": value},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.time() - t0,
    }
    print(json.dumps(line))


def output_rows(vec, begin: int, n_total: int) -> dict:
    """This rank's rows of what the last step handed its caller (the per-env output tensors of VecWorld), as float32 numpy arrays,
    plus their global env ids as float64.  All envs when their rows fit in DUMP_BYTES, else a fixed seeded sample of the global
    env ids, the same for every rank count."""
    import numpy as np
    import torch

    tensors = {name: getattr(vec, name) for name in OUTPUTS}
    row_bytes = 8 + sum(4 * t[0].numel() for t in tensors.values())
    n_keep = min(n_total, DUMP_BYTES // row_bytes)
    ids = np.arange(n_total) if n_keep == n_total else np.sort(np.random.default_rng(DUMP_SEED).choice(n_total, n_keep, replace=False))
    ids = ids[(ids >= begin) & (ids < begin + vec.n_envs)]
    rows = torch.from_numpy(ids - begin).to(vec.device)
    out = {name: t.index_select(0, rows).float().cpu().numpy() for name, t in tensors.items()}
    out["env_id"] = ids.astype(np.float64)
    return out


def pin_rank_to_cores(local_rank: int, local_world: int) -> list[int] | None:
    """One disjoint slice of the host cores per rank: the step loop of a rank is host-driven (one launch per step), and
    eight Python processes migrating over the same cores show up as per-rank jitter in the MAX-over-ranks timing."""
    if local_world <= 1:
        return None
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // local_world)
        mine = cores[local_rank * per:(local_rank + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:
        return None


def run_ours(args) -> None:
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = pin_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", str(world_size))))

    import numpy as np
    import torch
    import torch.distributed as dist

    import lle_b200
    from lle_b200 import workloads

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world_size > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner (and any warning) to stdout unless told otherwise
        # (NCCL_DEBUG_FILE is honoured only above the VERSION level)
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    from lle_b200.sharding import reduce_stats, shard_range

    begin, end = shard_range(args.envs * world_size, rank, world_size)  # weak scaling: args.envs worlds per GPU
    n_envs = end - begin
    vec = lle_b200.VecWorld(lle_b200.Map(level=LEVEL), n_envs, device=dev, seed=SEED, env_id_base=begin, auto_reset=True)
    A, R = vec.n_agents, vec.reward_dim
    K, Wm = args.steps, max(args.warmup, 3)

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        if world_size > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def gather(x: float) -> list[float]:
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        if world_size == 1:
            return [float(tt.item())]
        out = [torch.zeros_like(tt) for _ in range(world_size)]
        dist.all_gather(out, tt)
        return [float(o.item()) for o in out]

    # ---------------- device-resident arm: K fused steps back to back, no host sync inside.
    # Untimed preheat first (not counted as warm-up steps): a fresh process finds the GPU at idle clocks, and W = 5 steps are
    # 0.4 ms of work; the timed window should see the clocks a running job sees.  The preheat runs for a wall-clock time, so
    # its number of steps varies: the state after SETTLE_STEPS is restored after it, and every run with the same arguments
    # times the same steps on the same inputs.
    for _ in range(SETTLE_STEPS):
        vec.step(None)
    settled = vec.checkpoint()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t0 = time.perf_counter()
    preheat = 0
    while True:
        elapsed = time.perf_counter() - t0
        # the GPUs stay loaded until rank 0's nvidia-smi has delivered a few samples (bounded: 2 s); every rank stops together
        more = 1.0 if (elapsed < args.preheat_ms / 1e3 or (sampler is not None and sampler.proc is not None and sampler.n_samples() < 3 and elapsed < 2.0)) else 0.0
        if reduce_max(more) == 0.0:
            break
        for _ in range(64):
            vec.step(None)
        preheat += 64
        torch.cuda.synchronize()
    vec.restore(settled)
    del settled
    for _ in range(Wm):
        vec.step(None)
    barrier()
    launches0 = vec.launch_count
    vec.timing_begin()
    for _ in range(K):
        vec.step(None)
    ms_total, timed_launches = vec.timing_end()
    barrier()
    launches = vec.launch_count - launches0
    dumped = None
    if args.dump_outputs:
        dumped = output_rows(vec, begin, args.envs * world_size)
        if world_size > 1:
            parts = [None] * world_size
            dist.all_gather_object(parts, dumped)
            dumped = {name: np.concatenate([p[name] for p in parts]) for name in dumped}
    per_rank = gather(ms_total / K)
    ms_max = max(per_rank) * K
    value = world_size * n_envs * K / (ms_max / 1e3)

    # ---------------- the same K steps as lle_vec_rollout launches (up to 128 steps per launch, bit-identical results):
    # reported beside the headline as "rollout", not as the headline (the contract's step = one launch)
    RL = min(128, max(K, 1))
    n_roll = max(1, K // RL)
    vec.rollout(RL)
    barrier()
    vec.timing_begin()
    for _ in range(n_roll):
        vec.rollout(RL)
    ms_roll, roll_launches = vec.timing_end()
    barrier()
    clocks = sampler.stop() if sampler else None
    ms_roll_max = reduce_max(ms_roll)
    rollout_value = world_size * n_envs * n_roll * RL / (ms_roll_max / 1e3)

    # ---------------- end-to-end arms: host actions in (pinned, H2D), reward + done out (D2H) every step
    Ke = max(1, min(K, args.e2e_steps))
    T0 = 10_000_000
    vec.reset()
    vec.step_count = T0
    rec_act = torch.empty((Ke, n_envs, A), dtype=torch.int8).pin_memory()
    rec_done = torch.empty((Ke, n_envs), dtype=torch.uint8).pin_memory()
    for s in range(Ke):  # record a valid action stream (and the done flags it leads to) on the device, then drive from the host
        vec.step(None)
        rec_act[s].copy_(vec.actions, non_blocking=True)
        rec_done[s].copy_(vec.done, non_blocking=True)
    torch.cuda.synchronize()
    stay = torch.full((n_envs, A), 4, dtype=torch.int8).pin_memory()
    D = max(1, min(8, args.e2e_depth))
    reward_h = [torch.empty((n_envs, R), dtype=torch.float32).pin_memory() for _ in range(D)]
    done_h = [torch.empty((n_envs,), dtype=torch.uint8).pin_memory() for _ in range(D)]

    done_np0, rec_done_np0 = done_h[0].numpy(), rec_done.numpy()

    def restart(v, t=T0):
        v.reset()
        v.step_count = t

    def e2e_sync() -> float:
        """lle_vec_step_host, closed loop: H2D, step, D2H, stream sync — one blocking call per step; the actions of step s are
        chosen only after every done flag of step s-1 has been read (they match the recording, so the recorded actions stay
        valid; otherwise everyone would STAY)."""
        restart(vec)
        barrier()
        t0 = time.perf_counter()
        acts = rec_act[0]
        for s in range(Ke):
            vec.step_host(acts, reward_h[0], done_h[0])
            if s + 1 < Ke:
                acts = rec_act[s + 1] if np.array_equal(done_np0, rec_done_np0[s]) else stay
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def e2e_pipelined() -> float:
        """lle_vec_pipeline_submit / _wait with D steps in flight (OPEN loop: step s+D is submitted before step s is read —
        what a replay buffer or a scripted evaluation can do, not an acting agent)."""
        restart(vec)
        barrier()
        t0 = time.perf_counter()
        n_done = 0
        for s in range(Ke):
            if s >= D:
                vec.wait_host()
                n_done += int(done_h[(s - D) % D][0])  # the host consumes the result of step s - D
            vec.submit_host(rec_act[s], reward_h[s % D], done_h[s % D])
        for s in range(max(Ke - D, 0), Ke):
            vec.wait_host()
            n_done += int(done_h[s % D][0])
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    # Closed loop over parts of the batch (lle_vec_parts_*): every step is ONE launch over the whole batch; the step kernel waits
    # part by part for the actions the host releases, and publishes each part's reward / done to pinned host memory as the part
    # completes.  The host reads every done flag of a part's step s before it chooses and releases the part's actions of step
    # s + 1, while the other parts (and the next launch) keep the device busy.
    P = max(1, args.e2e_parts)
    act_p = torch.empty((n_envs, A), dtype=torch.int8).pin_memory()
    rew_p = torch.empty((n_envs, R), dtype=torch.float32).pin_memory()
    done_p = torch.empty((n_envs,), dtype=torch.uint8).pin_memory()
    act_np, done_np, rec_act_np, rec_done_np = act_p.numpy(), done_p.numpy(), rec_act.numpy(), rec_done.numpy()
    mismatches = [0]

    def e2e_closed_loop() -> float:
        restart(vec)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        with vec.parts_loop(P, act_p, rew_p, done_p, after_current_stream=False) as loop:
            slices = [loop.slice(k) for k in range(loop.n_parts)]
            loop.launch()
            for k, sl in enumerate(slices):
                act_np[sl] = rec_act_np[0][sl]
                loop.feed(k)
            if Ke > 1:
                loop.launch()
            for s in range(Ke):
                for k, sl in enumerate(slices):
                    loop.wait(k)  # reward / done of this part's step s are in host memory
                    ok = np.array_equal(done_np[sl], rec_done_np[s][sl])  # the policy reads every result byte (a memcmp)
                    if not ok:
                        mismatches[0] += 1
                    if s + 1 < Ke:
                        act_np[sl] = rec_act_np[s + 1][sl] if ok else 4  # the recorded action stays valid; otherwise everybody STAYs
                        loop.feed(k)
                if s + 2 < Ke:
                    loop.launch()
        return time.perf_counter() - t0

    for s in range(min(3, Ke)):
        vec.step_host(rec_act[s], reward_h[0], done_h[0])
    e2e_pipelined()  # warm-up (creates the pipeline's streams and ring)
    # Under a profiler that serialises launches (ncu makes a launch call return when the kernel has finished) a parts-loop step would
    # wait on the device for actions that its own host thread releases after the launch call: the closed loop is skipped there.
    profiled = args.no_closed_loop or any(k in os.environ for k in ("CUDA_INJECTION64_PATH", "NV_COMPUTE_PROFILER_PERFWORKS_DIR"))
    if not profiled:
        e2e_closed_loop()
    e2e_sync_value = world_size * n_envs * Ke / reduce_max(e2e_sync())
    e2e_pipe_value = world_size * n_envs * Ke / reduce_max(e2e_pipelined())
    assert int(vec.err.sum()) == 0, "replayed actions must be valid"
    mismatches[0] = 0
    e2e_closed_value = None
    if not profiled:
        e2e_closed_value = world_size * n_envs * Ke / reduce_max(e2e_closed_loop())
        assert mismatches[0] == 0 and int(vec.err.sum()) == 0, "the closed loop left the recorded trajectory"

    # the same closed loop driven by a COMPILED host on the C ABI alone (examples/c_closed_loop.c): what the reference's Rust side
    # would see through FFI.  One process per rank on the rank's own device, all ranks at once.
    compiled = None
    exe = os.path.join(ROOT, "examples", "_build", "c_closed_loop")
    if os.path.exists(exe) and not args.no_compiled_host and not profiled:
        barrier()
        try:
            res = subprocess.run([exe, str(local_rank), str(n_envs), str(Ke), f"s{P}", str(P)], capture_output=True, text=True, timeout=300)
            got = json.loads(res.stdout.strip().splitlines()[-1]) if res.returncode == 0 else None
        except Exception:
            got = None
        us = reduce_max(got["parts"][f"s{P}"]["us_per_step"] if got else float("inf"))
        us_sub = reduce_max(got["parts"][str(P)]["us_per_step"] if got else float("inf"))
        if us != float("inf"):
            compiled = {"value": world_size * n_envs / (us / 1e6), "us_per_step": us, "parts": P, "steps": Ke,
                        "sub_batch_vecs_value": world_size * n_envs / (us_sub / 1e6),
                        "host": "compiled C program on the C ABI alone (examples/c_closed_loop.c), one per rank"}

    # end-of-run stats reduction: the only collective on this path (NCCL all-reduce of a few counters)
    stats = reduce_stats(torch.stack([vec.done.sum().to(torch.int64), vec.reward.sum().to(torch.int64),
                                      torch.tensor(n_envs, dtype=torch.int64, device=dev)]))
    bytes_env = workloads.algorithmic_bytes(vec)
    obs_shape = [vec.n_channels, vec.height, vec.width]
    del vec
    torch.cuda.empty_cache()

    # ---------------- the other BASELINE.json workloads at their stated per-GPU sizes (bounded steps)
    peak, peak_src = measured_peak()
    configs = {}
    for cfg in ([] if args.no_configs else [1, 3, 4, 5]):
        n_cfg = workloads.DEFAULT_ENVS[cfg]
        free_b, _ = torch.cuda.mem_get_info(dev)
        if cfg == 5:
            per_env = 4 * 20 * 64 * 64 + 4096
            while n_cfg * per_env > 0.92 * free_b and n_cfg > 1024:
                n_cfg //= 2  # a GPU with less memory than a B200: say so in the line
        b0, _ = shard_range(n_cfg * world_size, rank, world_size)
        wl = workloads.build(cfg, n_cfg, device=dev, seed=SEED, env_id_base=b0)
        steps_c, warm_c = CONFIG_STEPS[cfg]
        barrier()
        ms_c = reduce_max(wl.measure(steps_c, warm_c))
        ach = wl.algorithmic_bytes() / (ms_c / 1e3) / 1e9
        errs = sum(int(p.err.sum()) for p in wl.parts)
        configs[str(cfg)] = {
            "workload": wl.description, "envs_per_gpu": wl.n_envs, "envs": wl.n_envs * world_size, "steps": steps_c, "warmup": warm_c,
            "ms_per_step": ms_c, "env_steps_per_s": world_size * wl.n_envs / (ms_c / 1e3),
            "agent_env_steps_per_s": world_size * wl.agent_envs / (ms_c / 1e3), "launches_per_step": len(wl.parts),
            "algorithmic_bytes_per_step_per_gpu": wl.algorithmic_bytes(), "env_errors": errs,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak},
        }
        del wl
        torch.cuda.empty_cache()

    if rank == 0:
        kernel_ms = ms_total / max(timed_launches, 1)
        achieved = bytes_env["total"] * n_envs / (kernel_ms / 1e3) / 1e9
        traffic = ncu_traffic()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": K, "warmup": Wm,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u64 bitmasks, f32 encodings", "data": "synthetic",
            "config": {
                "workload": f"World.level({LEVEL}) 4 agents, 3 laser sources (BASELINE.json says 4; the level file has 3), "
                            f"{n_envs} batched envs per GPU with layered observations (BASELINE.json configs[1])",
                "envs_per_gpu": n_envs, "agents": A, "obs_shape": obs_shape,
                "actions": "device Philox4x32-10, uniform over available",
                "auto_reset": True, "agent_env_steps_per_s": value * A,
                "l2": f"each step rewrites {n_envs * bytes_env['obs'] / 1e6:.0f} MB of observations per GPU (> 126 MB L2); no flush needed",
                "sharding": "contiguous env ranges per rank, no collective on the step path",
                "launch": "one fused kernel launch per step (programmatic dependent launch between steps); "
                          "lle_vec_rollout(K) runs K steps in one launch with identical results",
                "preheat": f"{preheat} untimed steps (~{args.preheat_ms:.0f} ms) before the {Wm} warm-up steps, so that the timed window "
                           f"runs at the clocks of a running job",
                "host_cores_of_rank0": cores,
            },
            "ranks": {"ms_per_step_min": min(per_rank), "ms_per_step_max": max(per_rank), "ms_per_step": per_rank},
            "clocks": clocks,
            "e2e": {"value": compiled["value"] if compiled else (e2e_closed_value if e2e_closed_value is not None else e2e_sync_value), "unit": UNIT, "h2d_bytes_per_step": n_envs * A,
                    "d2h_bytes_per_step": n_envs * (4 * R + 1), "steps": Ke, "closed_loop": True, "parts": P,
                    "host": compiled["host"] if compiled else ("python" if e2e_closed_value is not None else "python, one blocking call per step (closed loop over parts skipped: profiler or --no-closed-loop)"), "python_host_value": e2e_closed_value,
                    "pipelined_value": e2e_pipe_value, "pipeline_depth": D, "sync_value": e2e_sync_value,
                    "sub_batch_vecs_value": compiled["sub_batch_vecs_value"] if compiled else None,
                    "note": f"value: CLOSED loop through lle_vec_parts_* from a compiled host on the C ABI (the reference's host side is Rust; "
                            f"python_host_value is the same loop driven from Python): ONE launch per step of the whole batch, {P} parts; the host "
                            "reads every done flag of a part's step t from pinned memory before it writes and releases that part's actions of "
                            "step t+1 (the step kernel waits for them part by part on the device), while the other parts and the next launch "
                            "run; the kernel reads the actions from and writes reward+done to pinned host memory inside the timed region "
                            "(zero-copy, counted as h2d/d2h bytes). sub_batch_vecs_value: the same dependency with the batch cut into "
                            f"{P} vecs stepped through lle_vec_pipeline_submit/_wait (round 2's first design). sync_value: one blocking "
                            "lle_vec_step_host call per step on the whole batch. "
                            f"pipelined_value: OPEN loop, {D} recorded steps in flight (not what an acting agent can do). "
                            "Observations stay in HBM (zero-copy DLPack hand-off to a device policy)"},
            "gpu_launches": launches,
            "rollout": {"value": rollout_value, "unit": UNIT, "steps_per_launch": RL, "launches": int(roll_launches),
                        "ms_per_step": ms_roll_max / (n_roll * RL),
                        "note": "lle_vec_rollout: the same steps, many per launch, ordered by the per-ticket epoch flags; device-timed"},
            "configs": configs,
            "stats_allreduce": {"done_last_step": int(stats[0]), "reward_last_step": int(stats[1]), "envs_total": int(stats[2])},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic.get("dram_bytes_per_launch"), "traffic_source": traffic.get("source"),
                         "traffic_commit": traffic.get("commit"), "peak_source": peak_src,
                         "kernel": "lle_world_kernel<MODE_STEP, FAST>", "kernel_ms": kernel_ms,
                         "algorithmic_bytes_per_env_step": bytes_env, "algorithmic_bytes_per_launch": bytes_env["total"] * n_envs},
        }
        if world_size == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline()
            cb.pop("seconds", None)
            line["cpu_baseline"] = cb
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumped.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
        print(json.dumps(line))
    if world_size > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8192)
    ap.add_argument("--warmup", type=int, default=128)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU")
    ap.add_argument("--e2e-steps", type=int, default=2048)
    ap.add_argument("--e2e-depth", type=int, default=8, help="steps in flight in the open-loop pipelined arm (1..8)")
    ap.add_argument("--e2e-parts", type=int, default=8, help="sub-batches in flight in the closed-loop arm")
    ap.add_argument("--preheat-ms", type=float, default=250.0, help="untimed device work before the warm-up steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-compiled-host", action="store_true", help="skip the compiled-host closed loop of the e2e arm")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE workloads")
    ap.add_argument("--no-closed-loop", action="store_true", help="skip the closed loop over parts (implied under ncu, which serialises launches)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (float32; "
                    "env_id.npy: the envs the rows belong to, a fixed sample when all envs would exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
