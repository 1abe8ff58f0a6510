#!/usr/bin/env python
"""Headline benchmark: env-steps/s on 40x40 (81x81 block) mazes -- BASELINE.json configs[1].

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo, N=1 default
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # one rank per GPU
    python bench.py --impl reference ...                           # the reference's CPU path

Workload (per GPU): a pool of 1000 r-prim euclidean 81x81 mazes generated on the device
(Philox seed 1234), B envs = 1000 mazes x A agents, uniform random actions from a device-resident
tape, gymnasium next-step autoreset on.  One "step" = one maze_step launch over all B envs.
Prints ONE JSON line (rank 0).

    python bench.py --workload toroidal-regen     # configs[2]: toroidal 81x81, mixed generators, regenerate on every win
    python bench.py --workload curriculum-dq      # configs[3]: 21x21 -> 129x129 curriculum, double Q-learning on the device
    python bench.py --workload ddqn               # configs[4]: DDQN loop, 8192 envs per GPU, NCCL gradient all-reduce

(the other configs of BASELINE.json as one-line measurements of the same shape; the default is configs[1], the
configuration the headline metric is quoted on).

    python bench.py ... --dump-outputs DIR        # also write what the last timed step computed as DIR/<name>.npy

The inputs depend on the arguments only (seeded mazes and actions), so the dumps of two builds run with the same
arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG_DIR = os.path.join(ROOT, "maze-solving-agent-gymnasium_b200")
for p in (ROOT, PKG_DIR):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "env-steps/sec (40x40 mazes, whole job)"
UNIT = "env-steps/s"
SHAPE = (81, 81)
NUM_MAZES = 1000
ALGO_BYTES_PER_STEP = 58   # SURVEY.md section 8(d): action 1 + state 16 + tables 7 + outputs 34
DUMP_BYTES = 64 * 10**6


def workload_name(envs_per_gpu):
    return (f"configs[1]: {NUM_MAZES} constant-size 40x40 (81x81 block) r-prim euclidean mazes per GPU, "
            f"{envs_per_gpu} envs per GPU, uniform random actions, autoreset")


def workload_config(envs_per_gpu, world):
    """The `config` object of the line: identical for this repo's arm and the reference arm."""
    return {"workload": workload_name(envs_per_gpu), "envs_per_gpu": envs_per_gpu, "mazes_per_gpu": NUM_MAZES,
            "l2": "inputs larger than L2: per-step working set (~100 B x envs = 400 MB) and the 13 KB/env visit arrays exceed the 126 MB L2; no flush needed",
            "parallelism": f"env-index sharding over {world} GPU(s), no per-step collective"}


def pattern_peak():
    """The scattered read-modify-write micro-benchmark of this access pattern (tools/perf_scatter_rmw.py, committed
    summary in profiles/): what HBM3e + L2 give 'coalesced streams + one 2-byte RMW at a random 64-byte atom for 40 %
    of the envs' with no maze logic at all."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_scatter_rmw.json")))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "5"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_step_byte():
    """dram bytes per env-step of maze_step from the committed ncu summary, if there is one."""
    path = os.path.join(ROOT, "profiles", "step_kernel_ncu_summary.json")
    try:
        return json.load(open(path))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
def reference_mazes(n, seed=1234):
    """81x81 r-prim mazes for the CPU arms (oracle generator; the device generator is the product's)."""
    import random

    from oracle.generation import gen_maze
    rng = random.Random(seed)
    out = []
    for _ in range(n):
        start, goal, grid = gen_maze(SHAPE, "r-prim", rng)
        out.append(dict(grid=grid, start=start, goal=goal, toroidal=False))
    return out


def run_reference(args, rank):
    """The reference's own CPU implementation of the path (the oracle's A*-per-step port of
    gymnasium_env/envs/base_maze_env.py; the Python reference itself cannot travel to the GPU box),
    one worker process per host core, each 'step' a bounded sample."""
    if rank != 0:
        return None
    from oracle import ref_runtime
    from oracle.baseline import PersistentVector
    cores = os.cpu_count() or 1
    # baseline/_ref (a copy of the unmodified reference, tools/install_reference.py) present -> time the reference's own
    # SimpleMazeEnv; otherwise the oracle's port of it
    kind = "reference" if ref_runtime.available() and not os.environ.get("MAZE_REF_FORCE_PORT") else "port"
    mazes = reference_mazes(min(cores, 8) if kind == "port" else 1)
    vec = PersistentVector(mazes, cores, kind)
    # A 'step' is a fixed slice of wall time in which every worker steps its own env as fast as it can (free running:
    # the best this implementation can do on the box -- stepping the envs in lock step like gymnasium's
    # AsyncVectorEnv would wait for the slowest A* search every time and lands at about 40 % of this rate).  The slice
    # is sized so that warm-up + timed steps take about BUDGET_S in total, whatever K and W are.
    BUDGET_S = float(os.environ.get("MAZE_REF_BUDGET_S", "120"))   # (tests shrink it)
    per = max(0.02, BUDGET_S / max(1, args.steps + args.warmup))
    for _ in range(args.warmup):
        vec.run_for(per)
    steps, secs = 0, 0.0
    for _ in range(args.steps):
        r = vec.run_for(per)
        steps += r["steps"]; secs += r["seconds"]
    vec.close()
    value = steps / secs
    what = ("the unmodified reference's gymnasium_env.envs.simple_maze_env.SimpleMazeEnv((81, 81)) from baseline/_ref (gymnasium / pygame "
            "stubbed to no-ops: an upper bound on its speed) on its own r-prim maze" if kind == "reference" else
            "the oracle port (A* per step) of the reference env on an 81x81 r-prim maze")
    sample = (f"{args.steps} steps x {per * 1e3:.0f} ms x {cores} free-running worker processes ({steps} env-steps in {secs:.1f} s), each "
              f"worker stepping {what}, random actions, reset on done")
    return ({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.envs_per_gpu, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ------------------------------------------------------------------------------------------------
def pin_to_gpu_numa_node(index):
    """Run this rank on the CPUs next to its GPU, so that the pinned staging buffers of the e2e path
    are allocated on the GPU's NUMA node (8 ranks sharing one node's memory halve the copy rate)."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:      # CUDA_VISIBLE_DEVICES may renumber the devices: go through the UUID
            handle = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(index).uuid))
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
    except Exception as exc:   # not fatal: only the host-copy rate depends on it
        print(f"[bench] no CPU affinity for GPU {index}: {exc}", file=sys.stderr)


def measure_extras(mb, torch, device):
    """Secondary numbers of the same path, one GPU (rank 0), CUDA events: valid mazes generated/s
    (BASELINE.json's second metric), difficulty-metric throughput, the -v1 (window) step and the
    fused Q-learning rollout.  Each is a few hundred milliseconds."""
    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps

    out = {"per_gpu": True}
    M = 131072
    pool = mb.MazePool(M, SHAPE, device)
    gen = {}
    for algo in ("r-prim", "dfs", "prim&kill"):
        seed = [7]

        pool.generate(algorithms=algo, seed=6)        # writes the per-slot configuration once

        def go():
            seed[0] += 1
            pool.generate(seed=seed[0], configure=False)
        gen[algo] = M / timed(go, 3)
    out["mazes_per_s_81x81"] = gen
    seed = [100]

    def go6():
        seed[0] += 1
        pool.generate(ids=torch.arange(16384, device=device, dtype=torch.int32), algorithms="r-prim", seed=seed[0],
                      candidates=6, configure=False)
    pool.generate(algorithms="r-prim", seed=5)
    out["best_of_6_mazes_per_s_81x81"] = 16384 / timed(go6, 1)
    ids = torch.arange(32768, device=device, dtype=torch.int32)
    out["difficulty_mazes_per_s_81x81"] = 32768 / timed(lambda: pool.difficulty(ids), 2)
    del pool
    # -v1 observation: step + 15x15 window (2 700 B written per env-step)
    Bv = 262144
    venv = mb.MazeVectorEnv(Bv, shape=SHAPE, num_mazes=1000, enrich=True, seed=1234, on_win="next", stats=False, device=device)
    venv.reset()
    acts = torch.randint(0, 4, (Bv,), dtype=torch.uint8, device=device)
    t = timed(lambda: venv.step(acts), 100)
    out["v1_window_env_steps_per_s"] = Bv / t
    out["v1_window_write_GBps"] = Bv * 2700 / t / 1e9
    # DQN data path: step + bit-packed observation + replay push (245 B per transition), and batch sampling
    from maze_b200.dqn import DeviceReplay
    memory = DeviceReplay(venv, 1 << 20, seed=1)
    memory.observe()

    def step_push():
        venv.batch.step(acts, venv._mode)
        memory.push(acts)
    out["dqn_step_push_env_steps_per_s"] = Bv / timed(step_push, 100)
    out["dqn_replay_samples_per_s"] = 65536 / timed(lambda: memory.sample(65536), 20)
    del venv, memory
    # fused tabular Q-learning rollout (policy + step + update per env, 64 steps per launch)
    from maze_b200.agents import QAgent
    Bq = 1048576
    qenv = mb.MazeVectorEnv(Bq, shape=SHAPE, num_mazes=1000, seed=1234, on_win="next", stats=True, device=device,
                            visit_layout="tile")
    agent = QAgent(qenv, learning_rate=0.1, initial_epsilon=0.9, epsilon_decay=2000, final_epsilon=0.05,
                   discount_factor=0.7, eta=1e-3, envs_per_agent=Bq, capacity=1 << 24)
    qenv.reset()
    K = 64
    t = timed(lambda: agent.rollout(K), 3)
    agent.core.check_overflow()
    out["q_rollout_env_steps_per_s"] = Bq * K / t
    del qenv, agent
    # open-loop bursts: maze_step_many over a 64-step action tape, every per-step output written (bit-identical
    # to 64 maze_step launches); tiled visit layout.  Reported beside the headline, which is one launch per step.
    Bm = 4096000
    menv = mb.MazeVectorEnv(Bm, shape=SHAPE, num_mazes=1000, seed=1234, on_win="next", stats=False, device=device,
                            visit_layout="tile")
    menv.reset()
    tape = torch.randint(0, 4, (K, Bm), dtype=torch.uint8, device=device)
    for _ in range(5):
        menv.step_many(tape, trace=False)
    t = timed(lambda: menv.step_many(tape, trace=True), 4)
    out["step_many_env_steps_per_s"] = Bm * K / t
    out["step_many"] = {"k_steps": K, "envs": Bm, "us_per_step_equivalent": t / K * 1e6, "trace": "agent, best_dir, reward, terminated, truncated for every step",
                        "algorithmic_GBps": ALGO_BYTES_PER_STEP * Bm * K / t / 1e9, "frac_of_measured_hbm_peak": ALGO_BYTES_PER_STEP * Bm * K / t / 1e9 / measured_peak_gbs()[0]}
    return out


def env_step_outputs(env):
    """The arrays MazeVectorEnv.step() returned for its last step: obs['agent'], obs['target'], obs['best dir'], reward,
    terminated, truncated (they alias these output buffers of the batch)."""
    b = env.batch
    return {"agent": b.agent, "target": b.target, "best_dir": b.best_dir, "reward": b.reward,
            "terminated": b.terminated, "truncated": b.truncated}


def dump_outputs(path, arrays, seed=0):
    """Write device arrays that share their first dimension (one row per env) as path/<name>.npy: float64 arrays as
    float64, all others as float32 (exact for the coordinates, flags and float32 values written here).  When the rows
    of all arrays would take more than DUMP_BYTES, the same fixed, seeded sample of rows is written from every array,
    and the sampled row indices as rows.npy."""
    import numpy as np
    import torch
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum((8 if a.dtype == torch.float64 else 4) * (a.numel() // max(1, n)) for a in arrays.values())
    budget = DUMP_BYTES - 128 * (len(arrays) + 1)      # .npy headers
    rows = None
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(seed).choice(n, budget // (row_bytes + 8), replace=False))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if rows is not None:
            a = a[torch.from_numpy(rows).to(a.device)]
        a = a.double() if a.dtype == torch.float64 else a.float()
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy())
    if rows is not None:
        np.save(os.path.join(path, "rows.npy"), rows.astype(np.float64))


def pattern_summary(step_us, B):
    """Where the step kernel stands against the measured rate of its own access pattern (DESIGN.md section 4.1)."""
    p = pattern_peak()
    if not p or p.get("envs") != B:
        return None
    return {"what": "tools/perf_scatter_rmw.py on this batch: maze_step's coalesced streams plus one 2-byte read-modify-write at a scattered "
                    "64-byte atom for 40 % of the envs, no maze logic (committed summary: profiles/r02_scatter_rmw.json)",
            "streams_only_us": p["streams_only_us"], "rmw_only_us": p["rmw_only_cell_major_per_env_us"],
            "streams_plus_rmw_us": p["streams_plus_rmw_cell_major_per_env_us"], "maze_step_us_same_run": p["maze_step_us"],
            "frac_of_pattern_same_run": p["streams_plus_rmw_cell_major_per_env_us"] / p["maze_step_us"],
            "frac_of_pattern_this_run": p["streams_plus_rmw_cell_major_per_env_us"] / step_us}


def secondary_metrics(extra):
    """BASELINE.json's second metric and its neighbours as a driver-parsed list."""
    if not extra:
        return None
    out = []
    for algo, v in extra["mazes_per_s_81x81"].items():
        out.append({"metric": f"valid mazes generated/sec (40x40, {algo}, per GPU)", "value": v, "unit": "mazes/s",
                    "roofline": {"bound": "sm issue slots (sequential carving)", "issue_slots_busy": 0.77,
                                 "source": "ncu profiles/r01f_gen_warp_details.txt (maze_generate_warp_kernel)"}})
    out.append({"metric": "valid mazes kept/sec, best of 6 by McClendon difficulty (40x40, r-prim, per GPU)", "value": extra["best_of_6_mazes_per_s_81x81"],
                "unit": "mazes/s"})
    out.append({"metric": "difficulty metrics (MD, MC, ML, MDE, MDs) mazes scored/sec (40x40, r-prim, per GPU)", "value": extra["difficulty_mazes_per_s_81x81"],
                "unit": "mazes/s"})
    return out


# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist

    import maze_b200 as mb

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    pin_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B = args.envs_per_gpu
    env = mb.MazeVectorEnv(num_envs=B, shape=SHAPE, topology="euclid", algorithms="r-prim", num_mazes=NUM_MAZES,
                           device=device, seed=1234, slot_id_base=rank * NUM_MAZES, autoreset=True, on_win="next",
                           stats=False)
    gen = torch.Generator(device=device)
    gen.manual_seed(99 + rank)
    TAPE = 16
    tape = torch.randint(0, 4, (TAPE, B), dtype=torch.uint8, device=device, generator=gen)
    env.reset()
    sampler = ClockSampler(local_rank)   # samples from the warm-up on: same kernel, same load
    sampler.start()
    for t in range(args.warmup):
        env.step(tape[t % TAPE])
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    # one event per launch boundary (cheap: a few hundred events) -> the total AND the median per-launch time
    n_ev = min(args.steps, 512)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_ev + 1)]
    e1 = torch.cuda.Event(enable_timing=True)
    evs[0].record()
    for t in range(args.steps):
        env.step(tape[t % TAPE])
        if t + 1 <= n_ev:
            evs[t + 1].record()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env_step_outputs(env))
    ms = max_over_ranks(evs[0].elapsed_time(e1))
    per_launch_us = sorted(evs[i].elapsed_time(evs[i + 1]) * 1e3 for i in range(n_ev))
    median_launch_us = per_launch_us[len(per_launch_us) // 2]
    value = world * B * args.steps / (ms * 1e-3)
    ms_per_step = ms / args.steps

    # end to end through the public API with HOST buffers on both sides, per step: numpy actions -> pinned -> device,
    # maze_step, results -> pinned host memory, one stream synchronisation.  Two wire formats for the results:
    #   packed: one uint32 record per env (MAZE_STEP_PACKED | MAZE_STEP_NO_WIDE), decoded lazily on the host
    #   wide:   the 26 bytes per env of round 1 (agent, best dir, reward, terminated, truncated as separate arrays)
    # the actions of a step live in pinned host memory (env.pinned_actions(): the buffer a policy on the host writes into)
    host_tape = []
    for i in range(4):
        buf = env.pinned_actions()
        buf.copy_(tape[i])
        host_tape.append(buf)
    torch.cuda.synchronize()
    e2e_steps = max(3, min(args.steps, args.e2e_steps))

    def time_e2e(fn):
        for t in range(3):
            fn(host_tape[t % 4])
        barrier()
        torch.cuda.synchronize()
        env.reset_host_counters()      # d2h_bytes_per_step() = bytes actually copied in the timed region / steps
        t0 = time.perf_counter()
        for t in range(e2e_steps):
            out = fn(host_tape[t % 4])
        torch.cuda.synchronize()
        secs = max_over_ranks(time.perf_counter() - t0)
        barrier()
        return world * B * e2e_steps / secs, env.d2h_bytes_per_step(), out

    e2e_wide, d2h_wide, (obs, rew, term, trunc, _) = time_e2e(env.step_host)
    e2e_packed, d2h_packed, records = time_e2e(env.step_host_packed)

    # The floor of that path on this box: the same bytes over PCIe with no kernel in between (4 MB in, 16 MB out per step
    # and rank, all ranks at once).  e2e.value close to this number means the step is bound by the host link, not the GPU.
    pin_out = torch.empty(B, dtype=torch.int32, pin_memory=True)
    d_in = torch.empty(B, dtype=torch.uint8, device=device)

    def copies_only(actions):
        d_in.copy_(actions, non_blocking=True)
        pin_out.copy_(env.batch.packed, non_blocking=True)
        torch.cuda.current_stream(device).synchronize()
        return None
    transfer_only, _, _ = time_e2e(copies_only)
    # the records decode to exactly what the wide path returns: one more step taken with both outputs switched on,
    # decoded record against the device's wide buffers
    t0 = time.perf_counter()
    dec = mb.cabi.decode_records(records)
    decode_s = time.perf_counter() - t0
    env.step(host_tape[0].to(device), extra_mode=mb.cabi.STEP_PACKED)
    chk = mb.cabi.decode_records(env.batch.packed.cpu().numpy())
    assert (chk["agent"] == env.batch.agent.cpu().numpy()).all() and (chk["best_dir"] == env.batch.best_dir.cpu().numpy()).all()
    assert (chk["reward"].view(np.uint64) == env.batch.reward.cpu().numpy().view(np.uint64)).all()
    assert (chk["terminated"] == env.batch.terminated.cpu().numpy().astype(bool)).all() and (chk["truncated"] == env.batch.truncated.cpu().numpy().astype(bool)).all()
    clocks = sampler.stop()    # sampled from the first warm-up launch to the end of the end-to-end runs (5 ms period)

    extra = None
    if rank == 0 and not args.no_extras:
        extra = measure_extras(mb, torch, device)
    barrier()

    # independent check that the timed kernel did the work: episode bookkeeping must be moving
    st = env.batch.state_host()
    assert st["steps"].max() > 0 and int(rew.shape[0]) == B and int(dec["reward"].shape[0]) == B

    line = None
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        achieved = ALGO_BYTES_PER_STEP * B / (ms_per_step * 1e-3) / 1e9
        prof = ncu_traffic_per_step_byte()
        traffic = None
        if prof and prof.get("dram_bytes_per_env_step") is not None:
            traffic = prof["dram_bytes_per_env_step"] * B   # ncu --set full capture of a steady-state launch
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle.baseline import time_env_steps
            cores = os.cpu_count() or 1
            # same mazes as the GPU run: copy a few pool grids back and hand them to the CPU port
            meta = env.pool.meta_host()
            mazes = []
            for m in range(min(cores, 8)):
                mazes.append(dict(grid=env.pool.grid_host(m), start=(int(meta[m, 2]) & 0xffff, int(meta[m, 2]) >> 16),
                                  goal=(int(meta[m, 3]) & 0xffff, int(meta[m, 3]) >> 16), toroidal=False))
            r = time_env_steps(mazes, args.cpu_seconds, cores, "port")
            r2 = time_env_steps(mazes, min(3.0, args.cpu_seconds), cores, "closed")
            cpu = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{r['steps']} env-steps in {r['seconds']:.1f} s: {cores} processes, each one oracle-port env "
                             f"(A* per step, the reference's algorithm) on one of the GPU run's own 81x81 mazes, random actions",
                   "optimised_cpu_closed_form_value": r2["value"]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/int32 state+obs, f64 reward", "data": "synthetic",
            "config": workload_config(B, world),
            "median_launch_us": median_launch_us,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": "ncu --set full capture of a steady-state launch of the same command (profiles/step_kernel_ncu_summary.json), not measured by this run",
                         "peak_source": peak_src, "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_STEP, "kernel": "maze_step_kernel",
                         "pattern": pattern_summary(median_launch_us, B)},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_packed, "unit": UNIT, "wire": "packed", "h2d_bytes_per_step": env.h2d_bytes_per_step(),
                    "d2h_bytes_per_step": d2h_packed, "steps": e2e_steps,
                    "wide": {"value": e2e_wide, "d2h_bytes_per_step": d2h_wide},
                    "transfer_only_value": transfer_only,
                    "host_decode_s_per_step": decode_s,
                    "note": "MazeVectorEnv.step_host_packed: actions in pinned host memory -> device, maze_step writing ONE uint32 record per env "
                            "(row, col, best-next code, terminated, truncated, reward kind + index; include/maze_b200.h MAZE_REC_*), one copy to "
                            "pinned host memory, one stream synchronisation; `target` (and, under a curriculum, the per-env shapes) travel only on "
                            "steps whose launch changed a maze (maze_env_batch.target_dirty).  Records decode to the wide arrays bit for bit "
                            "(cabi.decode_records, asserted in this run); decoding is left to the consumer and is not inside the timed region "
                            "(host_decode_s_per_step: the library's single-threaded C loop over all envs).  `wide` is round 1's format: "
                            "26 bytes per env in six arrays.  transfer_only_value: the same host<->device copies with no kernel between them, "
                            "all ranks at once -- the floor the host link sets for this path on this box"},
            "gpu_launches": args.steps * world,
            "clocks": clocks,
            "secondary": secondary_metrics(extra),
            "extra": extra,
        }
    if world > 1:
        dist.destroy_process_group()
    return line


# ------------------------------------------------------------------------------------------------
# The other configs of BASELINE.json as one-line measurements (same contract: W warm-up steps, K timed steps between
# barriers + synchronisations, CUDA events, max over ranks, rank 0 prints).
def _dist_setup(local_rank, world):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    return device, barrier, max_over_ranks


def _timed_loop(torch, step_fn, args, barrier, max_over_ranks):
    for _ in range(args.warmup):
        step_fn()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_fn()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    return max_over_ranks(e0.elapsed_time(e1))


def _follow_best_dir(torch, best_dir, u, p_follow):
    """Action that realises obs['best dir'] (= agent - next; +-(S - 1) components are wrapped moves) with probability
    p_follow, a uniform random action otherwise."""
    r, c = best_dir[:, 0], best_dir[:, 1]
    wrapped = (r.abs() > 1) | (c.abs() > 1)
    a = torch.where(r < 0, 0, torch.where(r > 0, 1, torch.where(c < 0, 2, 3)))
    a = torch.where(wrapped, a ^ 1, a)
    rnd = (u * 4096).long() % 4
    return torch.where(u < p_follow, a, rnd).to(torch.uint8)


def _regen_summary(env):
    if not env.regenerate_ahead:
        return {"mode": "in place, on the stepping stream (MAZE_REGEN_AHEAD=0)"}
    fast, slow, jobs = env.regeneration_statistics()
    return {"mode": f"{env.regenerate_depth} mazes ahead per slot (shadow ring refilled on a side stream; include/maze_b200.h maze_regen_swap)",
            "installed_from_shadow": fast, "drawn_in_place": slow, "refill_jobs": jobs, "counted": "rank 0, since construction"}


def run_toroidal_regen(args, rank, local_rank, world):
    """configs[2]: toroidal 40x40 (81x81 block; the reference's examples pass the same odd block shape to both topologies)
    mazes, r-prim / dfs / prim&kill mixed per slot, one maze slot per env, every win regenerates the env's maze on the
    device before its autoreset (maze_curriculum is off; maze_generate runs every step on the device-side queue)."""
    import torch

    import maze_b200 as mb
    device, barrier, max_over_ranks = _dist_setup(local_rank, world)
    B = args.envs_per_gpu if args.envs_per_gpu_set else 262144
    env = mb.MazeVectorEnv(B, shape=SHAPE, topology="toroidal", algorithms=["r-prim", "dfs", "prim&kill"], device=device, seed=1234,
                           slot_id_base=rank * B, on_win="regenerate", stats=True)
    env.reset()
    gen = torch.Generator(device=device)
    gen.manual_seed(7 + rank)

    def step():
        u = torch.rand(B, device=device, generator=gen)
        env.step(_follow_best_dir(torch, env.batch.best_dir, u, 0.7))

    sampler = ClockSampler(local_rank)
    sampler.start()
    s0 = None
    for _ in range(args.warmup):
        step()
    s0 = env.episode_statistics(reduce=world > 1)
    args_w, args.warmup = args.warmup, 0
    ms = _timed_loop(torch, step, args, barrier, max_over_ranks)
    args.warmup = args_w
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env_step_outputs(env))
    s1 = env.episode_statistics(reduce=world > 1)
    clocks = sampler.stop()
    if rank != 0:
        return None
    value = world * B * args.steps / (ms * 1e-3)
    regen = _regen_summary(env)
    return {"metric": "env-steps/sec (toroidal 40x40 mazes, mixed generators, regeneration on win, whole job)", "regeneration": regen, "value": value, "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/int32 state+obs, f64 reward", "data": "synthetic",
            "config": {"workload": f"configs[2]: toroidal 81x81-block mazes (41 logical lines), r-prim / dfs / prim&kill mixed, {B} envs and maze slots per GPU, "
                                   "70 % best-dir following / 30 % uniform actions, every win installs a freshly generated maze (maze_generate on the device; drawn ahead of time into a shadow ring unless MAZE_REGEN_AHEAD=0)",
                       "envs_per_gpu": B, "l2": "inputs larger than L2 (6.5 KB table + 13 KB visits per env)",
                       "parallelism": f"env-index sharding over {world} GPU(s), no per-step collective"},
            "mazes_regenerated_per_s": (s1["wins"] - s0["wins"]) / (ms * 1e-3), "episodes_per_s": (s1["episodes"] - s0["episodes"]) / (ms * 1e-3),
            "gpu_launches": args.steps * world * 4, "clocks": clocks,
            "launches_per_step": "policy (torch elementwise ops) + maze_regen_swap + in-place maze_generate of the not-ready slots (2 kernels, usually empty) + queue resets + maze_step; "
                                 "refills (prepare, maze_generate per ring entry, publish) on the side stream"}


def run_curriculum_dq(args, rank, local_rank, world):
    """configs[3]: variable-size mazes 10x10 -> 64x64 cells (21 -> 129 blocks, + (4, 4) per win: simple_variable_maze_env.py:93-112),
    generator switched by win count (off_policy_trainer.py:302-310), tabular double Q-learning on the device (dq_agent.py:5-73),
    one learner per env (the reference's one table per agent)."""
    import torch

    import maze_b200 as mb
    from maze_b200.agents import DQAgent
    device, barrier, max_over_ranks = _dist_setup(local_rank, world)
    B = args.envs_per_gpu if args.envs_per_gpu_set else 131072
    env = mb.MazeVectorEnv(B, shape=(129, 129), start_shape=(21, 21), grow=4, algorithms="r-prim", device=device, seed=1234, slot_id_base=rank * B,
                           on_win="regenerate", algorithm_schedule=((5, "prim&kill"), (10, "dfs")), stats=True)
    agent = DQAgent(env, learning_rate=0.1, initial_epsilon=0.9, epsilon_decay=2000, final_epsilon=0.05, discount_factor=0.7, eta=1e-3,
                    envs_per_agent=1, seed=1 + rank, capacity=1 << 26)
    env.reset()
    gen = torch.Generator(device=device)
    gen.manual_seed(11 + rank)

    def step():   # behaviour policy: mostly the 'best dir' hint, otherwise the agent's own epsilon-greedy action (off-policy learning)
        acts = agent.get_action()
        u = torch.rand(B, device=device, generator=gen)
        follow = _follow_best_dir(torch, env.batch.best_dir, torch.zeros_like(u), 1.0)
        acts = torch.where(u < 0.85, follow, acts)
        agent.core.last_action.copy_(acts)
        env.step(acts)
        agent.update()

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = _timed_loop(torch, step, args, barrier, max_over_ranks)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env_step_outputs(env))
    clocks = sampler.stop()
    agent.core.check_overflow()
    stats = env.episode_statistics(reduce=world > 1)
    shapes = env.pool.meta[:, 0].float()
    if rank != 0:
        return None
    value = world * B * args.steps / (ms * 1e-3)
    return {"metric": "env-steps/sec (variable-size 10x10 -> 64x64 curriculum, double Q-learning on device, whole job)", "value": value, "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/int32 state+obs, f64 reward and Q values", "data": "synthetic",
            "config": {"workload": f"configs[3]: {B} envs per GPU, mazes from 21x21 blocks growing by (4, 4) per win up to 129x129, r-prim -> prim&kill -> dfs "
                                   "after 5 / 10 wins, device DQAgent (maze_q_act + maze_step + maze_q_update per step), 85 % best-dir behaviour policy",
                       "envs_per_gpu": B, "l2": "inputs larger than L2 (33 KB visits per env at the pool shape)",
                       "parallelism": f"env-index sharding over {world} GPU(s), replicas only (one Q table per env, as in the reference)"},
            "wins": stats["wins"], "mean_block_shape_after_run": float(shapes.mean().item()), "max_block_shape_after_run": float(shapes.max().item()),
            "regeneration": _regen_summary(env), "gpu_launches": args.steps * world * 7, "clocks": clocks}


def run_ddqn(args, rank, local_rank, world):
    """configs[4]: the DDQN loop of examples/train_ddqn.py (8192 envs per GPU; net on the tensor cores; one NCCL all-reduce of the
    8.7 MB gradient per optimiser step)."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    from train_ddqn import DDQNLoop
    device, barrier, max_over_ranks = _dist_setup(local_rank, world)
    B = args.envs_per_gpu if args.envs_per_gpu_set else 8192
    n = args.batch or B
    loop = DDQNLoop(B, n, SHAPE[0], 1 << 20, rank, world, device, overlap=not args.no_overlap)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, (n + B - 1) // B + 2)):
        loop.iterate()
    loop.ar_events, opt0 = [], loop.opt_steps
    args_w, args.warmup = args.warmup, 0
    ms = _timed_loop(torch, lambda: loop.iterate(time_allreduce=True), args, barrier, max_over_ranks)
    args.warmup = args_w
    if args.dump_outputs and rank == 0:      # the env step plus the policy's Q values that chose its actions
        dump_outputs(args.dump_outputs, dict(env_step_outputs(loop.env), q=loop.q))
    clocks = sampler.stop()
    ar_ms = sum(a.elapsed_time(b) for a, b in loop.ar_events)
    # the dominant kernel inside the step, measured live: maze_dqn_backward records a CUDA event after every launch while the
    # in-situ profiler is on (outside the timed region: the events cost a little)
    kernel = None
    try:
        loop.net.profile(True)
        seen = {}
        for _ in range(8):
            loop.iterate()
            for i, (label, k_ms) in enumerate(loop.net.profile_read()):
                seen.setdefault((i, label), []).append(k_ms)
        loop.net.profile(False)
        med = {k: sorted(v)[len(v) // 2] for k, v in seen.items()}
        total = sum(med.values())
        by_label = {}
        for (_, label), k_ms in med.items():
            by_label.setdefault(label, []).append(k_ms)
        label, times = max(by_label.items(), key=lambda kv: sum(kv[1]))   # the kernel with the largest share of the pass
        gemm_flop = {"fc1 forward GEMM": 2.0 * n * 1024 * 1600, "fc2 forward GEMM": 2.0 * n * 512 * 1024,
                     "fc1 weight gradient GEMM (split-K)": 2.0 * n * 1024 * 1600, "fc1 backward-data GEMM": 2.0 * n * 1568 * 1024}.get(label)
        k_ms = sum(times) / len(times)
        kernel = {"label": label, "launches_per_backward": len(times), "ms_per_launch": k_ms, "share_of_backward": sum(times) / total if total else None,
                  "flop_per_launch": gemm_flop, "tflops": gemm_flop / (k_ms * 1e-3) / 1e12 if gemm_flop else None,
                  "how": "median of 8 in-situ measurements per launch (CUDA events between the launches of maze_dqn_backward, maze_dqn_net_profile)"}
    except Exception as e:   # a profile that cannot be taken must not cost the bench line
        kernel = {"error": repr(e)}
    if rank != 0:
        return None
    n_opt = loop.opt_steps - opt0
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        peak, peak_src = 1400.0, "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"
    tflops = loop.flop_per_iteration() * args.steps / (ms * 1e-3) / 1e12
    return {"metric": "env-steps/sec (DDQN training loop on 40x40 mazes, whole job)", "value": world * B * args.steps / (ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 operands, fp32 accumulate / master weights", "data": "synthetic",
            "config": {"workload": f"configs[4]: DDQN loop, {B} -v1 envs per GPU on 81x81 r-prim mazes regenerated on win, replay batch {n} per GPU per "
                                   "optimiser step, one optimiser step per env step, net of agents/ddqn_agent.py:18-52 (dropout off)",
                       "envs_per_gpu": B, "batch_per_gpu": n, "parallelism": f"data parallel over {world} GPU(s): envs and replay sharded, one NCCL all-reduce "
                                   "(sum) of the flat fp32 gradient (8.7 MB) per optimiser step"},
            "samples_per_s": world * n * n_opt / (ms * 1e-3), "optimizer_steps_per_s": n_opt / (ms * 1e-3),
            "allreduce": ("separate: the whole gradient is reduced after the backward pass (timed: allreduce_share)" if args.no_overlap or world == 1 else
                          "overlapped: grads[MAZE_NET_OFF_W1:] are reduced on a side stream while the backward-data GEMM and the conv gradient run "
                          "(maze_dqn_backward's fc_ready_event); run with --no-overlap for the separate, timed variant"),
            "allreduce_share": (ar_ms / ms) if (args.no_overlap and world > 1) else None,
            "roofline": {"bound": "tensor", "achieved": tflops, "peak": peak, "unit": "TFLOP/s", "frac": tflops / peak, "traffic": None, "peak_source": peak_src,
                         "flop_per_step_per_gpu": loop.flop_per_iteration(),
                         "dominant_kernel": (dict(kernel, frac_of_peak=(kernel["tflops"] / peak if kernel.get("tflops") else None)) if kernel else None),
                         "note": "whole loop per GPU (policy forward on B envs + forward on 3 n and backward on n samples per optimiser step; env step, "
                                 "replay, sampling, AdamW and the all-reduce included in the time)"},
            "final_loss": float(loop.net.loss.item()), "gpu_launches": args.steps * world * 40, "clocks": clocks}


class JsonOnlyStdout:
    """The driver parses stdout as ONE JSON line: everything else a library prints there (NCCL's
    version banner, for one) is sent to stderr by pointing fd 1 at fd 2 for the duration of the run."""

    def __enter__(self):
        sys.stdout.flush()
        self._real = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line: str):
        sys.stdout.flush()
        os.write(self._real, (line + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._real, 1)
        os.close(self._real)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 2000 for configs1, 200 for the other workloads)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default: 500 for configs1, 20 for the other workloads)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=None)
    ap.add_argument("--workload", default="configs1", choices=["configs1", "toroidal-regen", "curriculum-dq", "ddqn"])
    ap.add_argument("--batch", type=int, default=0, help="ddqn: replay batch per GPU per optimiser step (default: envs per GPU)")
    ap.add_argument("--no-overlap", action="store_true", help="ddqn: all-reduce the whole gradient after the backward pass and time it (allreduce_share)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's envs) as DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()
    args.envs_per_gpu_set = args.envs_per_gpu is not None
    if args.envs_per_gpu is None:
        args.envs_per_gpu = 4096 * NUM_MAZES
    if args.steps is None:      # configs1 steps take about 90 us, the other workloads' several times that
        args.steps = 2000 if args.workload == "configs1" else 200
    if args.warmup is None:
        args.warmup = 500 if args.workload == "configs1" else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    with JsonOnlyStdout() as out:
        if args.impl == "reference":
            line = run_reference(args, rank)
        elif args.workload == "configs1":
            line = run_ours(args, rank, local_rank, world)
        else:
            fn = {"toroidal-regen": run_toroidal_regen, "curriculum-dq": run_curriculum_dq, "ddqn": run_ddqn}[args.workload]
            line = fn(args, rank, local_rank, world)
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()
        if line is not None:
            out.emit(json.dumps(line))


if __name__ == "__main__":
    main()
