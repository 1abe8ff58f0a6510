#!/usr/bin/env python
"""What does the memory system give maze_step's access pattern?  (VERDICT r01 item 3.)

Times maze_bench_scatter_rmw (csrc/maze_bench.cu) on the bench's own batch -- 4 096 000 envs on 1 000 81 x 81
mazes, a [slot, B] uint16 visit array of 54 GB -- for every combination of {streams only, RMW only, both} x
{uniform, cell-major per env, cell-major per warp}, and the real maze_step kernel at steady state beside them.
Writes gpurun_out/scatter_rmw.json (copy the summary into profiles/).

--order times the CTA order instead: streams + cell-major RMW with the CTAs in the same order every launch
("fwd") against reversed on odd launches ("alt", what maze_step does), with and without lag-1 re-touches (a
share of the touched atoms that the same env touched one launch earlier: 0.20 in a count of the bench's random
walk), under the L2-policy variants of csrc/maze_bench.cu.  Writes its summary to --out.

    python tools/perf_scatter_rmw.py [--envs 4096000] [--iters 200] [--once PATTERN STREAMS]   # --once: one config, for ncu
    python tools/perf_scatter_rmw.py --order [--rounds 3] [--out scatter_order.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb  # noqa: E402
from maze_b200 import cabi  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096000)
    ap.add_argument("--mazes", type=int, default=1000)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--once", nargs=2, type=int, default=None)
    ap.add_argument("--order", action="store_true")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="scatter_order.json", help="--order: file the summary is written to")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    B = args.envs
    env = mb.MazeVectorEnv(B, shape=(81, 81), algorithms="r-prim", num_mazes=args.mazes, seed=1234, device=dev, stats=False)
    env.reset()
    b = env.batch
    lib, ctx = cabi.lib(), b.ctx
    acts = torch.randint(0, 4, (64, B), device=dev, dtype=torch.uint8)
    arr, n_elems = b.visits, b.visits.numel()
    stream = cabi.current_stream(dev)

    def launch(pattern, rate, it, streams, order=0, retouch=0, hints=0):
        rc = lib.maze_bench_scatter_rmw(ctx.handle, C.byref(b._c), cabi.ptr(acts[it % 64]), cabi.ptr(arr), n_elems, pattern, rate, it, streams,
                                        order, retouch, hints, stream)
        ctx.check(rc, "maze_bench_scatter_rmw")

    def timed(fn, iters):
        for i in range(20):
            fn(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(20 + i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters * 1e3   # microseconds per launch

    if args.once is not None:
        pattern, streams = args.once
        for i in range(30):
            launch(pattern, 410, i, streams)
        torch.cuda.synchronize()
        return
    if args.order:
        return order_study(args, b, acts, launch, timed)
    out = {"envs": B, "array_bytes": n_elems * 2, "rmw_fraction": 410 / 1024}
    # the real kernel at steady state (autoreset on, same maze pool): what the patterns are compared with
    mode = cabi.STEP_AUTORESET
    for i in range(300):
        b.step(acts[i % 64], mode)
    out["maze_step_us"] = timed(lambda i: b.step(acts[i % 64], mode), args.iters)
    state_keep = b.state.clone()
    out["streams_only_us"] = timed(lambda i: launch(0, 0, i, 1), args.iters)
    for pattern, name in ((0, "uniform"), (1, "cell_major_per_env"), (2, "cell_major_per_warp")):
        out[f"rmw_only_{name}_us"] = timed(lambda i: launch(pattern, 410, i, 0), args.iters)
        out[f"streams_plus_rmw_{name}_us"] = timed(lambda i: launch(pattern, 410, i, 1), args.iters)
    for rate in (102, 205, 410, 820, 1024):
        out[f"streams_plus_rmw_cell_major_per_env_rate{rate}_us"] = timed(lambda i: launch(1, rate, i, 1), args.iters)
    b.state.copy_(state_keep)
    n_rmw = B * 410 / 1024
    out["rmw_per_launch"] = n_rmw
    out["atoms_gbs_rmw_only_cell_major_per_env"] = n_rmw * 128 / out["rmw_only_cell_major_per_env_us"] / 1e3
    out["step_vs_pattern"] = out["streams_plus_rmw_cell_major_per_env_us"] / out["maze_step_us"]
    print(json.dumps(out, indent=1))
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "scatter_rmw.json"), "w"), indent=1)


HINTS = {1: "all_evict_last", 2: "state_evict_first_visits_evict_last", 3: "state_evict_last_visits_default"}


def order_study(args, b, acts, launch, timed):
    import statistics
    mode = cabi.STEP_AUTORESET
    for i in range(300):
        b.step(acts[i % 64], mode)
    state_keep = b.state.clone()
    configs = []
    for rate in (410, 530):                       # the r02 assumption; 0.518 legal moves per env-step in the walk count
        for lag1 in (0.0, 0.20):                  # share of touched atoms last touched one launch earlier
            retouch = min(1024, round(lag1 * 1024 * 1024 / rate))   # of the envs whose previous launch did an RMW
            for hints in HINTS:
                for order in (0, 1):
                    configs.append((rate, lag1, retouch, hints, order))
    times = {c: [] for c in configs}
    step_us = []
    for _ in range(args.rounds):                  # rounds interleave the configs, so drift hits all of them alike
        for c in configs:
            rate, _, retouch, hints, order = c
            times[c].append(timed(lambda i: launch(1, rate, i, 1, order, retouch, hints), args.iters))
        b.state.copy_(state_keep)
        step_us.append(timed(lambda i: b.step(acts[i % 64], mode), args.iters))
    b.state.copy_(state_keep)
    props = torch.cuda.get_device_properties(0)
    out = {"envs": b.num_envs, "iters": args.iters, "rounds": args.rounds, "device": props.name,
           "what": "median us per launch of streams + cell-major RMW (maze_bench_scatter_rmw pattern 1); fwd = same CTA order every launch, "
                   "alt = reversed on odd launches",
           "maze_step_us_this_build": statistics.median(step_us), "variants": []}
    for rate in (410, 530):
        for lag1 in (0.0, 0.20):
            for hints, hname in HINTS.items():
                fwd, alt = (statistics.median(times[c]) for c in configs if c[0] == rate and c[1] == lag1 and c[3] == hints)
                retouch = next(c[2] for c in configs if c[0] == rate and c[1] == lag1)
                out["variants"].append({"rmw_per_1024": rate, "lag1_share": lag1, "retouch_per_1024": retouch, "hints": hname,
                                        "fwd_us": fwd, "alt_us": alt, "alt_over_fwd": alt / fwd,
                                        "fwd_runs_us": times[(rate, lag1, retouch, hints, 0)], "alt_runs_us": times[(rate, lag1, retouch, hints, 1)]})
    print(json.dumps(out, indent=1))
    if os.path.dirname(args.out):
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
