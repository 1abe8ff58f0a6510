"""Scratch: maze_step time per launch for visit layouts x batch sizes, steady state, CUDA-graph replay.
usage: python tools/perf_step.py [layouts] [sizes]   e.g.  cell,tile 1048576,4096000"""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb

layouts = (sys.argv[1] if len(sys.argv) > 1 else "cell,tile").split(",")
sizes = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "1048576,4096000").split(",")]
M, TAPE = 1000, 16
S = int(sys.argv[3]) if len(sys.argv) > 3 else 81
pool = mb.MazePool(M, (S, S))
pool.generate(algorithms="r-prim", seed=1234)
mode = mb.cabi.STEP_AUTORESET | mb.cabi.STEP_WIN_NEXT
for B in sizes:
    acts = torch.randint(0, 4, (TAPE, B), dtype=torch.uint8, device="cuda")
    for lay in layouts:
        env_maze = (torch.arange(B, device="cuda", dtype=torch.int32) // max(1, B // M)).clamp_(max=M - 1)
        batch = mb.MazeBatch(pool, B, env_maze=env_maze, visit_layout=lay)
        batch.reset()
        for t in range(TAPE):
            batch.step(acts[t], mode)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for t in range(TAPE):
                batch.step(acts[t], mode)
        for _ in range(600 // TAPE):
            g.replay()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        reps = 400 // TAPE
        ev[0].record()
        for _ in range(reps):
            g.replay()
        ev[1].record(); torch.cuda.synchronize()
        us = ev[0].elapsed_time(ev[1]) / (reps * TAPE) * 1e3
        print(f"S={S} B={B:8d} layout={lay:5s} {us:7.1f} us/step  {B/us*1e6:.3e} steps/s  algorithmic {58*B/us/1e3:.0f} GB/s  frac {58*B/us/1e3/6545.3:.3f}", flush=True)
        del batch, g
