"""Scratch: maze_generate throughput per algorithm, bordered and toroidal."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb
M = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
tors = (False, True) if len(sys.argv) <= 2 else (False,)
for tor in tors:
    for algo in ("r-prim", "dfs", "prim&kill"):
        pool = mb.MazePool(M, (81, 81))
        pool.generate(algorithms=algo, toroidal=tor, seed=1)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for r in range(3):
            pool.generate(algorithms=algo, toroidal=tor, seed=2 + r)
        ev[1].record(); torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / 3
        print(f"{algo:10s} tor={tor} M={M}: {ms:.2f} ms  {M/ms*1e3:.3e} mazes/s", flush=True)
        del pool
