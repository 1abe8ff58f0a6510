"""Scratch: maze_difficulty throughput per generation algorithm."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb
M = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
for algo in ("r-prim", "dfs", "prim&kill"):
    pool = mb.MazePool(M, (81, 81)); pool.generate(algorithms=algo, seed=3)
    pool.difficulty(); torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(); pool.difficulty(); pool.difficulty(); ev[1].record(); torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 2
    print(f"{algo:10s} M={M}: {ms:.2f} ms  {M/ms*1e3:.3e} mazes/s", flush=True)
    del pool
