"""Scratch: best-of-6 generation rate of the bulk path (planes kernel + scoring kernel)."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb
n = 16384
for algo in ("r-prim", "dfs", "prim&kill"):
    pool = mb.MazePool(n, (81, 81)); pool.generate(algorithms=algo, seed=5)
    pool.generate(algorithms=algo, seed=6, candidates=6, configure=False); torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(); pool.generate(algorithms=algo, seed=7, candidates=6, configure=False); ev[1].record(); torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1])
    print(f"{algo:10s}: {ms:8.1f} ms  {n/ms*1e3:.3e} kept mazes/s", flush=True)
    del pool
