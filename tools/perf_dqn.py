"""Scratch: DQN data path rates (step + bit-packed observe + replay push; batch sampling)."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb
from maze_b200.dqn import DeviceReplay
def timed(fn, reps):
    fn(); torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e[0].record()
    for _ in range(reps): fn()
    e[1].record(); torch.cuda.synchronize()
    return e[0].elapsed_time(e[1]) / reps * 1e-3
for lay in ("tile", "cell"):
    B = 1048576
    venv = mb.MazeVectorEnv(B, shape=(81, 81), num_mazes=1000, enrich=True, seed=1234, on_win="next", stats=False, visit_layout=lay)
    venv.reset()
    acts = torch.randint(0, 4, (B,), dtype=torch.uint8, device="cuda")
    for _ in range(300): venv.batch.step(acts, venv._mode)
    memory = DeviceReplay(venv, 1 << 20, seed=1)
    memory.observe()
    def step_push():
        venv.batch.step(acts, venv._mode); memory.push(acts)
    t = timed(step_push, 100)
    t2 = timed(lambda: memory.push(acts), 100)
    print(f"{lay}: step+push {t*1e6:.0f} us {B/t:.3e} env-steps/s; push alone {t2*1e6:.0f} us {B/t2:.3e}/s", flush=True)
    del venv, memory
