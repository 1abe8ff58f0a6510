"""Scratch: -v1 step (maze_step + maze_window) and maze_window alone."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb
for B, lay in ((262144, "cell"), (1048576, "cell"), (1048576, "tile")):
    venv = mb.MazeVectorEnv(B, shape=(81, 81), num_mazes=1000, enrich=True, seed=1234, on_win="next", stats=False, visit_layout=lay)
    venv.reset()
    acts = torch.randint(0, 4, (B,), dtype=torch.uint8, device="cuda")
    for _ in range(300): venv.batch.step(acts, venv._mode)
    def timed(fn, reps=50):
        fn(); torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        for _ in range(reps): fn()
        e[1].record(); torch.cuda.synchronize()
        return e[0].elapsed_time(e[1]) / reps * 1e-3
    tw = timed(lambda: venv.batch.compute_window())
    ts = timed(lambda: venv.step(acts))
    print(f"B={B} {lay}: window {tw*1e6:.1f} us  {B*2700/tw/1e9:.0f} GB/s written ({B*2700/tw/1e9/6545.3:.2f} of peak);  step+window {ts*1e6:.1f} us  {B/ts:.3e} env-steps/s")
    del venv
