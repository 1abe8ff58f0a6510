#!/usr/bin/env python
"""BASELINE.json configs[4]: a DDQN training loop on thousands of parallel 40x40 maze envs per GPU, sharded over the
GPUs of one box, gradients summed with one NCCL all-reduce per optimiser step.

    python examples/train_ddqn.py --envs 8192 --iters 200
    python examples/train_ddqn.py --agent dqn --dropout 0.2      # the plain DQN target; Dropout(0.2) in the conv stage
    torchrun --nproc-per-node 8 --master-addr 127.0.0.1 examples/train_ddqn.py --envs 8192 --iters 200

Everything runs in this repo's kernels: env step (maze_step), masked epsilon-greedy (maze_dqn_select), bit-packed replay
ring (maze_dqn_push / maze_dqn_sample_packed), regeneration of won mazes (maze_generate) and the network itself -- the
architecture of the reference's agents/ddqn_agent.py:18-52 and its update :113-152 -- on the tensor cores
(maze_dqn_forward / maze_dqn_backward / maze_dqn_adamw: tcgen05 GEMMs fed by TMA, csrc/maze_net.cu).  The loop is
lib/trainers/off_policy_trainer.py:163-222 for B envs at once: act, step, memorize, optimize_model, periodic target update.
Prints one JSON line with env-steps/s, samples/s and the all-reduce share of the step.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
import maze_b200 as mb  # noqa: E402
from maze_b200.dqn import DeviceReplay, MaskedEpsilonGreedy  # noqa: E402
from maze_b200.dqn_net import DQNNet  # noqa: E402

FWD_FLOP = 2 * (225 * 32 * 27 + 1574 * 1024 + 1024 * 512 + 512 * 4)   # per sample, forward


class DDQNLoop:
    """One rank's share of config 5."""

    def __init__(self, envs: int, batch: int, shape: int = 81, memory: int = 1 << 20, rank: int = 0, world: int = 1, device="cuda",
                 lr: float = 1e-4, gamma: float = 0.9, target_every: int = 50, seed: int = 1, overlap: bool = True,
                 agent: str = "ddqn", dropout: float = 0.0):
        if agent not in ("ddqn", "dqn"):
            raise ValueError(f"agent must be 'ddqn' or 'dqn', got {agent!r}")
        self.B, self.n, self.rank, self.world, self.overlap = envs, batch, rank, world, overlap
        self.agent, self.dropout = agent, float(dropout)
        self.lr, self.gamma, self.target_every = lr, gamma, target_every
        self.device = torch.device(device)
        self.env = mb.MazeVectorEnv(envs, shape=(shape, shape), enrich=True, on_win="regenerate", algorithms="r-prim", seed=seed,
                                    slot_id_base=rank * envs, device=self.device, stats=True,
                                    algorithm_schedule=((5, "prim&kill"), (10, "dfs")))   # off_policy_trainer.py:302-310
        self.memory = DeviceReplay(self.env, max(memory, envs), seed=rank)
        self.actor = MaskedEpsilonGreedy(self.env, 0.9, 0.05, 2000, seed=7, env_id_base=rank * envs)
        # same initial weights on every rank; each rank draws its own dropout masks
        self.net = DQNNet(self.device, max_batch=max(envs, batch), seed=0, dropout=dropout, double_q=agent == "ddqn",
                          dropout_seed=(int(seed) << 32) | rank)
        self.q = torch.zeros((envs, 4), dtype=torch.float32, device=self.device)
        self.iters = 0
        self.opt_steps = 0
        self.env.reset()
        self.memory.observe()
        self.ar_events = []

    def iterate(self, time_allreduce: bool = False):
        net, mem, env = self.net, self.memory, self.env
        net.forward(mem.stage_vec, mem.stage_win, out=self.q)          # source_net(state) for every env
        actions = self.actor.select(self.q)
        env.step(actions, observe=False)                               # the net reads the packed windows, not the float ones
        mem.push(actions)
        self.iters += 1
        if self.iters * self.B >= self.n:                              # len(memory) >= batch_size, without a device sync
            batch = mem.sample_packed(self.n)
            if self.world > 1 and self.overlap:
                # the fc gradients are all-reduced on a side stream while the tail of the backward pass still runs
                net.train_step_overlapped(*batch, gamma=self.gamma, lr=self.lr, world=self.world)
            else:
                net.backward(*batch, gamma=self.gamma)
                if self.world > 1:
                    if time_allreduce:
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                    dist.all_reduce(net.grads)                         # the DQN gradient all-reduce: 8.7 MB of fp32
                    if time_allreduce:
                        e1.record()
                        self.ar_events.append((e0, e1))
                net.adamw(self.lr, grad_scale=1.0 / self.world)
            self.opt_steps += 1
        if self.iters % self.target_every == 0:
            net.update_target()

    def flop_per_iteration(self):
        """Forward on B envs; per optimiser step forward on 3 n samples (DQN: 2 n) and backward (2 x forward) on n."""
        return FWD_FLOP * (self.B + (5 if self.agent == "ddqn" else 4) * self.n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192, help="envs per GPU")
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--batch", type=int, default=8192, help="replay batch per GPU per optimiser step")
    ap.add_argument("--shape", type=int, default=81)
    ap.add_argument("--memory", type=int, default=1 << 20)
    ap.add_argument("--no-overlap", action="store_true", help="all-reduce the whole gradient after the backward pass (and time it)")
    ap.add_argument("--agent", choices=["ddqn", "dqn"], default="ddqn", help="double-Q target (ddqn_agent.py) or max target (dqn_agent.py)")
    ap.add_argument("--dropout", type=float, default=0.0, help="Dropout p after the conv's LeakyReLU (the reference's DDQN: 0.2)")
    args = ap.parse_args()
    rank, local, world = mb.dist.env_from_torchrun()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    loop = DDQNLoop(args.envs, args.batch, args.shape, args.memory, rank, world, device, overlap=not args.no_overlap, agent=args.agent,
                    dropout=args.dropout)
    warmup = max(5, min(20, args.iters // 4))
    for _ in range(warmup):
        loop.iterate()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    loop.ar_events, opt0 = [], loop.opt_steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.iters):
        loop.iterate(time_allreduce=True)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    dt = float(ms.item()) * 1e-3
    ar_ms = sum(a.elapsed_time(b) for a, b in loop.ar_events)
    stats = loop.env.episode_statistics(reduce=world > 1)
    if rank == 0:
        n_opt = loop.opt_steps - opt0
        print(json.dumps({"agent": args.agent, "dropout": args.dropout, "env_steps_per_s": world * args.envs * args.iters / dt, "optimizer_steps_per_s": n_opt / dt,
                          "samples_per_s": world * args.batch * n_opt / dt, "n_gpus": world, "envs_per_gpu": args.envs,
                          "batch_per_gpu": args.batch, "ms_per_iteration": dt / args.iters * 1e3,
                          "allreduce_share": ar_ms * 1e-3 / dt, "tflops_per_gpu": loop.flop_per_iteration() * args.iters / dt / 1e12,
                          "final_loss": float(loop.net.loss.item()), "episodes": stats["episodes"], "wins": stats["wins"]}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
