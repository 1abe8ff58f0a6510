"""Train-step time (backward + AdamW) of the net's three update variants at n = 8192, alternated in one process:
DDQN without dropout (the default), DDQN with Dropout(0.2), DQN (max target) without dropout.

    python tools/perf_net_variants.py [--out profiles/net_variants.json] [--steps 200] [--rounds 5]

Each round times `steps` train steps of every variant in turn (CUDA events around each step, after a warm-up), so that
clock and neighbour drift hit all three alike; the reported step time is the median over all rounds' steps, with the
spread of the per-round medians.  A separate pass with the in-situ profiler (maze_dqn_net_profile) gives the feature
passes' times inside the step.  The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

VARIANTS = (("ddqn_p0", dict(dropout=0.0, double_q=True)), ("ddqn_p0.2", dict(dropout=0.2, double_q=True)),
            ("dqn_p0", dict(dropout=0.0, double_q=False)))


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + [None] * 3)[:3] if q.returncode == 0 else (torch.cuda.get_device_name(0), None, None)
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def batch(n, seed):
    from net_reference import pack_windows
    g = torch.Generator(device="cpu").manual_seed(seed)
    win = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).float().cuda()
    nwin = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).float().cuda()
    vec, nvec = torch.rand(n, 6, generator=g).cuda(), torch.rand(n, 6, generator=g).cuda()
    action = torch.randint(0, 4, (n,), generator=g).to(torch.uint8).cuda()
    reward = (torch.rand(n, generator=g) - 0.5).cuda()
    return vec, pack_windows(win), nvec, pack_windows(nwin), action, reward


def main():
    from maze_b200.dqn_net import DQNNet
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per variant and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    n = args.n
    data = batch(n, 30)
    nets = {name: DQNNet("cuda", max_batch=n, seed=6, **kw) for name, kw in VARIANTS}
    for net in nets.values():   # warm-up: modules loaded, every launch shape seen
        for _ in range(10):
            net.train_step(*data, gamma=0.9, lr=1e-4)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    times = {name: [] for name in nets}
    round_medians = {name: [] for name in nets}
    for _ in range(args.rounds):
        for name, net in nets.items():
            for e0, e1 in ev:
                e0.record()
                net.train_step(*data, gamma=0.9, lr=1e-4)
                e1.record()
            torch.cuda.synchronize()
            ms = [e0.elapsed_time(e1) for e0, e1 in ev]
            times[name] += ms
            round_medians[name].append(statistics.median(ms))
    insitu = {}
    for name, net in nets.items():   # the in-situ launch list, in a pass of its own (an event after every launch)
        net.profile(True)
        feats, heads, total = [], [], []
        for _ in range(20):
            net.backward(*data, 0.9)
            launches = net.profile_read()
            net.adamw(1e-4)
            feats.append([ms for lab, ms in launches if lab.startswith("features")])
            heads.append([ms for lab, ms in launches if lab.startswith("head")][0])
            total.append(sum(ms for _, ms in launches))
        net.profile(False)
        labels = [lab for lab, _ in launches]
        insitu[name] = {"feature_passes": len(feats[0]), "feature_labels": [lab for lab in labels if lab.startswith("features")],
                        "feature_pass_ms_median": [statistics.median(f[i] for f in feats) for i in range(len(feats[0]))],
                        "head_ms_median": statistics.median(heads), "backward_launches_ms_median": statistics.median(total)}
    res = {"what": "train step (maze_dqn_backward + maze_dqn_adamw) at n = %d, CUDA events per step, median over %d rounds x %d steps, "
                   "variants alternated per round" % (n, args.rounds, args.steps),
           "card": card(), "n": n,
           "variants": {name: {"step_ms_median": statistics.median(times[name]), "round_medians_ms": round_medians[name],
                               "round_spread_ms": max(round_medians[name]) - min(round_medians[name]), **insitu[name]} for name in nets}}
    base = res["variants"]["ddqn_p0"]["step_ms_median"]
    for name in nets:
        res["variants"][name]["vs_ddqn_p0"] = res["variants"][name]["step_ms_median"] / base
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
