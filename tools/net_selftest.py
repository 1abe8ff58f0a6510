#!/usr/bin/env python
"""GPU self-test of the tensor-core network kernels against PyTorch (run on a B200 through gpurun):

    python tools/net_selftest.py            # every case, each in its own process (a trap in one does not hide the others)
    python tools/net_selftest.py gemm0      # one case

Prints one line per check: name, max abs error, reference scale, verdict.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

CASES = ["gemm0", "gemm1", "gemm2", "gemm_mask", "gemm_red", "features", "forward", "backward", "adamw", "perf"]


def report(name, got, ref, tol):
    import torch
    got, ref = got.float(), ref.float()
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    bad = ((got - ref).abs() > tol * max(scale, 1e-6)).float().mean().item()
    ok = err <= tol * max(scale, 1e-6)
    print(f"{'ok  ' if ok else 'FAIL'} {name}: max_abs_err {err:.4g} ref_max {scale:.4g} frac_bad {bad:.4f}", flush=True)
    if not ok and got.dim() == 2:
        e = (got - ref).abs() > tol * max(scale, 1e-6)
        R, Cc = e.shape
        rows = e.float().mean(1)
        cols = e.float().mean(0)
        print("   bad rows by (row % 128)//8:", [round(rows[i::128].mean().item(), 2) for i in range(0, min(128, R), 8)], flush=True)
        print("   bad cols by (col % 64)//8 :", [round(cols[i::64].mean().item(), 2) for i in range(0, min(64, Cc), 8)], flush=True)
        print("   bad cols by col//32 (first 16):", [round(cols[i * 32:(i + 1) * 32].mean().item(), 2) for i in range(min(16, Cc // 32))], flush=True)
        print("   got[0,:8]", got[0, :8].tolist(), "\n   ref[0,:8]", ref[0, :8].tolist(), flush=True)
    return ok


def case_gemm(M, N, K, tile_n, epi=0, act=0, splits=1, seed=0):
    import torch
    from maze_b200.dqn_net import gemm_bf16
    torch.manual_seed(seed)
    d = "cuda"
    A = (torch.randn(M, K, device=d) * 0.5).bfloat16()
    B = (torch.randn(N, K, device=d) * 0.5).bfloat16()
    ref = A.float() @ B.float().t()
    name = f"gemm M{M} N{N} K{K} tile{tile_n} epi{epi} act{act} splits{splits}"
    if epi == 0:
        bias = torch.randn(N, device=d)
        C = torch.zeros(M, N, device=d, dtype=torch.bfloat16)
        gemm_bf16(A, B, C, 0, act, bias=bias, tile_n=tile_n)
        r = ref + bias
        if act == 1:
            r = torch.nn.functional.leaky_relu(r, 0.01)
        elif act == 2:
            r = torch.relu(r)
        return report(name, C, r, 1e-2)
    if epi == 1:
        aux = torch.randn(M, N, device=d).bfloat16()
        C = torch.zeros(M, N, device=d, dtype=torch.bfloat16)
        gemm_bf16(A, B, C, 1, act, aux=aux, tile_n=tile_n)
        fac = torch.where(aux.float() > 0, 1.0, 0.01 if act == 1 else 0.0)
        return report(name, C, ref * fac, 1e-2)
    C = torch.ones(M, N, device=d, dtype=torch.float32)
    gemm_bf16(A, B, C, 2, 0, tile_n=tile_n, splits=splits)
    return report(name, C, ref + 1.0, 2e-3)


def make_batch(n, seed=0, device="cuda"):
    import torch
    from net_reference import pack_windows
    g = torch.Generator(device="cpu").manual_seed(seed)
    win = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).float().to(device)
    vec = torch.rand(n, 6, generator=g).to(device)
    vec[:, 4:] = torch.randint(-1, 2, (n, 2), generator=g).float().to(device)
    nwin = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).float().to(device)
    nvec = torch.rand(n, 6, generator=g).to(device)
    action = torch.randint(0, 4, (n,), generator=g).to(torch.uint8).to(device)
    reward = (torch.rand(n, generator=g) - 0.5).to(device)
    return dict(vec=vec, win=win, pwin=pack_windows(win), nvec=nvec, nwin=nwin, pnwin=pack_windows(nwin), action=action, reward=reward)


def ref_nets(net):
    import torch
    from net_reference import RefDQN
    src, tgt = RefDQN().to(net.device), RefDQN().to(net.device)
    src.load_state_dict(net.state_dict("source"))
    tgt.load_state_dict(net.state_dict("target"))
    return src, tgt


def run_case(case):
    import torch
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ok = True
    if case == "gemm0":
        ok &= case_gemm(128, 256, 64, 256)
        ok &= case_gemm(128, 256, 256, 256)
        ok &= case_gemm(128, 128, 128, 128)
    elif case == "gemm1":
        ok &= case_gemm(256, 512, 1600, 256, act=1)
        ok &= case_gemm(1000, 1568, 1024, 256, act=2)
        ok &= case_gemm(8192, 1024, 1600, 256)
        ok &= case_gemm(384, 1024, 512, 128, act=1)
    elif case == "gemm2":
        ok &= case_gemm(72, 8, 40, 128)
        ok &= case_gemm(130, 264, 200, 256)
    elif case == "gemm_mask":
        ok &= case_gemm(512, 1024, 512, 256, epi=1, act=1)
        ok &= case_gemm(200, 520, 128, 128, epi=1, act=2)
    elif case == "gemm_red":
        ok &= case_gemm(512, 1024, 4096, 256, epi=2, splits=4)
        ok &= case_gemm(1024, 1600, 1024, 256, epi=2, splits=3)
        ok &= case_gemm(128, 128, 8192, 128, epi=2, splits=8)
    elif case == "features":
        from maze_b200.dqn_net import DQNNet
        net = DQNNet("cuda", max_batch=512, seed=1)
        b = make_batch(300, seed=2)
        src, _ = ref_nets(net)
        X, idx = net.features(b["vec"], b["pwin"], save_idx=True)
        with torch.no_grad():
            pre = torch.nn.functional.conv2d(b["win"], src.conv[0].weight.bfloat16().float(), src.conv[0].bias, padding=1)
            fw = torch.nn.functional.max_pool2d(torch.nn.functional.leaky_relu(pre, 0.01), 2, 2).flatten(1)
        ok &= report("features conv", X[:, :1568], fw, 1e-2)
        ok &= report("features vec", X[:, 1568:1574], b["vec"], 1e-2)
        ok &= report("features pad", X[:, 1574:], torch.zeros(300, 26, device="cuda"), 1e-6)
        # the pool choice must point at a maximal element and carry its sign
        pre_p = pre[:, :, :14, :14].reshape(300, 32, 7, 2, 7, 2).permute(0, 1, 2, 4, 3, 5).reshape(300, 32 * 49, 4)
        choice = (idx & 3).long()
        picked = pre_p.gather(2, choice.unsqueeze(-1)).squeeze(-1)
        ok &= report("features pool choice", picked, pre_p.max(-1)[0], 2e-2)
        sign_ok = (((idx >> 2) & 1).bool() == (picked > 0)) | (picked.abs() < 2e-2)
        print(("ok  " if sign_ok.all() else "FAIL") + f" features sign bit: mismatches {(~sign_ok).sum().item()}", flush=True)
        ok &= bool(sign_ok.all())
    elif case == "forward":
        from maze_b200.dqn_net import DQNNet
        net = DQNNet("cuda", max_batch=1024, seed=3)
        src, tgt = ref_nets(net)
        for n in (1, 37, 1000):
            b = make_batch(n, seed=n)
            q = net.forward(b["vec"], b["pwin"])
            with torch.no_grad():
                r = src((b["vec"], b["win"]))
            ok &= report(f"forward n={n}", q, r, 2e-2)
    elif case == "backward":
        from maze_b200.dqn_net import DQNNet
        from net_reference import ddqn_loss
        net = DQNNet("cuda", max_batch=1024, seed=4)
        # make the target differ from the source
        sd = net.state_dict("source")
        g = torch.Generator().manual_seed(9)
        net.load_state_dict({k: v + 0.01 * torch.randn(v.shape, generator=g).to(v.device) for k, v in sd.items()}, which="target")
        src, tgt = ref_nets(net)
        for n in (256, 1000):
            b = make_batch(n, seed=10 + n)
            net.grads.zero_()
            qsa = torch.zeros(n, device="cuda")
            net.backward(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], 0.9, qsa_out=qsa)
            src.zero_grad()
            loss, rq = ddqn_loss(src, tgt, (b["vec"], b["win"]), b["action"], b["reward"], (b["nvec"], b["nwin"]), 0.9)
            loss.backward()
            ok &= report(f"backward n={n} q(s,a)", qsa, rq.detach(), 2e-2)
            ok &= report(f"backward n={n} loss", net.loss, loss.detach().view(1), 3e-2)
            from maze_b200.dqn_net import _views
            gv = _views(net.grads)
            for name, p in src.named_parameters():
                got = gv[name]
                if name == "fc.0.weight":
                    ok &= report(f"backward n={n} grad {name} pad", got[:, 1574:], torch.zeros_like(got[:, 1574:]), 1e-9)
                    got = got[:, :1574]
                ok &= report(f"backward n={n} grad {name}", got.reshape(p.grad.shape), p.grad, 5e-2)
    elif case == "adamw":
        from maze_b200.dqn_net import DQNNet, _views
        from net_reference import ddqn_loss
        net = DQNNet("cuda", max_batch=512, seed=5)
        src, tgt = ref_nets(net)
        opt = torch.optim.AdamW(src.parameters(), 1e-3)
        for it in range(3):
            b = make_batch(512, seed=20 + it)
            before = {k: v.clone() for k, v in net.state_dict("source").items()}
            net.train_step(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma=0.9, lr=1e-3)
            loss, _ = ddqn_loss(src, tgt, (b["vec"], b["win"]), b["action"], b["reward"], (b["nvec"], b["nwin"]), 0.9)
            opt.zero_grad()
            loss.backward()
            for p in src.parameters():
                p.grad.data.clamp_(-1, 1)
            opt.step()
            after = net.state_dict("source")
            for name, p in src.named_parameters():
                ok &= report(f"adamw it{it} delta {name}", after[name] - before[name], p.detach() - before[name], 0.25)
            ok &= report(f"adamw it{it} grads zeroed", net.grads, torch.zeros_like(net.grads), 1e-12)
            # keep the two copies from drifting apart: continue from the device net's weights
            src.load_state_dict(after)
    elif case == "perf":
        from maze_b200.dqn_net import DQNNet, gemm_bf16
        out = {}
        for (M, N, K, tn) in ((8192, 1024, 1600, 256), (16384, 1024, 1600, 256), (16384, 512, 1024, 256), (8192, 1024, 1600, 128), (8192, 8192, 8192, 256),
                              (8192, 1024, 1600, 512), (16384, 1024, 1600, 512), (16384, 512, 1024, 512), (8192, 8192, 8192, 512)):
            A = torch.randn(M, K, device="cuda").bfloat16()
            B = torch.randn(N, K, device="cuda").bfloat16()
            Cc = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
            for _ in range(3):
                gemm_bf16(A, B, Cc, tile_n=tn)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                gemm_bf16(A, B, Cc, tile_n=tn)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 20
            e0.record()
            for _ in range(20):
                torch.matmul(A, B.t(), out=Cc)
            e1.record()
            torch.cuda.synchronize()
            ms_t = e0.elapsed_time(e1) / 20
            out[f"gemm_{M}x{N}x{K}_t{tn}"] = dict(ms=ms, tflops=2 * M * N * K / ms / 1e9, cublas_ms=ms_t, cublas_tflops=2 * M * N * K / ms_t / 1e9)
            print(f"perf gemm {M}x{N}x{K} tile{tn}: {ms:.4f} ms {2 * M * N * K / ms / 1e9:.1f} TFLOP/s (cuBLAS {ms_t:.4f} ms {2 * M * N * K / ms_t / 1e9:.1f})", flush=True)
        for n in (8192,):
            net = DQNNet("cuda", max_batch=n, seed=6)
            b = make_batch(n, seed=30)
            for _ in range(3):
                net.forward(b["vec"], b["pwin"])
                net.train_step(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma=0.9, lr=1e-4)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                net.forward(b["vec"], b["pwin"])
            e1.record()
            torch.cuda.synchronize()
            ms_f = e0.elapsed_time(e1) / 20
            e0.record()
            for _ in range(20):
                net.train_step(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma=0.9, lr=1e-4)
            e1.record()
            torch.cuda.synchronize()
            ms_t = e0.elapsed_time(e1) / 20
            fwd_flop = 2 * (225 * 32 * 27 + 1574 * 1024 + 1024 * 512 + 512 * 4)
            out[f"net_n{n}"] = dict(forward_ms=ms_f, forward_tflops=fwd_flop * n / ms_f / 1e9, train_ms=ms_t,
                                   train_tflops=5 * fwd_flop * n / ms_t / 1e9, samples_per_s=n / ms_t * 1e3)
            print(f"perf net n={n}: forward {ms_f:.3f} ms ({fwd_flop * n / ms_f / 1e9:.1f} TFLOP/s), train step {ms_t:.3f} ms "
                  f"({5 * fwd_flop * n / ms_t / 1e9:.1f} TFLOP/s, {n / ms_t * 1e3:.3g} samples/s)", flush=True)
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        json.dump(out, open(os.path.join(ROOT, "gpurun_out", "net_perf.json"), "w"), indent=1)
    elif case == "profile":   # in-situ launch times of the backward pass (CUDA events between the launches)
        from maze_b200.dqn_net import DQNNet
        n = int(os.environ.get("NET_BATCH", "8192"))
        net = DQNNet("cuda", max_batch=n, seed=6)
        b = make_batch(n, seed=30)
        net.profile(True)
        acc = {}
        order = []
        reps = 20
        for it in range(reps + 5):
            net.forward(b["vec"], b["pwin"])
            net.train_step(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma=0.9, lr=1e-4)
            rows = net.profile_read()
            if it >= 5:
                for i, (label, ms) in enumerate(rows):
                    key = (i, label)
                    if key not in acc:
                        acc[key] = []
                        order.append(key)
                    acc[key].append(ms)
        net.profile(False)
        total = 0.0
        lines = []
        by_label = {}
        for key in order:
            v = sorted(acc[key])
            med = v[len(v) // 2]
            total += med
            by_label.setdefault(key[1], [0.0, 0])
            by_label[key[1]][0] += med
            by_label[key[1]][1] += 1
        for label, (ms, cnt) in by_label.items():
            lines.append(f"{ms * 1e3:9.1f} us  {cnt:3d} x  {label}")
        lines.append(f"{total * 1e3:9.1f} us  backward pass, sum of medians over {reps} steps (n = {n})")
        print("\n".join(lines), flush=True)
    elif case == "trainloop":   # a short loop for the ncu launch list
        from maze_b200.dqn_net import DQNNet
        n = int(os.environ.get("NET_BATCH", "8192"))
        net = DQNNet("cuda", max_batch=n, seed=6)
        b = make_batch(n, seed=30)
        for _ in range(6):
            net.forward(b["vec"], b["pwin"])
            net.train_step(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma=0.9, lr=1e-4)
    else:
        raise SystemExit(f"unknown case {case}")
    torch.cuda.synchronize()
    print(("CASE ok   " if ok else "CASE FAIL ") + case, flush=True)
    return ok


def main():
    if len(sys.argv) > 1:
        sys.exit(0 if run_case(sys.argv[1]) else 1)
    failed = []
    for c in CASES:
        t0 = time.time()
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), c], timeout=240)
            rc = r.returncode
        except subprocess.TimeoutExpired:
            rc = "timeout"
        print(f"== {c}: rc {rc} in {time.time() - t0:.0f}s", flush=True)
        if rc != 0:
            failed.append(c)
    print("SELFTEST", "ok" if not failed else f"FAILED {failed}", flush=True)
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
