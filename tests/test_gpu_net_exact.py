"""The tensor-core DQN net (csrc/maze_net.cu) against the bf16-faithful float64 reference (tests/net_bf16_reference.py):
bit for bit where the operands make every fp32 sum exact, and at the production batch (n = 8192) with tolerances an
order of magnitude tighter than test_gpu_net.py's, tight enough to see one lost 128-sample tile.

Measured on a B200 (1000 W power limit), worst case over every parameter set and switch; TOL holds the bounds:
  forward q: row error / max |q|                       2.0e-3   (TOL 5e-3)
  q(s, a): error / max |q(s, a)|                       1.6e-3   (TOL 4e-3)
  loss: relative                                       9.5e-5   (TOL 3e-4)
  gradients, relative Frobenius error: conv, fc1, fc2  4.8e-3   (TOL 1e-2; one lost 128-sample tile at n = 8192: >= 2.5e-2)
                                       fc3             5.4e-4   (TOL 1.5e-3)
  AdamW parameters: error / lr                         2.9e-5   (TOL 1e-4)
  features with the default init: bit-exact (no entry 1 ulp off, no pool choice different)
"""
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import net_bf16_reference as nbr  # noqa: E402
from net_reference import pack_windows  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMS = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148

# Bounds from measurement (see the module docstring).  A gradient passes at relative Frobenius error <= TOL[name] and no
# entry off by more than WORST_FACTOR TOL[name] of the tensor's largest magnitude.  The per-entry bound is wider because a
# sample whose ReLU / LeakyReLU pre-activation lies within fp32 accumulation error of 0 can take the other mask in the
# kernel, which moves one column of dW2 and gb2 by that sample's whole share: 1 / n of the batch, measured 2.8e-2 of the
# largest entry at n = 200.
TOL = {"q": 5e-3, "qsa": 4e-3, "loss": 3e-4, "conv.0.weight": 1e-2, "conv.0.bias": 1e-2, "fc.0.weight": 1e-2, "fc.0.bias": 1e-2,
       "fc.2.weight": 1e-2, "fc.2.bias": 1e-2, "fc.4.weight": 1.5e-3, "fc.4.bias": 1.5e-3, "adamw": 1e-4}
WORST_FACTOR = 6
KNIFE_EDGE_RATE = 1e-3      # at most this share of pool choices / activation signs / arg-maxes may sit on a knife edge


def _report(what, value):
    print(f"MEASURED {what} {value:.3e}")


@pytest.fixture(autouse=True)
def _no_tf32():
    a, b = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = a, b


def _batch(n, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    win = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).float()
    nwin = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).float()
    vec, nvec = torch.rand(n, 6, generator=g), torch.rand(n, 6, generator=g)
    action = torch.randint(0, 4, (n,), generator=g).to(torch.uint8)
    reward = torch.rand(n, generator=g) - 0.5
    b = dict(vec=vec, win=win, nvec=nvec, nwin=nwin, action=action, reward=reward)
    b = {k: v.cuda() for k, v in b.items()}
    b["pwin"], b["pnwin"] = pack_windows(b["win"]), pack_windows(b["nwin"])
    return b


def _make_net(max_batch, seed=11):
    """Source net from the default init, target net = source + 1 % noise (both from CPU generators)."""
    from maze_b200.dqn_net import DQNNet
    net = DQNNet("cuda", max_batch=max_batch, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    net.load_state_dict({k: v + 0.01 * torch.randn(v.shape, generator=g).to(v.device) for k, v in net.state_dict("source").items()}, which="target")
    return net


def _weights(sd):
    return nbr.NetWeights(sd, nbr.Rounding(True))


def _sd_from_flat(flat):
    from maze_b200.dqn_net import _views
    sd = {k: v.clone() for k, v in _views(flat).items()}
    sd["fc.0.weight"] = sd["fc.0.weight"][:, :1574]
    return sd


def _rel(got, ref):
    got, ref = got.double(), ref.double()
    rel = ((got - ref).norm() / ref.norm().clamp_min(1e-300)).item()
    worst = ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()
    return rel, worst


def _check_grad(name, got, ref, what):
    rel, worst = _rel(got, ref)
    _report(f"{what} {name} frob", rel)
    _report(f"{what} {name} worst", worst)
    assert rel <= TOL[name] and worst <= WORST_FACTOR * TOL[name], f"{what} {name}: relative Frobenius error {rel:.3g}, worst entry {worst:.3g} (tol {TOL[name]})"


def _reference_backward(sd_src, sd_tgt, b, gamma=0.9, tc=True, keep=None):
    return nbr.ddqn_backward(_weights(sd_src), _weights(sd_tgt), b["vec"], b["win"], b["nvec"], b["nwin"], b["action"], b["reward"], gamma,
                             tc=tc, keep=keep)


def _check_backward(loss, qsa, grads_flat, ref, what):
    """Every output of maze_dqn_backward against the reference; then that knife edges were rare."""
    from maze_b200.dqn_net import _views
    n = qsa.shape[0]
    e_q = ((qsa.double() - ref["qsa"]).abs().max() / ref["qsa"].abs().max()).item()
    e_l = abs(loss - ref["loss"].item()) / ref["loss"].item()
    _report(f"{what} qsa", e_q)
    _report(f"{what} loss", e_l)
    gv = _views(grads_flat)
    assert (gv["fc.0.weight"][:, 1574:] == 0).all(), f"{what}: fc1 weight gradient padding columns"
    for name, r in ref["grads"].items():
        got = gv[name][:, :1574] if name == "fc.0.weight" else gv[name]
        _check_grad(name, got, r, what)
    assert e_q <= TOL["qsa"], (what, e_q)
    assert e_l <= TOL["loss"], (what, e_l)
    assert ref["argmax_near"].sum().item() <= max(1, KNIFE_EDGE_RATE * n), (what, ref["argmax_near"].sum().item())
    for f in ("fs", "fn", "ft"):
        for key in ("pool_near", "act_near", "h1_near", "h2_near"):
            rate = ref[f][key].double().mean().item()
            assert rate <= KNIFE_EDGE_RATE, (what, f, key, rate)


# ---- a. the GEMM hook, bit for bit ------------------------------------------------------------------------------
# Operands are k / 8 (|k| <= 8), bias and accumulated-onto C multiples of 1 / 64 in [-1, 1]: every product is a multiple
# of 1 / 64 and every partial sum s satisfies |s| * 64 <= (K + 2) * 64 < 2^24 (K <= 8200), so fp32 holds every partial sum
# exactly, in any order and over any split-K partition, and C must equal the float64 result rounded as the epilogue
# rounds (maze_net.cu:119-143).
def _grid(shape, g, denom=8, lim=8):
    return (torch.randint(-lim, lim + 1, shape, generator=g).double() / denom).cuda()


def _padded(rows, cols, pad, dtype, fill):
    """A [rows, cols] view with row pitch cols + pad of a tensor whose padding holds `fill`."""
    full = torch.full((rows, cols + pad), fill, dtype=dtype, device="cuda")
    return full, full[:, :cols]


SENTINEL = 96.0   # bf16- and fp32-exact; outside every product and sum a k / 8 operand can form in a padding column


@pytest.mark.parametrize("M,N,K,tile,act,bias,pad_a,pad_c", [
    (1, 8, 8, 128, 0, True, 0, 0), (127, 24, 40, 128, 1, True, 8, 8), (129, 1568, 1000, 128, 2, False, 0, 32),
    (8200, 1568, 40, 128, 0, True, 0, 0),                                   # 845 tiles: persistent walk over the SMs
    (127, 1568, 40, 256, 0, True, 0, 0), (257, 24, 40, 256, 1, False, 24, 0), (8200, 24, 1000, 256, 2, True, 0, 8),
    (1, 24, 8, 512, 1, True, 0, 0), (129, 8, 1000, 512, 2, True, 8, 0),
    (257, 1568, 1000, 512, 0, False, 0, 32),                                # the dX GEMM: no bias, ldc 1600 > N
    (8200, 1568, 40, 512, 1, True, 0, 0)])                                  # 231 pair tiles > SMs / 2
def test_gemm_bias_act_exact(M, N, K, tile, act, bias, pad_a, pad_c):
    from maze_b200.dqn_net import gemm_bf16
    g = torch.Generator().manual_seed(M * 7 + N + K + tile + act)
    _, A = _padded(M, K, pad_a, torch.bfloat16, SENTINEL)
    A.copy_(_grid((M, K), g))
    B = _grid((N, K), g).bfloat16()
    bv = _grid((N,), g, denom=64, lim=64).float() if bias else None
    Cfull, C = _padded(M, N, pad_c, torch.bfloat16, SENTINEL)
    gemm_bf16(A, B, C, 0, act, bias=bv, tile_n=tile)
    x = A.double() @ B.double().t() + (bv.double() if bias else 0.0)
    if act == 1:
        x = torch.where(x > 0, x, (x * nbr.SLOPE_F32).float().double())
    elif act == 2:
        x = x.clamp_min(0.0)
    assert torch.equal(C, x.float().bfloat16()), f"{(C.double() != x.float().bfloat16().double()).sum().item()} entries differ"
    assert (Cfull[:, N:] == SENTINEL).all(), "columns past N were written"


@pytest.mark.parametrize("M,N,K,tile,act,pad_a,pad_c", [
    (127, 24, 40, 128, 1, 0, 8), (129, 1568, 1000, 128, 2, 8, 0),
    (257, 1568, 40, 256, 1, 0, 0), (1, 8, 8, 256, 2, 0, 0),
    (8200, 1568, 40, 512, 1, 0, 32),                                        # the net's dh1 GEMM mode at the pair tile
    (257, 24, 1000, 512, 2, 8, 8), (129, 1568, 8, 512, 1, 0, 0)])
def test_gemm_mask_exact(M, N, K, tile, act, pad_a, pad_c):
    """EPI_MASK: C = acc * act'(aux), the derivative taken from the sign of the stored bf16 activation; +0 and -0 take
    the negative slope (the LeakyReLU slope 0.01f, or 0 for ReLU)."""
    from maze_b200.dqn_net import gemm_bf16
    g = torch.Generator().manual_seed(M * 5 + N + K + tile + act)
    _, A = _padded(M, K, pad_a, torch.bfloat16, SENTINEL)
    A.copy_(_grid((M, K), g))
    B = _grid((N, K), g).bfloat16()
    aux = _grid((M, N), g, denom=4, lim=2).bfloat16()
    aux[torch.rand(M, N, generator=g).cuda() < 0.1] = -0.0
    assert (aux == 0).any() and (aux.view(torch.int16) == -32768).any()
    Cfull, C = _padded(M, N, pad_c, torch.bfloat16, SENTINEL)
    gemm_bf16(A, B, C, 1, act, aux=aux, tile_n=tile)
    neg = nbr.SLOPE_F32 if act == 1 else 0.0
    x = ((A.double() @ B.double().t()) * torch.where(aux.double() > 0, 1.0, neg)).float()
    assert torch.equal(C, x.bfloat16()), f"{(C.double() != x.bfloat16().double()).sum().item()} entries differ"
    assert (Cfull[:, N:] == SENTINEL).all(), "columns past N were written"


@pytest.mark.parametrize("K,M,N,tile,splits,pad_a,pad_c", [
    (1000, 24, 1568, 128, 3, 0, 0),          # 16 k-blocks in 3 uneven splits
    (40, 8200, 24, 256, 4, 8, 8),            # one (zero-filled) k-block: splits clamped to 1
    (1000, 1568, 24, 256, 5, 0, 32), (200, 8, 1568, 256, 7, 0, 0),   # 4 k-blocks, 7 splits -> 4
    (8200, 24, 1568, 128, 6, 0, 0),          # K = batch 8200: 129 k-blocks, the last one 8 rows
    (1000, 1024, 1600, 256, 5, 8, 0)])       # the fc1 weight gradient's shape: 280 tiles
def test_gemm_mn_major_split_k_exact(K, M, N, tile, splits, pad_a, pad_c):
    """C += A^T . B from [K, M] / [K, N] operands (the weight gradients), split-K partial sums added with red.add onto a
    non-zero C."""
    from maze_b200.dqn_net import gemm_bf16
    g = torch.Generator().manual_seed(K + M * 3 + N + splits)
    _, A = _padded(K, M, pad_a, torch.bfloat16, SENTINEL)
    A.copy_(_grid((K, M), g))
    B = _grid((K, N), g).bfloat16()
    Cfull, C = _padded(M, N, pad_c, torch.float32, SENTINEL)
    C.copy_(_grid((M, N), g, denom=64, lim=64))
    ref = (C.double() + A.double().t() @ B.double()).float()
    gemm_bf16(A, B, C, 3, 0, tile_n=tile, splits=splits)
    assert torch.equal(C, ref), f"{(C != ref).sum().item()} entries differ"
    assert (Cfull[:, N:] == SENTINEL).all(), "columns past N were written"


def test_gemm_k_major_split_k_exact():
    from maze_b200.dqn_net import gemm_bf16
    g = torch.Generator().manual_seed(3)
    A, B = _grid((129, 1000), g).bfloat16(), _grid((24, 1000), g).bfloat16()
    C = _grid((129, 24), g, denom=64, lim=64).float()
    ref = (C.double() + A.double() @ B.double().t()).float()
    gemm_bf16(A, B, C, 2, 0, tile_n=128, splits=3)
    assert torch.equal(C, ref)


# ---- b. features, bit for bit ------------------------------------------------------------------------------------
FEATURE_NS = [1, 2, 3, 8 * SMS - 1, 8 * SMS, 8 * SMS + 1, 4097, 8192]   # above 8 SMs: every CTA walks a second pair


@pytest.fixture(scope="module")
def dyadic_net():
    """Conv weights and bias on multiples of 2^-6 in [-0.25, 0.25], different for source and target: every conv sum is
    exact in fp32 and pool ties are frequent."""
    net = _make_net(8, seed=21)
    g = torch.Generator().manual_seed(22)
    for which in ("source", "target"):
        sd = net.state_dict(which)
        sd["conv.0.weight"] = torch.randint(-16, 17, (32, 3, 3, 3), generator=g).float() / 64
        sd["conv.0.bias"] = torch.randint(-16, 17, (32,), generator=g).float() / 64
        net.load_state_dict(sd, which=which)
    return net


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("n", FEATURE_NS)
def test_features_exact(dyadic_net, n, which):
    b = _batch(n, 1000 + n)
    X, idx = dyadic_net.features(b["vec"], b["pwin"], which=which, save_idx=True)
    ref = nbr.features(_weights(dyadic_net.state_dict("target" if which else "source")), b["vec"], b["win"])
    assert ref["pool_ties"] > 0 and not ref["pool_near"].any()
    assert torch.equal(idx, ref["idx"]), f"{(idx != ref['idx']).sum().item()} pool choices differ"
    assert torch.equal(X[:, :1574].double(), ref["X"]), f"{(X[:, :1574].double() != ref['X']).sum().item()} features differ"
    assert (X[:, 1574:] == 0).all()


@pytest.mark.parametrize("n", [8 * SMS + 1, 8192])
def test_features_default_init_within_one_ulp(n):
    net = _make_net(8, seed=23)
    b = _batch(n, 2000 + n)
    X, idx = net.features(b["vec"], b["pwin"], save_idx=True)
    ref = nbr.features(_weights(net.state_dict("source")), b["vec"], b["win"])
    edge = ref["pool_near"] | ref["act_near"]
    assert edge.double().mean().item() <= KNIFE_EDGE_RATE
    assert torch.equal(idx[~edge], ref["idx"][~edge])
    got, want = X[:, :1568].view(torch.int16).int(), ref["X"][:, :1568].float().bfloat16().view(torch.int16).int()
    ulps = (got - want).abs()
    assert (ulps[~edge] <= 1).all(), ulps.max().item()
    _report(f"features n={n} entries 1 ulp off", (ulps == 1).double().mean().item())
    assert torch.equal(X[:, 1568:1574].double(), ref["X"][:, 1568:])


# ---- c. forward --------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def net8192():
    return _make_net(8192)


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("n", [1, 7, 128, 129, 4736, 4737, 8192])
def test_forward_matches_bf16_reference(net8192, n, which):
    """n = 129: the first pair-tile batch; 4737 > 32 SMs: net_head_q_kernel's sample loop takes a second turn."""
    b = _batch(n, 3000 + n)
    q = net8192.forward(b["vec"], b["pwin"], which=which)
    ref = nbr.forward(_weights(net8192.state_dict("target" if which else "source")), b["vec"], b["win"])
    err = ((q.double() - ref["q"]).abs().max(1)[0] / ref["q"].abs().max()).max().item()
    _report(f"forward n={n} which={which}", err)
    assert err <= TOL["q"]


# ---- d. backward -------------------------------------------------------------------------------------------------
SENSITIVE = ("conv.0.weight", "conv.0.bias", "fc.0.weight", "fc.0.bias", "fc.2.weight", "fc.2.bias")


def _run_backward(net, b, gamma=0.9):
    n = b["vec"].shape[0]
    net.grads.zero_()
    qsa = torch.zeros(n, device="cuda")
    net.backward(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma, qsa_out=qsa)
    return net.loss.item(), qsa, net.grads.clone()


@pytest.mark.parametrize("n", [8, 200, 1000, 16 * SMS + 8, 16 * SMS + 16, 8192])
def test_backward_matches_bf16_reference(net8192, n):
    """n not a multiple of 64: the k-block and column-sum tails; n > 16 SMs: the head-loss kernel's warps take a second
    sample (its prefetch); n = 8192: the production batch, split-K 5 (fc1) and 8 (fc2).  At 8192 the reference without one
    128-sample block must fail every tolerance: a lost tile would not pass."""
    b = _batch(n, 4000 + n)
    loss, qsa, grads = _run_backward(net8192, b)
    ref = _reference_backward(net8192.state_dict("source"), net8192.state_dict("target"), b)
    _check_backward(loss, qsa, grads, ref, f"backward n={n}")
    if n == 8192:
        keep = torch.ones(n, device="cuda")
        keep[17 * 128:18 * 128] = 0.0
        lost = _reference_backward(net8192.state_dict("source"), net8192.state_dict("target"), b, keep=keep)
        moved = {name: _rel(lost["grads"][name], ref["grads"][name])[0] for name in SENSITIVE}
        for name, rel in moved.items():
            _report(f"lost tile {name}", rel)
        for name, rel in moved.items():
            assert rel > TOL[name], f"{name}: a lost 128-sample tile moves the gradient by {rel:.3g}, within the tolerance {TOL[name]}"


def test_backward_after_a_larger_batch(net8192):
    """The workspace still holds the rows of an n = 8192 call: an n = 200 call must not read any of them."""
    _run_backward(net8192, _batch(8192, 5))
    b = _batch(200, 6)
    loss, qsa, grads = _run_backward(net8192, b)
    _check_backward(loss, qsa, grads, _reference_backward(net8192.state_dict("source"), net8192.state_dict("target"), b), "stale workspace")


def test_double_q_exact_tie_takes_the_first_action():
    """Source rows 1 and 2 of fc3 equal (weights and bias, above the others): q_source(s', 1) == q_source(s', 2) for every
    sample, and the first maximum, action 1, picks the target row.  Target rows 1 and 2 differ, so the other choice
    would change the loss by far more than its tolerance."""
    net = _make_net(1000, seed=31)
    sd = net.state_dict("source")
    sd["fc.4.weight"][2] = sd["fc.4.weight"][1]
    sd["fc.4.bias"][1] = sd["fc.4.bias"][2] = sd["fc.4.bias"].max() + 1.0
    net.load_state_dict(sd, which="source")
    tsd = net.state_dict("target")
    tsd["fc.4.bias"][2] = tsd["fc.4.bias"][1] + 0.5
    net.load_state_dict(tsd, which="target")
    b = _batch(1000, 7)
    loss, qsa, grads = _run_backward(net, b)
    ref = _reference_backward(net.state_dict("source"), tsd, b)
    assert (ref["best"] == 1).all()
    _check_backward(loss, qsa, grads, ref, "exact tie")
    qt2 = ref["ft"]["q"][:, 2] * 0.9 + b["reward"].double()
    other = ((ref["qsa"] - qt2) ** 2).mean().item()
    assert abs(other - ref["loss"].item()) > 10 * TOL["loss"] * ref["loss"].item()


# ---- e. the A/B switches, each in a process of its own (the kernels read them once per process) ---------------------
def _child_main(out, ns, adam_step):
    """Run in a subprocess: backward (and forward) at each n on a fixed net and batches; with adam_step also AdamW, then
    a second backward with the updated weights.  Writes the results to `out` (.npz)."""
    net = _make_net(max(ns))
    res = {}
    for n in ns:
        b = _batch(n, 4000 + n)
        loss, qsa, grads = _run_backward(net, b)
        res[f"loss{n}"], res[f"qsa{n}"], res[f"grads{n}"] = np.float64(loss), qsa.cpu().numpy(), grads.cpu().numpy()
        res[f"q{n}"] = net.forward(b["vec"], b["pwin"]).cpu().numpy()
    if adam_step:
        n = ns[-1]
        net.backward(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], 0.9)   # grads accumulate: 2 x
        res["grads_acc"] = net.grads.cpu().numpy()
        net.adamw(1e-3, grad_scale=0.5)
        res["params1"], res["m1"], res["v1"] = net.params.cpu().numpy(), net.adam_m.cpu().numpy(), net.adam_v.cpu().numpy()
        b2 = _batch(n, 9000)
        loss, qsa, grads = _run_backward(net, b2)
        res["loss_2"], res["qsa_2"], res["grads_2"] = np.float64(loss), qsa.cpu().numpy(), grads.cpu().numpy()
    torch.cuda.synchronize()
    np.savez(out, **res)


def _run_child(tmp_path, env, ns, adam_step=False):
    out = str(tmp_path / "out.npz")
    code = (f"import test_gpu_net_exact as t; t._child_main({out!r}, {list(ns)!r}, {adam_step!r})")
    e = dict(os.environ)
    e.update(env)
    e["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "tests"), ROOT, os.path.join(ROOT, "maze-solving-agent-gymnasium_b200")])
    p = subprocess.run([sys.executable, "-c", code], env=e, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    return dict(np.load(out))


def _check_child(res, ns, tc=True, what=""):
    net = _make_net(8)
    src, tgt = net.state_dict("source"), net.state_dict("target")
    for n in ns:
        b = _batch(n, 4000 + n)
        ref = _reference_backward(src, tgt, b, tc=tc)
        _check_backward(float(res[f"loss{n}"]), torch.from_numpy(res[f"qsa{n}"]).cuda(), torch.from_numpy(res[f"grads{n}"]).cuda(), ref,
                        f"{what} n={n}")
        q = torch.from_numpy(res[f"q{n}"]).cuda().double()
        assert ((q - ref["fs"]["q"]).abs().max() / ref["fs"]["q"].abs().max()).item() <= TOL["q"]
    return src, tgt


def test_conv_gradient_on_cuda_cores(tmp_path):
    """MAZE_NET_CONV_BWD_CUDA_CORES=1: net_conv_bwd_kernel, which keeps gv * 0.01f in fp32 (the reference's tc=False)."""
    ns = [200, 8192]
    _check_child(_run_child(tmp_path, {"MAZE_NET_CONV_BWD_CUDA_CORES": "1"}, ns), ns, tc=False, what="cuda-core conv gradient")


def test_without_cta_pairs(tmp_path):
    ns = [1000, 8192]
    _check_child(_run_child(tmp_path, {"MAZE_NET_NO_PAIRS": "1"}, ns), ns, what="no pairs")


def test_forward_in_256_row_chunks(tmp_path):
    """MAZE_NET_CHUNK_ROWS=256: at n = 1000 the last chunk has 232 rows."""
    ns = [1000, 8192]
    _check_child(_run_child(tmp_path, {"MAZE_NET_CHUNK_ROWS": "256"}, ns), ns, what="chunks of 256")


def test_programmatic_dependent_launch(tmp_path):
    """MAZE_NET_PDL=1: every kernel of the train step may start before its predecessor has finished and waits in
    griddepcontrol.wait; one that touched global memory before its wait would race.  Backward, AdamW and a second
    backward with the refreshed weights, at n = 8192."""
    n = 8192
    res = _run_child(tmp_path, {"MAZE_NET_PDL": "1"}, [n], adam_step=True)
    src, tgt = _check_child(res, [n], what="PDL")
    # the second backward accumulated onto the first: twice the gradient
    g1, gacc = torch.from_numpy(res[f"grads{n}"]).cuda(), torch.from_numpy(res["grads_acc"]).cuda()
    rel, _ = _rel(gacc, 2 * g1)
    assert rel <= 1e-5, rel
    p0 = _make_net(8).params
    p1, m1, v1 = _adamw_reference(p0.double(), gacc.double(), torch.zeros_like(gacc, dtype=torch.float64), torch.zeros_like(gacc, dtype=torch.float64),
                                  step=1, lr=1e-3, wd=1e-2, grad_scale=0.5, clamp=1.0)
    _check_adamw(torch.from_numpy(res["params1"]).cuda(), p1, 1e-3, "PDL adamw")
    b2 = _batch(n, 9000)
    ref = _reference_backward(_sd_from_flat(torch.from_numpy(res["params1"]).cuda()), tgt, b2)
    _check_backward(float(res["loss_2"]), torch.from_numpy(res["qsa_2"]).cuda(), torch.from_numpy(res["grads_2"]).cuda(), ref, "PDL step 2")


# ---- f. AdamW ----------------------------------------------------------------------------------------------------
def _f32(x):
    return float(np.float32(x))


def _adamw_reference(p, g, m, v, step, lr, wd, grad_scale, clamp, betas=(0.9, 0.999), eps=1e-8):
    """torch.optim.AdamW's update in float64, on the fp32 values of the hyper-parameters the kernel receives."""
    b1, b2, lr, eps, wd = _f32(betas[0]), _f32(betas[1]), _f32(lr), _f32(eps), _f32(wd)
    gr = g * _f32(grad_scale)
    if clamp > 0:
        gr = gr.clamp(-clamp, clamp)
    m = b1 * m + (1 - b1) * gr
    v = b2 * v + (1 - b2) * gr * gr
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    p = p * (1 - lr * wd) - (lr / bc1) * m / (v.sqrt() / bc2 ** 0.5 + eps)
    return p, m, v


def _check_adamw(got, ref, lr, what):
    err = ((got.double() - ref).abs().max() / lr).item()
    _report(what, err)
    assert err <= TOL["adamw"], (what, err)


def test_adamw_grad_scale_no_clamp_late_step():
    """grad_scale = 1/8 (a world of eight ranks), the clamp off (|g / 8| > 1 on many entries), no weight decay, step 10 000
    (bias corrections from powf of a large exponent), non-zero moments."""
    from maze_b200.dqn_net import DQNNet
    net = DQNNet("cuda", max_batch=8, seed=41)
    g = torch.Generator().manual_seed(42)
    P = net.params.numel()
    net.grads.copy_(torch.randn(P, generator=g) * 16)
    net.adam_m.copy_(torch.randn(P, generator=g))
    net.adam_v.copy_(torch.rand(P, generator=g) * 4)
    p0, g0, m0, v0 = (t.double().clone() for t in (net.params, net.grads, net.adam_m, net.adam_v))
    assert ((g0 / 8).abs() > 1).any()
    net.step_count = 9_999
    net.adamw(1e-3, weight_decay=0.0, grad_scale=1 / 8, clamp=0.0)
    p1, m1, v1 = _adamw_reference(p0, g0, m0, v0, step=10_000, lr=1e-3, wd=0.0, grad_scale=1 / 8, clamp=0.0)
    gr = g0 / 8   # fp32 rounding of a two-term sum: a few ulps of the terms' magnitudes
    b1, b2 = _f32(0.9), _f32(0.999)
    assert ((net.adam_m.double() - m1).abs() <= 1e-6 * (b1 * m0.abs() + (1 - b1) * gr.abs())).all()
    assert ((net.adam_v.double() - v1).abs() <= 1e-6 * (b2 * v0 + (1 - b2) * gr * gr)).all()
    _check_adamw(net.params, p1, 1e-3, "adamw step 10000")
    assert (net.grads == 0).all()


def test_padding_columns_stay_zero_over_train_steps():
    from maze_b200.dqn_net import _views
    net = _make_net(256, seed=43)
    b = _batch(256, 44)
    for _ in range(20):
        net.train_step(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma=0.9, lr=1e-3)
    for flat in (net.params, net.adam_m, net.adam_v):
        pad = _views(flat)["fc.0.weight"][:, 1574:]
        assert (pad == 0).all()
    assert (_views(net.adam_v)["fc.0.weight"][:, :1574] > 0).any()
