"""The net's Dropout and the DQN target (csrc/maze_net.cu) against the bf16-faithful float64 reference with the modelled
keep masks (tests/net_dropout_reference.py), and against plain fp32 autograd through a fixed-mask Dropout.

The defaults (dropout 0, double-Q) are bit-identical to a net built without the new arguments; with p = 0.2 the features
are bit-exact against the model; forward, DDQN and DQN backward stay within test_gpu_net_exact.py's TOL table.  (The
loss and the gradients are summed with atomics, so even two runs of one net agree on them only to the last bits.)"""
import json
import os
import subprocess
import sys

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import net_dropout_reference as ndr  # noqa: E402
from net_reference import RefDQN, ddqn_loss  # noqa: E402
from test_gpu_net_exact import KNIFE_EDGE_RATE, SMS, TOL, _batch, _check_backward, _report, _weights  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 0.2


@pytest.fixture(autouse=True)
def _no_tf32():
    a, b = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = a, b


def _net(max_batch, seed=11, dyadic=False, **kw):
    """test_gpu_net_exact._make_net with the new arguments: source from the default init, target = source + 1 % noise;
    dyadic: conv weights and bias on multiples of 2^-6 (every conv sum exact in fp32)."""
    from maze_b200.dqn_net import DQNNet
    net = DQNNet("cuda", max_batch=max_batch, seed=seed, **kw)
    g = torch.Generator().manual_seed(seed + 1)
    net.load_state_dict({k: v + 0.01 * torch.randn(v.shape, generator=g).to(v.device) for k, v in net.state_dict("source").items()}, which="target")
    if dyadic:
        g = torch.Generator().manual_seed(seed + 2)
        for which in ("source", "target"):
            sd = net.state_dict(which)
            sd["conv.0.weight"] = torch.randint(-16, 17, (32, 3, 3, 3), generator=g).float() / 64
            sd["conv.0.bias"] = torch.randint(-16, 17, (32,), generator=g).float() / 64
            net.load_state_dict(sd, which=which)
    return net


def _drop(net, fwd, n, draw=None):
    return ndr.Drop(ndr.keep_mask(net._c.dropout_seed, net.draw if draw is None else draw, fwd, n, P), P)


def _backward(net, b, gamma=0.9):
    n = b["vec"].shape[0]
    net.grads.zero_()
    qsa = torch.zeros(n, device="cuda")
    net.backward(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma, qsa_out=qsa)
    return net.loss.item(), qsa, net.grads.clone()


# ---- 1. explicit defaults == defaults, bit for bit -------------------------------------------------------------------
def test_explicit_defaults_are_bitwise_the_default_net():
    n = 2048
    a, b_ = _net(n, seed=13), _net(n, seed=13, dropout=0.0, double_q=True)
    b = _batch(n, 77)
    outs = []
    for net in (a, b_):
        net.profile(True)
        X, idx = net.features(b["vec"], b["pwin"], save_idx=True)
        q = net.forward(b["vec"], b["pwin"])
        loss, qsa, grads = _backward(net, b)
        labels = [lab for lab, _ in net.profile_read()]
        net.profile(False)
        outs.append((X, idx, q, loss, qsa, grads, labels))
    (X0, i0, q0, l0, s0, g0, lab0), (X1, i1, q1, l1, s1, g1, lab1) = outs
    assert torch.equal(X0.view(torch.int16), X1.view(torch.int16)) and torch.equal(i0, i1)
    assert ((i0 & 8) == 0).all()
    assert torch.equal(q0, q1) and torch.equal(s0, s1)
    # the loss and the gradients are summed with atomics, whose order varies from run to run: two runs of one net differ
    # in the last bits too, so these are held to that spread
    assert abs(l0 - l1) <= 1e-6 * abs(l0)
    assert ((g0 - g1).norm() / g0.norm()).item() <= 1e-5
    assert lab0 == lab1 and sum(lab.startswith("features") for lab in lab0) == 3 and not any("dropout" in lab for lab in lab0)


# ---- 2. features with dropout, bit for bit ------------------------------------------------------------------------
@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("n,dyadic", [(8192, True), (8 * SMS + 1, True), (8192, False), (8 * SMS + 1, False)])
def test_dropout_features_exact(n, dyadic, which):
    net = _net(8, seed=21, dyadic=dyadic, dropout=P)
    net.features(_batch(2, 1)["vec"], _batch(2, 1)["pwin"])          # draw 0 used: the tested call runs at draw 1
    b = _batch(n, 1000 + n)
    drop = _drop(net, ndr.FWD_STANDALONE, n)
    X, idx = net.features(b["vec"], b["pwin"], which=which, save_idx=True)
    ref = ndr.features(_weights(net.state_dict("target" if which else "source")), b["vec"], b["win"], drop)
    dropped = ((idx & 8) != 0).double().mean().item()
    _report(f"dropout features n={n} dyadic={dyadic} winners dropped", dropped)
    assert 0.0 < dropped < 0.2
    if dyadic:
        assert not ref["pool_near"].any()
        edge = torch.zeros_like(ref["pool_near"])
    else:
        edge = ref["pool_near"] | ref["act_near"]
        assert edge.double().mean().item() <= KNIFE_EDGE_RATE
    assert torch.equal(idx[~edge], ref["idx"][~edge]), f"{(idx != ref['idx']).sum().item()} pool choices differ"
    got = X[:, :1574].double()
    assert torch.equal(got[:, :1568][~edge], ref["X"][:, :1568][~edge]), f"{(got != ref['X']).sum().item()} features differ"
    assert torch.equal(got[:, 1568:], ref["X"][:, 1568:]) and (X[:, 1574:] == 0).all()
    # the kernel drew forward 3's mask: forward 0's would not match
    other = ndr.features(_weights(net.state_dict("target" if which else "source")), b["vec"], b["win"], _drop(net, 0, n, draw=1))
    assert not torch.equal(idx, other["idx"])


# ---- 3. determinism and fresh masks -------------------------------------------------------------------------------
def test_same_seed_and_draw_same_bits_successive_calls_differ():
    n = 1000
    b = _batch(n, 5)
    a, c = _net(n, seed=31, dropout=P), _net(n, seed=31, dropout=P)
    Xa, ia = a.features(b["vec"], b["pwin"], save_idx=True)
    Xc, ic = c.features(b["vec"], b["pwin"], save_idx=True)
    assert a.draw == c.draw == 1
    assert torch.equal(Xa.view(torch.int16), Xc.view(torch.int16)) and torch.equal(ia, ic)
    Xa2, ia2 = a.features(b["vec"], b["pwin"], save_idx=True)
    assert not torch.equal(ia, ia2) and not torch.equal(Xa, Xa2)
    la = a.backward(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], 0.9).item()
    c.features(b["vec"], b["pwin"])                                 # c catches up with a's draw counter
    lc = c.backward(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], 0.9).item()
    assert abs(la - lc) <= 1e-6 * abs(la) and ((a.grads - c.grads).norm() / a.grads.norm()).item() <= 1e-5   # atomics: see above
    other = _net(n, seed=31, dropout=P, dropout_seed=32)
    Xo, io = other.features(b["vec"], b["pwin"], save_idx=True)
    assert not torch.equal(io, ia)
    # eval(): no dropout, the default net's features
    a.eval()
    Xe, ie = a.features(b["vec"], b["pwin"], save_idx=True)
    Xd, idd = _net(n, seed=31).features(b["vec"], b["pwin"], save_idx=True)
    assert torch.equal(Xe.view(torch.int16), Xd.view(torch.int16)) and torch.equal(ie, idd)
    # forward ids: the four masks of one draw are pairwise different
    masks = [ndr.keep_mask(a._c.dropout_seed, 9, f, 4, P) for f in range(4)]
    assert all(not torch.equal(masks[i], masks[j]) for i in range(4) for j in range(i + 1, 4))


# ---- 4. forward and DDQN backward with dropout at n = 8192 ----------------------------------------------------------
@pytest.fixture(scope="module")
def net_p():
    return _net(8192, seed=41, dropout=P)


@pytest.mark.parametrize("which", [0, 1])
def test_dropout_forward_within_tolerance(net_p, which):
    n = 8192
    b = _batch(n, 3000 + which)
    drop = _drop(net_p, ndr.FWD_STANDALONE, n)
    q = net_p.forward(b["vec"], b["pwin"], which=which)
    ref = ndr.forward(_weights(net_p.state_dict("target" if which else "source")), b["vec"], b["win"], drop)
    err = ((q.double() - ref["q"]).abs().max(1)[0] / ref["q"].abs().max()).max().item()
    _report(f"dropout forward which={which}", err)
    assert err <= TOL["q"]


def test_dropout_ddqn_backward_within_tolerance(net_p):
    n = 8192
    b = _batch(n, 4100)
    drops = [_drop(net_p, f, n) for f in range(3)]
    loss, qsa, grads = _backward(net_p, b)
    ref = ndr.ddqn_backward(_weights(net_p.state_dict("source")), _weights(net_p.state_dict("target")), b["vec"], b["win"], b["nvec"], b["nwin"],
                            b["action"], b["reward"], 0.9, drops=drops)
    _check_backward(loss, qsa, grads, ref, "dropout ddqn backward")


# ---- 5. DQN backward, with and without dropout --------------------------------------------------------------------
@pytest.mark.parametrize("p", [0.0, P])
def test_dqn_backward_within_tolerance_and_two_feature_passes(p):
    n = 8192
    net = _net(n, seed=51, dropout=p, double_q=False)
    b = _batch(n, 4200)
    drops = [_drop(net, f, n) if p > 0 else None for f in range(3)]
    net.profile(True)
    loss, qsa, grads = _backward(net, b)
    launches = [lab for lab, _ in net.profile_read()]
    net.profile(False)
    feats = [lab for lab in launches if lab.startswith("features")]
    assert len(feats) == 2, launches
    assert all(("dropout" in lab) == (p > 0) for lab in feats), feats
    assert any(lab.startswith("head: Q, max target") for lab in launches), launches
    ref = ndr.dqn_backward(_weights(net.state_dict("source")), _weights(net.state_dict("target")), b["vec"], b["win"], b["nvec"], b["nwin"],
                           b["action"], b["reward"], 0.9, drops=drops)
    _check_backward(loss, qsa, grads, {**ref, "fn": ref["fs"]}, f"dqn backward p={p}")
    dd = ndr.ddqn_backward(_weights(net.state_dict("source")), _weights(net.state_dict("target")), b["vec"], b["win"], b["nvec"], b["nwin"],
                           b["action"], b["reward"], 0.9, drops=drops)
    _report(f"dqn p={p}: double-Q loss of the same batch, relative difference", abs(dd["loss"].item() - loss) / loss)


# ---- 6. against plain fp32 autograd through a fixed-mask Dropout ---------------------------------------------------
def _close_norm(got, ref, tol, what):   # test_gpu_net.py's gradient bound
    got, ref = got.float(), ref.float()
    rel = ((got - ref).norm() / ref.norm().clamp_min(1e-12)).item()
    worst = ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-12)).item()
    assert rel <= tol and worst <= 3 * tol, f"{what}: relative Frobenius error {rel:.4g}, worst entry {worst:.4g} of max (tol {tol})"


def _ref_with_masks(net, masks_src, masks_tgt):
    src, tgt = RefDQN().cuda(), RefDQN().cuda()
    src.load_state_dict(net.state_dict("source"))
    tgt.load_state_dict(net.state_dict("target"))
    src.conv[2] = ndr.FixedMaskDropout(masks_src, P)
    tgt.conv[2] = ndr.FixedMaskDropout(masks_tgt, P)
    return src, tgt


@pytest.mark.parametrize("double_q", [True, False])
def test_dropout_matches_fp32_autograd(double_q):
    from maze_b200.dqn_net import _views
    n = 512
    net = _net(n, seed=61, dropout=P, double_q=double_q)
    b = _batch(n, 4300)
    m = [ndr.keep_mask(net._c.dropout_seed, net.draw, f, n, P) for f in range(3)]
    src, tgt = _ref_with_masks(net, [m[0], m[1]] if double_q else [m[0]], [m[2]])
    loss_fn = ddqn_loss if double_q else ndr.dqn_loss
    loss, _ = loss_fn(src, tgt, (b["vec"], b["win"]), b["action"], b["reward"], (b["nvec"], b["nwin"]), 0.9)
    loss.backward()
    dev_loss, _, grads = _backward(net, b)
    assert abs(dev_loss - loss.item()) <= 2e-2 * loss.item()
    gv = _views(grads)
    for name, prm in src.named_parameters():
        got = gv[name][:, :1574] if name == "fc.0.weight" else gv[name]
        _close_norm(got.reshape(prm.grad.shape), prm.grad, 4e-2, f"grad {name}")
    # forward (id 3) against the module
    mq = ndr.keep_mask(net._c.dropout_seed, net.draw, ndr.FWD_STANDALONE, n, P)
    src.conv[2] = ndr.FixedMaskDropout([mq], P)
    q = net.forward(b["vec"], b["pwin"])
    with torch.no_grad():
        qr = src((b["vec"], b["win"]))
    assert (q - qr).abs().max().item() <= 2e-2 * qr.abs().max().item()


@pytest.mark.parametrize("double_q", [True, False])
def test_dropout_train_steps_track_fp32_autograd(double_q):
    n, lr = 512, 1e-4
    net = _net(n, seed=71, dropout=P, double_q=double_q)
    src, tgt = _ref_with_masks(net, [], [])
    opt = torch.optim.AdamW(src.parameters(), lr)
    b = _batch(n, 33)
    loss_fn = ddqn_loss if double_q else ndr.dqn_loss
    dev, ref = [], []
    for it in range(12):
        d = net.draw
        src.conv[2].masks = [ndr.keep_mask(net._c.dropout_seed, d, f, n, P) for f in ((0, 1) if double_q else (0,))]
        tgt.conv[2].masks = [ndr.keep_mask(net._c.dropout_seed, d, 2, n, P)]
        src.conv[2].calls = tgt.conv[2].calls = 0
        net.train_step(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], gamma=0.9, lr=lr)
        dev.append(net.loss.item())
        loss, _ = loss_fn(src, tgt, (b["vec"], b["win"]), b["action"], b["reward"], (b["nvec"], b["nwin"]), 0.9)
        ref.append(loss.item())
        opt.zero_grad()
        loss.backward()
        for prm in src.parameters():
            prm.grad.data.clamp_(-1, 1)
        opt.step()
    for it, (a, r) in enumerate(zip(dev, ref)):
        assert abs(a - r) <= 0.1 * r + 1e-4, (it, dev, ref)


# ---- 7. out-of-range settings are errors --------------------------------------------------------------------------
def test_out_of_range_settings_return_errors():
    from maze_b200 import cabi
    from maze_b200.dqn_net import DQNNet
    for p in (1.0, -0.1, float("nan")):
        with pytest.raises(ValueError):
            DQNNet("cuda", max_batch=8, dropout=p)
    net = _net(64, seed=81)
    b = _batch(64, 1)
    for field, value in (("dropout", 1.0), ("dropout", -0.25), ("dropout", float("nan")), ("update", 2), ("update", -1), ("eval", 3)):
        old = getattr(net._c, field)
        setattr(net._c, field, value)
        with pytest.raises(cabi.MazeError):
            net.forward(b["vec"], b["pwin"])
        with pytest.raises(cabi.MazeError):
            net.backward(b["vec"], b["pwin"], b["nvec"], b["pnwin"], b["action"], b["reward"], 0.9)
        setattr(net._c, field, old)
    net.forward(b["vec"], b["pwin"])


# ---- 8. the example ----------------------------------------------------------------------------------------------
def test_train_example_runs_dqn_with_dropout():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "train_ddqn.py"), "--envs", "512", "--iters", "40", "--batch", "256",
                          "--shape", "21", "--memory", "65536", "--agent", "dqn", "--dropout", "0.2"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["agent"] == "dqn" and line["dropout"] == 0.2
    assert line["optimizer_steps_per_s"] > 0 and line["final_loss"] == line["final_loss"] and abs(line["final_loss"]) < float("inf")
