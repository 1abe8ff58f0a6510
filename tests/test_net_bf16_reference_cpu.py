"""The bf16-faithful float64 reference (tests/net_bf16_reference.py) checked on its own, without a GPU: with the rounding
switched off it is the fp32 net's float64 semantics (torch autograd on RefDQN in float64), its pool is max_pool2d's on
exact ties, and the packed window format round-trips."""
import pytest

torch = pytest.importorskip("torch")

import net_bf16_reference as nbr  # noqa: E402
from net_reference import RefDQN, ddqn_loss, pack_windows  # noqa: E402


def _batch(n, seed):
    g = torch.Generator().manual_seed(seed)
    win = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).double()
    nwin = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).double()
    vec, nvec = torch.rand(n, 6, generator=g, dtype=torch.float64), torch.rand(n, 6, generator=g, dtype=torch.float64)
    action = torch.randint(0, 4, (n,), generator=g).to(torch.uint8)
    reward = torch.rand(n, generator=g, dtype=torch.float64) - 0.5
    return vec, win, nvec, nwin, action, reward


@pytest.mark.parametrize("n", [3, 16])
def test_unrounded_reference_equals_float64_autograd(n):
    torch.manual_seed(n)
    src, tgt = RefDQN().double(), RefDQN().double()
    vec, win, nvec, nwin, action, reward = _batch(n, 100 + n)
    off = nbr.Rounding(False)
    ws, wt = nbr.NetWeights(src.state_dict(), off), nbr.NetWeights(tgt.state_dict(), off)
    with torch.no_grad():
        assert torch.allclose(nbr.forward(ws, vec, win)["q"], src((vec, win)), rtol=0, atol=1e-10)
        assert torch.allclose(nbr.forward(wt, nvec, nwin)["q"], tgt((nvec, nwin)), rtol=0, atol=1e-10)
    loss, qsa = ddqn_loss(src, tgt, (vec, win), action, reward, (nvec, nwin), 0.9)
    loss.backward()
    ref = nbr.ddqn_backward(ws, wt, vec, win, nvec, nwin, action, reward, 0.9)
    assert abs(ref["loss"].item() - loss.item()) <= 1e-10
    assert torch.allclose(ref["qsa"], qsa.detach(), rtol=0, atol=1e-10)
    for name, p in src.named_parameters():
        got = ref["grads"][name]
        assert got.shape == p.grad.shape, name
        err = (got - p.grad).abs().max().item()
        assert err <= 1e-10 * max(1.0, p.grad.abs().max().item()), (name, err)
    # both conv-gradient roundings are the same function without rounding
    gw, gb = nbr.conv_grad(ws, ref["dX"], ref["fs"]["idx"], win, tc=False)
    assert torch.equal(gw, ref["grads"]["conv.0.weight"]) and torch.equal(gb, ref["grads"]["conv.0.bias"])


def test_pool_and_idx_equal_max_pool2d_on_exact_ties():
    """Integer conv weights on binary windows: most pooled cells have tied candidates.  The winner must be the first
    maximum in scan order, which is what max_pool2d(return_indices=True) returns on CPU."""
    g = torch.Generator().manual_seed(7)
    n = 64
    win = (torch.rand(n, 3, 15, 15, generator=g) < 0.5).double()
    win[:4] = 0.0                        # all-zero windows: four-way ties everywhere
    win[4:8] = 1.0
    sd = RefDQN().double().state_dict()
    sd["conv.0.weight"] = torch.randint(-1, 2, (32, 3, 3, 3), generator=g).double()
    sd["conv.0.bias"] = torch.randint(-2, 3, (32,), generator=g).double()
    w = nbr.NetWeights(sd, nbr.Rounding(True))
    out = nbr.features(w, torch.zeros(n, 6, dtype=torch.float64), win)
    conv = torch.nn.functional.conv2d(win, sd["conv.0.weight"], sd["conv.0.bias"], padding=1)
    pooled, ind = torch.nn.functional.max_pool2d(conv, 2, 2, return_indices=True)
    assert out["pool_ties"] > n * 32 * 49 // 4          # the case is what it claims to be
    idx = out["idx"].view(n, 32, 7, 7).long()
    py, px = torch.arange(7).view(7, 1), torch.arange(7).view(1, 7)
    flat = (2 * py + ((idx >> 1) & 1)) * 15 + 2 * px + (idx & 1)
    assert torch.equal(flat, ind)
    assert torch.equal(out["pre"].view(n, 32, 7, 7), pooled)
    assert torch.equal(((idx >> 2) & 1).bool(), pooled > 0)
    assert not out["pool_near"].any()
    lrelu = torch.where(pooled > 0, pooled, (pooled * nbr.SLOPE_F32).float().double())
    assert torch.equal(out["X"][:, :1568], lrelu.reshape(n, -1).float().bfloat16().double())


def test_first_argmax_takes_the_first_maximum_and_flags_near_ties():
    q = torch.tensor([[0.0, 1.0, 1.0, 0.5], [2.0, 2.0, 2.0, 2.0], [1.0, 1.0 + 1e-7, 0.0, 0.0], [0.0, 0.0, 0.0, 3.0]], dtype=torch.float64)
    best, near = nbr.first_argmax(q)
    assert best.tolist() == [1, 0, 1, 3]
    assert near.tolist() == [False, False, True, False]


def test_pack_windows_round_trips():
    from maze_b200.dqn import unpack_windows
    g = torch.Generator().manual_seed(3)
    win = (torch.rand(50, 3, 15, 15, generator=g) < 0.5).float()
    win[0] = 1.0
    win[1] = 0.0
    words = pack_windows(win)
    assert words.dtype == torch.int32 and words.shape == (50, 24)
    assert torch.equal(unpack_windows(words), win)
    assert (words[0] & ~0x7fff7fff).eq(0).all() and (words[0, [7, 15, 23]] == 0x7fff).all()   # row 15 does not exist
    one = torch.zeros(1, 3, 15, 15)
    one[0, 2, 5, 9] = 1.0                 # channel 2, row 5 = 2 * 2 + 1, column 9: word 2 * 8 + 2, bit 16 + 9
    assert pack_windows(one)[0].tolist() == [0] * 18 + [1 << 25] + [0] * 5
