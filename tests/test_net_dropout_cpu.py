"""The Dropout mask model and the dropout / DQN extensions of the float64 reference (tests/net_dropout_reference.py),
checked without a GPU: the vectorised Philox equals the scalar oracle one, the keep rate is 1 - p, and with rounding
switched off the reference is torch autograd's float64 semantics through a fixed-mask Dropout, for the double-Q and
the DQN loss."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import net_bf16_reference as nbr  # noqa: E402
import net_dropout_reference as ndr  # noqa: E402
from net_reference import RefDQN, ddqn_loss  # noqa: E402


def test_vectorised_mask_equals_scalar_philox():
    from oracle.gen_stream import philox4x32_10
    rng = np.random.default_rng(5)
    for seed, draw, fwd in ((0, 0, 0), (7, 1, 2), (2 ** 40 + 3, 2 ** 33 + 9, 3)):
        o = ndr.philox4x32_10(seed & 0xFFFFFFFF, seed >> 32, np.array([0, 1, 783]), 5, draw & 0xFFFFFFFF, fwd)
        for i, blk in enumerate((0, 1, 783)):
            assert tuple(int(w[i]) for w in o) == philox4x32_10((seed & 0xFFFFFFFF, seed >> 32), (blk, 5, draw & 0xFFFFFFFF, fwd))
        n = 6
        mask = ndr.keep_mask(seed, draw, fwd, n, 0.2)
        assert mask.shape == (n, 32, 14, 14) and mask.dtype == torch.bool
        for _ in range(200):
            s, c, y, x = int(rng.integers(n)), int(rng.integers(32)), int(rng.integers(14)), int(rng.integers(14))
            assert bool(mask[s, c, y, x]) == ndr.keep_mask_scalar(seed, draw, fwd, s, c, y, x, 0.2), (seed, draw, fwd, s, c, y, x)


def test_masks_differ_by_draw_forward_and_sample():
    base = ndr.keep_mask(3, 10, 0, 4, 0.2)
    for other in (ndr.keep_mask(3, 11, 0, 4, 0.2), ndr.keep_mask(3, 10, 1, 4, 0.2), ndr.keep_mask(4, 10, 0, 4, 0.2)):
        assert (other != base).double().mean().item() > 0.2
    assert (base[0] != base[1]).any()
    assert torch.equal(base, ndr.keep_mask(3, 10, 0, 4, 0.2))


@pytest.mark.parametrize("p", [0.2, 0.5, 0.05])
def test_keep_fraction_within_five_sigma(p):
    n = 64
    frac = ndr.keep_mask(11, 2, 0, n, p).double().mean().item()
    N = n * 32 * 14 * 14
    assert ndr.threshold(0.2) == 52429 and ndr.scale(0.2) == 1.25
    sigma = (p * (1 - p) / N) ** 0.5
    assert abs(frac - (1 - p)) <= 5 * sigma, (frac, 1 - p, sigma)


def _batch(n, seed):
    g = torch.Generator().manual_seed(seed)
    win = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).double()
    nwin = (torch.rand(n, 3, 15, 15, generator=g) < 0.45).double()
    vec, nvec = torch.rand(n, 6, generator=g, dtype=torch.float64), torch.rand(n, 6, generator=g, dtype=torch.float64)
    action = torch.randint(0, 4, (n,), generator=g).to(torch.uint8)
    reward = torch.rand(n, generator=g, dtype=torch.float64) - 0.5
    return vec, win, nvec, nwin, action, reward


def _check_grads(ref, src, what):
    for name, prm in src.named_parameters():
        got = ref["grads"][name]
        assert got.shape == prm.grad.shape, (what, name)
        err = (got - prm.grad).abs().max().item()
        assert err <= 1e-10 * max(1.0, prm.grad.abs().max().item()), (what, name, err)


@pytest.mark.parametrize("update", ["ddqn", "dqn"])
@pytest.mark.parametrize("n", [3, 16])
def test_unrounded_dropout_reference_equals_float64_autograd(n, update):
    p = 0.2
    torch.manual_seed(n)
    src, tgt = RefDQN().double(), RefDQN().double()
    vec, win, nvec, nwin, action, reward = _batch(n, 200 + n)
    masks = [ndr.keep_mask(9, 4, f, n, p) for f in range(3)]
    assert not masks[0].all() and masks[0].any()
    src.conv[2] = ndr.FixedMaskDropout(masks[:2], p)       # source(state), then source(next state) (DDQN only)
    tgt.conv[2] = ndr.FixedMaskDropout(masks[2:], p)
    off = nbr.Rounding(False)
    ws, wt = nbr.NetWeights(src.state_dict(), off), nbr.NetWeights(tgt.state_dict(), off)
    drops = [ndr.Drop(m, p) for m in masks]
    if update == "ddqn":
        loss, qsa = ddqn_loss(src, tgt, (vec, win), action, reward, (nvec, nwin), 0.9)
        ref = ndr.ddqn_backward(ws, wt, vec, win, nvec, nwin, action, reward, 0.9, drops=drops)
        assert src.conv[2].calls == 2
    else:
        loss, qsa = ndr.dqn_loss(src, tgt, (vec, win), action, reward, (nvec, nwin), 0.9)
        ref = ndr.dqn_backward(ws, wt, vec, win, nvec, nwin, action, reward, 0.9, drops=drops)
        assert src.conv[2].calls == 1
    loss.backward()
    assert abs(ref["loss"].item() - loss.item()) <= 1e-10
    assert torch.allclose(ref["qsa"], qsa.detach(), rtol=0, atol=1e-10)
    _check_grads(ref, src, update)
    # the mask matters: without it the loss is another
    plain = nbr.ddqn_backward(ws, wt, vec, win, nvec, nwin, action, reward, 0.9)
    assert abs(plain["loss"].item() - loss.item()) > 1e-6


def test_dqn_without_dropout_equals_float64_autograd():
    n = 8
    torch.manual_seed(1)
    src, tgt = RefDQN().double(), RefDQN().double()
    vec, win, nvec, nwin, action, reward = _batch(n, 300)
    off = nbr.Rounding(False)
    ws, wt = nbr.NetWeights(src.state_dict(), off), nbr.NetWeights(tgt.state_dict(), off)
    loss, qsa = ndr.dqn_loss(src, tgt, (vec, win), action, reward, (nvec, nwin), 0.9)
    loss.backward()
    ref = ndr.dqn_backward(ws, wt, vec, win, nvec, nwin, action, reward, 0.9)
    assert abs(ref["loss"].item() - loss.item()) <= 1e-10
    _check_grads(ref, src, "dqn")


def test_no_mask_is_the_plain_reference():
    vec, win, nvec, nwin, action, reward = _batch(5, 400)
    w = nbr.NetWeights(RefDQN().double().state_dict(), nbr.Rounding(True))
    a, b = ndr.forward(w, vec, win), nbr.forward(w, vec, win)
    assert torch.equal(a["X"], b["X"]) and torch.equal(a["q"], b["q"]) and torch.equal(a["idx"], b["idx"])


def test_all_kept_mask_pools_the_same_values():
    """p -> a mask of all ones with scale 1: the dropout path (pool after the activation) gives the same pooled values as
    the plain path (activation after the pool), and idx bit 3 stays clear."""
    vec, win, _, _, _, _ = _batch(6, 500)
    sd = RefDQN().double().state_dict()
    w = nbr.NetWeights(sd, nbr.Rounding(True))
    d = ndr.Drop(torch.ones(6, 32, 14, 14, dtype=torch.bool), 0.0)
    assert d.scale == 1.0
    a, b = ndr.features(w, vec, win, d), nbr.features(w, vec, win)
    assert torch.equal(a["X"], b["X"])
    assert ((a["idx"] & 8) == 0).all()
