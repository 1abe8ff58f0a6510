"""The net's Dropout and the DQN target in the bf16-faithful float64 reference (test infrastructure).

Extends tests/net_bf16_reference.py (which stays the dropout-free, double-Q reference) with
  * `keep_mask`: a vectorised numpy model of the device's keep mask (include/maze_b200.h, "Dropout"): Philox4x32-10,
    key (seed lo, seed hi), counter (e / 8, sample, draw lo 32 bits, forward id), element
    e = ((py * 7 + px) * 32 + channel) * 4 + 2 dy + dx, 16-bit draw k = e % 8 from bits 16 (k & 1) of word k / 2,
    keep iff draw < round(65536 (1 - p)).  `philox4x32_10` is oracle/gen_stream.philox4x32_10 on numpy arrays.
  * `features` / `forward` with an optional per-forward mask: candidate = keep ? f32(f32(LeakyReLU(f32(conv + b))) *
    scale) : +0, first maximum over the 2 x 2 candidates, bf16; idx bit 3 = the winner was dropped.
  * `ddqn_backward` with the three forwards' masks, and `dqn_backward`: y = r + gamma * max_a q_target(s', a).
  * `conv_grad` through the Dropout: 0 for a dropped winner, else bf16(f32(g * scale) [* slope]).
With masks=None every function is net_bf16_reference's own.
"""
from __future__ import annotations

import numpy as np
import torch

import net_bf16_reference as nbr

M32 = np.uint64(0xFFFFFFFF)
FWD_SOURCE_S, FWD_SOURCE_SN, FWD_TARGET_SN, FWD_STANDALONE = 0, 1, 2, 3


def threshold(p: float) -> int:
    """round(65536 (1 - p)) with p as the fp32 the struct holds."""
    return int(np.floor(65536.0 * (1.0 - float(np.float32(p))) + 0.5))


def scale(p: float) -> float:
    """fp32(1 / (1 - p))."""
    return float(np.float32(1.0 / (1.0 - float(np.float32(p)))))


def philox4x32_10(k0, k1, c0, c1, c2, c3):
    """Philox4x32-10 on arrays (broadcast): the same rounds as oracle/gen_stream.philox4x32_10."""
    a, b = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    x0, x1, x2, x3 = (np.asarray(c, dtype=np.uint64) & M32 for c in (c0, c1, c2, c3))
    x0, x1, x2, x3 = np.broadcast_arrays(x0, x1, x2, x3)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * x0
        p1 = np.uint64(0xCD9E8D57) * x2
        x0, x1, x2, x3 = ((p1 >> np.uint64(32)) ^ x1 ^ a) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ x3 ^ b) & M32, p0 & M32
        a = (a + np.uint64(0x9E3779B9)) & M32
        b = (b + np.uint64(0xBB67AE85)) & M32
    return x0, x1, x2, x3


def keep_draws(seed: int, draw: int, fwd: int, samples):
    """The 16-bit draws of every element of the given samples: uint16 [len(samples), 6272] in element order."""
    samples = np.asarray(samples, dtype=np.uint64).reshape(-1, 1)
    blocks = np.arange(49 * 16, dtype=np.uint64).reshape(1, -1)
    o = philox4x32_10(seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF, blocks, samples, draw & 0xFFFFFFFF, fwd)
    words = np.stack(o, -1)                                                   # [S, 784, 4]
    halves = np.stack([words & np.uint64(0xFFFF), words >> np.uint64(16)], -1)  # [S, 784, 4, 2]: draw k = 2 word + half
    return halves.reshape(samples.shape[0], 49 * 16 * 8).astype(np.uint16)


def keep_mask(seed: int, draw: int, fwd: int, n: int, p: float, device=None):
    """bool [n, 32, 14, 14]: keep bit of conv output (channel, y, x) for samples 0 .. n-1 (y, x < 14: what the pool reads)."""
    k = keep_draws(seed, draw, fwd, np.arange(n)) < threshold(p)            # [n, (py, px, c, dy, dx)]
    k = k.reshape(n, 7, 7, 32, 2, 2).transpose(0, 3, 1, 4, 2, 5).reshape(n, 32, 14, 14)   # -> [n, c, (py dy), (px dx)]
    return torch.from_numpy(np.ascontiguousarray(k)).to(device) if device is not None else torch.from_numpy(np.ascontiguousarray(k))


def keep_mask_scalar(seed: int, draw: int, fwd: int, sample: int, c: int, y: int, x: int, p: float) -> bool:
    """One element's keep bit with the scalar oracle Philox (the layout spelled out once more)."""
    from oracle.gen_stream import philox4x32_10 as philox_scalar
    e = (((y // 2) * 7 + x // 2) * 32 + c) * 4 + 2 * (y % 2) + (x % 2)
    o = philox_scalar((seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF), (e // 8, sample, draw & 0xFFFFFFFF, fwd))
    k = e % 8
    return ((o[k // 2] >> (16 * (k % 2))) & 0xFFFF) < threshold(p)


class Drop:
    """One forward's Dropout: the keep mask [n, 32, 14, 14] (bool) and the fp32 scale."""

    def __init__(self, mask, p: float):
        self.mask = mask
        self.scale = scale(p)
        self.p = p


def features(w: nbr.NetWeights, vec, win, drop: Drop | None = None):
    """net_features_kernel; with `drop`, its dropout instantiation."""
    if drop is None:
        return nbr.features(w, vec, win)
    r, n = w.r, win.shape[0]
    conv = torch.matmul(w.conv_w.view(32, 27), nbr.window_patches(win)).view(n, 32, 15, 15)[..., :14, :14]
    pre = r.f32(conv + w.conv_b.view(1, 32, 1, 1))
    s = drop.scale if r.on else 1.0 / (1.0 - drop.p)
    mask = drop.mask.to(pre.device)
    cand = torch.where(mask, r.f32(r.lrelu(pre) * s), torch.zeros_like(pre))   # a dropped candidate is +0
    m, cls, _ = nbr.pool_first_max(cand)
    split = lambda t: torch.stack([t[..., dy::2, dx::2] for dy in (0, 1) for dx in (0, 1)], -1)   # [n, 32, 7, 7, 4]
    sel = lambda t: split(t).gather(-1, cls.long()[..., None])[..., 0]
    win_pre, win_kept = sel(pre), sel(mask)
    idx = cls | ((win_pre > 0).to(torch.uint8) << 2) | ((~win_kept).to(torch.uint8) << 3)
    X = torch.cat([r.bf16(m).reshape(n, -1), r.bf16(vec.double())], 1)
    # knife edges: a candidate's fp32 error is the conv sum's, times its slope and the scale (a dropped one is exact 0)
    conv_scale = w.conv_w.abs().view(32, 27).sum(1).view(1, 32, 1, 1) + w.conv_b.abs().view(1, 32, 1, 1)
    err = split(torch.where(mask, nbr.NEAR_REL * conv_scale * s * torch.where(pre > 0, 1.0, r.slope), torch.zeros_like(pre)))
    gaps = m[..., None] - split(cand)
    others = torch.arange(4, device=pre.device) != cls.long()[..., None]
    near = (others & (gaps > 0) & (gaps <= err + err.gather(-1, cls.long()[..., None]))).any(-1)
    return dict(X=X, idx=idx.reshape(n, -1), pre=win_pre.reshape(n, -1), pool_near=near.reshape(n, -1),
                pool_ties=int((others & (gaps == 0)).sum()),
                act_near=((win_pre.abs() <= nbr.NEAR_REL * conv_scale) & win_kept).reshape(n, -1))


def forward(w: nbr.NetWeights, vec, win, drop: Drop | None = None):
    """nbr.forward with the features of `features`."""
    if drop is None:
        return nbr.forward(w, vec, win)
    r = w.r
    out = features(w, vec, win, drop)
    X = out["X"]
    h1_pre = r.f32(r.f32(X @ w.w1.t()) + w.b1)
    h1 = r.bf16(r.lrelu(h1_pre))
    h2_pre = r.f32(r.f32(h1 @ w.w2.t()) + w.b2)
    h2 = r.bf16(torch.clamp_min(h2_pre, 0.0))
    q = (h2.unsqueeze(1) * w.w3).sum(-1) + w.b3
    h1_scale = X.abs() @ w.w1.abs().t() + w.b1.abs()
    h2_scale = h1.abs() @ w.w2.abs().t() + w.b2.abs()
    out.update(h1_pre=h1_pre, h1=h1, h2_pre=h2_pre, h2=h2, q=q, h1_near=h1_pre.abs() <= nbr.NEAR_REL * h1_scale,
               h2_near=h2_pre.abs() <= nbr.NEAR_REL * h2_scale)
    return out


def conv_grad(w: nbr.NetWeights, dX, idx, win, drop: Drop | None = None):
    """nbr.conv_grad; with `drop`, the Dropout backward before the LeakyReLU backward."""
    if drop is None:
        return nbr.conv_grad(w, dX, idx, win)
    r, n = w.r, dX.shape[0]
    g = dX.view(n, 32, 49)
    b = idx.view(n, 32, 49)
    s = drop.scale if r.on else 1.0 / (1.0 - drop.p)
    gs = torch.where((b & 8) != 0, torch.zeros_like(g), r.f32(g * s))
    gv = torch.where((b & 4) != 0, r.bf16(gs), r.bf16(r.f32(gs * r.slope)))
    q = torch.arange(49, device=dX.device)
    y = 2 * (q // 7) + ((b >> 1) & 1).long()
    x = 2 * (q % 7) + (b & 1).long()
    G = torch.zeros(n, 32, 225, dtype=torch.float64, device=dX.device)
    G.scatter_(2, y * 15 + x, gv)
    gw = torch.einsum("nop,nkp->ok", G, nbr.window_patches(win)).view(32, 3, 3, 3)
    return gw, G.sum((0, 2))


def _backward_from(src, fs, qsa, y, action, win, n, drop0):
    r = src.r
    a = action.long()
    d = qsa - y
    loss = (d * d).mean()
    gq = 2.0 * d / n
    h2, h1, X = fs["h2"], fs["h1"], fs["X"]
    dh2 = r.bf16(torch.where(h2 > 0, r.f32(gq[:, None] * src.w3[a]), torch.zeros_like(h2)))
    gw3 = torch.zeros_like(src.w3).index_add_(0, a, gq[:, None] * h2)
    gb3 = torch.zeros_like(src.b3).index_add_(0, a, gq)
    gb2 = dh2.sum(0)
    gw2 = dh2.t() @ h1
    dh1 = r.bf16(r.f32(r.f32(dh2 @ src.w2) * torch.where(h1 > 0, 1.0, r.slope)))
    gb1 = dh1.sum(0)
    gw1 = dh1.t() @ X
    dX = r.bf16(dh1 @ src.w1[:, :1568])
    gcw, gcb = conv_grad(src, dX, fs["idx"], win, drop0)
    grads = {"conv.0.weight": gcw, "conv.0.bias": gcb, "fc.0.weight": gw1, "fc.0.bias": gb1, "fc.2.weight": gw2, "fc.2.bias": gb2,
             "fc.4.weight": gw3, "fc.4.bias": gb3}
    return dict(loss=loss, qsa=qsa, grads=grads, dh2=dh2, dh1=dh1, dX=dX)


def ddqn_backward(src, tgt, vec, win, next_vec, next_win, action, reward, gamma: float, drops=(None, None, None)):
    """maze_dqn_backward with update = 0; drops: the Dropout of forwards 0 (source on s), 1 (source on s'), 2 (target on s')."""
    if all(d is None for d in drops):
        return nbr.ddqn_backward(src, tgt, vec, win, next_vec, next_win, action, reward, gamma)
    n = vec.shape[0]
    fs = forward(src, vec, win, drops[0])
    fn = forward(src, next_vec, next_win, drops[1])
    ft = forward(tgt, next_vec, next_win, drops[2])
    best, argmax_near = nbr.first_argmax(fn["q"])
    qsa = fs["q"].gather(1, action.long()[:, None])[:, 0]
    y = ft["q"].gather(1, best[:, None])[:, 0] * gamma + reward.double()
    out = _backward_from(src, fs, qsa, y, action, win, n, drops[0])
    out.update(best=best, argmax_near=argmax_near, fs=fs, fn=fn, ft=ft)
    return out


def dqn_backward(src, tgt, vec, win, next_vec, next_win, action, reward, gamma: float, drops=(None, None, None)):
    """maze_dqn_backward with update = 1: y = r + gamma * max_a q_target(s', a); drops[1] is unused (no source forward on s')."""
    n = vec.shape[0]
    fs = forward(src, vec, win, drops[0])
    ft = forward(tgt, next_vec, next_win, drops[2])
    qsa = fs["q"].gather(1, action.long()[:, None])[:, 0]
    y = ft["q"].max(1)[0] * gamma + reward.double()
    out = _backward_from(src, fs, qsa, y, action, win, n, drops[0])
    out.update(argmax_near=torch.zeros(n, dtype=torch.bool, device=qsa.device), fs=fs, ft=ft)
    return out


class FixedMaskDropout(torch.nn.Module):
    """nn.Dropout with given masks, one per call in order ([n, 32, 14, 14] bool, padded to the 15 x 15 conv output):
    x * mask * 1 / (1 - p), the autograd graph torch's Dropout builds."""

    def __init__(self, masks, p: float):
        super().__init__()
        self.masks, self.p, self.calls = list(masks), p, 0

    def forward(self, x):
        m = torch.ones(x.shape, dtype=x.dtype, device=x.device)
        m[..., :14, :14] = self.masks[self.calls].to(device=x.device, dtype=x.dtype)
        self.calls += 1
        return x * m * (1.0 / (1.0 - self.p))


def dqn_loss(source, target, state, action, reward, next_state, gamma: float):
    """The DQN update's loss: mse(q(s, a), r + gamma * max_a q_target(s', a)) (agents/dqn_agent.py; see DESIGN.md §4.3)."""
    qsa = source(state).gather(1, action.long().unsqueeze(1))
    with torch.no_grad():
        nxt = target(next_state).max(1)[0]
    expected = nxt * gamma + reward
    return torch.nn.functional.mse_loss(qsa, expected.unsqueeze(1)), qsa.squeeze(1)
