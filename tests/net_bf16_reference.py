"""A float64 reference of the tensor-core DQN net that rounds where the kernels round (test infrastructure).

`net_reference.RefDQN` is the net in plain fp32: it differs from csrc/maze_net.cu by bf16 noise, so tests against it
need loose tolerances.  The functions here compute every stage in float64 and round to bf16 (through fp32) at exactly
the points where the kernels store bf16, and to fp32 where a kernel result passes through an fp32 register before such
a store.  What remains between them and the kernels is the order of the fp32 accumulations: with operands on a coarse
dyadic grid those sums are exact in any order and the results agree bit for bit.

Rounding points (line numbers of maze_net.cu):
  * conv weights -> bf16 (net_conv_image_kernel, :587); the conv bias stays fp32 (:618, :704).
  * W1, W2 -> bf16 (net_refresh_kernel, :1241, :1247); b1, b2, W3, b3 stay fp32.
  * state vector -> bf16 when it is written into X (net_features_kernel, :721, `xrow[NET_CONV_OUT + tid]`).
  * features (net_features_kernel, :684-708): the conv sum over the binary window is exact; the 2 x 2 pool takes the
    FIRST maximum in the scan order (0,0), (0,1), (1,0), (1,1) (`x > m[ch]`, :693); then fp32 bias, LeakyReLU with
    slope 0.01f, bf16.  idx byte: bit 0 = x parity of the winner, bit 1 = y parity, bit 2 = pre-activation > 0 (:705).
  * forward GEMM epilogue (epi_bf16_tile, :119-131): h1 = bf16(lrelu(acc + b1)), h2 = bf16(relu(acc + b2)).
  * fc3 head (net_head_q_kernel / net_head_loss_kernel, :773-906): fp32 W3, b3 on the bf16 h2; double-Q target from
    the first maximum of the source net's q(s') (:884-887); gq = 2 d / n; dh2 = bf16(h2 > 0 ? gq W3[a] : 0) (:897-898);
    the fc3 gradients from the bf16 h2 (:902-903).
  * backward: gb2 = colsum(dh2), dW2 = dh2^T h1; dh1 = bf16((dh2 W2) * (h1 > 0 ? 1 : 0.01f)) with the sign of the
    STORED bf16 activation, an exact zero taking the slope (EPI_MASK, :133-144); gb1 = colsum(dh1), dW1 = dh1^T X;
    dX = bf16(dh1 W1) over the 1568 conv columns (EPI_BIAS_ACT without bias, :1552-1554).
  * conv gradient: dX routed to the pool winner, times LeakyReLU' from idx bit 2.  net_conv_bwd_tc_kernel rounds
    gv * 0.01f to bf16 before the MMA (:1131-1133, tc=True); net_conv_bwd_kernel keeps it in fp32 (:981-984, tc=False).

With rounding=False every rounding point is the identity and the slope is 0.01: the functions then compute the fp32
net's exact float64 semantics, which tests/test_net_bf16_reference_cpu.py checks against autograd.

Knife edges: where the kernels' fp32 accumulation order can decide a discrete outcome, the stages report it -- a pool
whose top two candidates, or a pre-activation whose distance to 0, is within fp32 accumulation error (`*_near`), and a
q(s') arg-max whose top two values are within 1e-5 relative (`argmax_near`).  Exact ties are not knife edges: equal
float64 sums of the same terms are equal fp32 sums too, and both sides break them the same way.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

SLOPE_F32 = float(np.float32(0.01))      # LRELU_SLOPE = 0.01f
NEAR_REL = 2.0 ** -16                    # fp32 accumulation error bound, relative to the sum of |terms| (K <= 1600)
ARGMAX_NEAR_REL = 1e-5
NAMES = ("conv.0.weight", "conv.0.bias", "fc.0.weight", "fc.0.bias", "fc.2.weight", "fc.2.bias", "fc.4.weight", "fc.4.bias")


class Rounding:
    """The rounding points, switchable: bf16(x) and f32(x) on float64 tensors, and the LeakyReLU slope."""

    def __init__(self, on: bool = True):
        self.on = on
        self.slope = SLOPE_F32 if on else 0.01

    def bf16(self, x):
        return x.float().bfloat16().double() if self.on else x

    def f32(self, x):
        return x.float().double() if self.on else x

    def lrelu(self, x):   # x > 0 ? x : slope * x, the product rounded like the kernels' fp32 multiply
        return torch.where(x > 0, x, self.f32(self.slope * x))


class NetWeights:
    """One net's parameters (a DQNNet / RefDQN state_dict) as float64, with the bf16 operands the kernels use."""

    def __init__(self, sd, rounding: Rounding, device=None):
        d = device if device is not None else sd["fc.0.weight"].device
        g = {k: sd[k].detach().to(device=d, dtype=torch.float32).double() for k in NAMES}
        self.r = rounding
        self.conv_w = rounding.bf16(g["conv.0.weight"])
        self.conv_b = g["conv.0.bias"]
        self.w1 = rounding.bf16(g["fc.0.weight"])       # [1024, 1574]
        self.b1 = g["fc.0.bias"]
        self.w2 = rounding.bf16(g["fc.2.weight"])       # [512, 1024]
        self.b2 = g["fc.2.bias"]
        self.w3 = g["fc.4.weight"]
        self.b3 = g["fc.4.bias"]


def pool_first_max(pre):
    """2 x 2 / stride 2 max-pool of [n, C, 15, 15] over the top-left 14 x 14, the first maximum in scan order
    (0,0), (0,1), (1,0), (1,1) winning.  Returns (max [n, C, 7, 7], winner 0..3 = 2 dy + dx, the gap between the
    maximum and the best candidate below it: 0 for an exact tie)."""
    p = pre[..., :14, :14]
    cand = [p[..., dy::2, dx::2] for dy in (0, 1) for dx in (0, 1)]
    best, win = cand[0].clone(), torch.zeros(cand[0].shape, dtype=torch.uint8, device=pre.device)
    for k in (1, 2, 3):
        take = cand[k] > best
        best = torch.where(take, cand[k], best)
        win = torch.where(take, torch.full_like(win, k), win)
    below = torch.full_like(best, float("inf"))
    for k in range(4):
        gap = best - cand[k]
        below = torch.minimum(below, torch.where(win == k, torch.full_like(gap, float("inf")), gap))
    return best, win, below


def window_patches(win):
    """[n, 3, 15, 15] -> [n, 27, 225]: the 3 x 3 neighbourhoods (zero padding 1), tap order c * 9 + dy * 3 + dx."""
    return F.unfold(win.double(), 3, padding=1)


def features(w: NetWeights, vec, win):
    """net_features_kernel.  X [n, 1574] (conv features in (channel, py, px) order, then the state), idx [n, 1568]
    uint8, the pre-activations, and the knife edges."""
    r, n = w.r, win.shape[0]
    patches = window_patches(win)
    conv = torch.matmul(w.conv_w.view(32, 27), patches).view(n, 32, 15, 15)          # exact: binary window
    scale = w.conv_w.abs().view(32, 27).sum(1).view(1, 32, 1, 1) + w.conv_b.abs().view(1, 32, 1, 1)
    m, cls, gap = pool_first_max(conv)
    pre = r.f32(m + w.conv_b.view(1, 32, 1, 1))
    act = r.bf16(r.lrelu(pre))
    idx = cls | ((pre > 0).to(torch.uint8) << 2)      # cls = 2 dy + dx: bit 0 x parity, bit 1 y parity
    X = torch.cat([act.reshape(n, -1), r.bf16(vec.double())], 1)
    return dict(X=X, idx=idx.reshape(n, -1), pre=pre.reshape(n, -1),
                pool_near=((gap > 0) & (gap <= NEAR_REL * scale)).reshape(n, -1),
                pool_ties=int((gap == 0).sum()),
                act_near=(pre.abs() <= NEAR_REL * scale).reshape(n, -1))


def forward(w: NetWeights, vec, win):
    """Features, fc1 (LeakyReLU), fc2 (ReLU), fc3: every intermediate."""
    r = w.r
    out = features(w, vec, win)
    X = out["X"]
    h1_pre = r.f32(r.f32(X @ w.w1.t()) + w.b1)
    h1 = r.bf16(r.lrelu(h1_pre))
    h2_pre = r.f32(r.f32(h1 @ w.w2.t()) + w.b2)
    h2 = r.bf16(torch.clamp_min(h2_pre, 0.0))
    q = (h2.unsqueeze(1) * w.w3).sum(-1) + w.b3      # equal fc3 rows give equal q, bit for bit
    h1_scale = X.abs() @ w.w1.abs().t() + w.b1.abs()
    h2_scale = h1.abs() @ w.w2.abs().t() + w.b2.abs()
    out.update(h1_pre=h1_pre, h1=h1, h2_pre=h2_pre, h2=h2, q=q, h1_near=h1_pre.abs() <= NEAR_REL * h1_scale,
               h2_near=h2_pre.abs() <= NEAR_REL * h2_scale)
    return out


def first_argmax(q):
    """.max(1)[1] with the first maximum winning, and whether the top two are within ARGMAX_NEAR_REL (not equal)."""
    best = torch.zeros(q.shape[0], dtype=torch.long, device=q.device)
    for a in range(1, q.shape[1]):
        best = torch.where(q[:, a] > q.gather(1, best[:, None])[:, 0], torch.full_like(best, a), best)
    top = q.gather(1, best[:, None])
    gap = torch.where(torch.arange(q.shape[1], device=q.device)[None] == best[:, None], torch.full_like(q, float("inf")), top - q).min(1)[0]
    return best, (gap > 0) & (gap <= ARGMAX_NEAR_REL * top[:, 0].abs().clamp_min(1e-30))


def conv_grad(w: NetWeights, dX, idx, win, tc: bool = True):
    """d loss / d conv weight [32, 3, 3, 3] and bias [32] from dX [n, 1568], the pool choices and the windows."""
    r, n = w.r, dX.shape[0]
    g = dX.view(n, 32, 49)
    b = idx.view(n, 32, 49)
    neg = r.f32(g * r.slope)
    gv = torch.where((b & 4) != 0, g, r.bf16(neg) if tc else neg)
    q = torch.arange(49, device=dX.device)
    y = 2 * (q // 7) + ((b >> 1) & 1).long()
    x = 2 * (q % 7) + (b & 1).long()
    G = torch.zeros(n, 32, 225, dtype=torch.float64, device=dX.device)
    G.scatter_(2, y * 15 + x, gv)
    gw = torch.einsum("nop,nkp->ok", G, window_patches(win)).view(32, 3, 3, 3)
    return gw, G.sum((0, 2))


def ddqn_backward(src: NetWeights, tgt: NetWeights, vec, win, next_vec, next_win, action, reward, gamma: float, tc: bool = True,
                  keep=None):
    """maze_dqn_backward: loss, q(s, a) and the gradients of the source net (state_dict names and shapes).
    keep: optional [n] 0/1 weights on the samples' gradient contributions (1 / n stays the batch's), to model a kernel
    that lost some samples."""
    r, n = src.r, vec.shape[0]
    fs = forward(src, vec, win)
    fn = forward(src, next_vec, next_win)
    ft = forward(tgt, next_vec, next_win)
    best, argmax_near = first_argmax(fn["q"])
    a = action.long()
    qsa = fs["q"].gather(1, a[:, None])[:, 0]
    y = ft["q"].gather(1, best[:, None])[:, 0] * gamma + reward.double()
    d = qsa - y
    loss = (d * d).mean()
    gq = 2.0 * d / n
    if keep is not None:
        gq = gq * keep.double()
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
    gcw, gcb = conv_grad(src, dX, fs["idx"], win, tc=tc)
    grads = {"conv.0.weight": gcw, "conv.0.bias": gcb, "fc.0.weight": gw1, "fc.0.bias": gb1, "fc.2.weight": gw2, "fc.2.bias": gb2,
             "fc.4.weight": gw3, "fc.4.bias": gb3}
    return dict(loss=loss, qsa=qsa, grads=grads, dh2=dh2, dh1=dh1, dX=dX, best=best, argmax_near=argmax_near, fs=fs, fn=fn, ft=ft)
