"""The DQN / DDQN network of agents/ddqn_agent.py:18-52 and its update (:113-152) on the B200 tensor cores.

    net = DQNNet(device, max_batch=8192, seed=0)                  # source + target net, AdamW state
    q = net.forward(memory.stage_vec, memory.stage_win)            # [B, 4] float32 (policy inference)
    batch = memory.sample_packed(n)                                # windows stay bit-packed
    loss = net.train_step(*batch, gamma=0.9, lr=1e-4)              # double-Q target, MSE, clamp +-1, AdamW
    net.update_target()                                            # target_net.load_state_dict(source_net.state_dict())

    DQNNet(device, dropout=0.2)                   # ddqn_agent.py as written: Dropout(0.2) in every forward
    DQNNet(device, double_q=False)                # dqn_agent.py: y = r + gamma * max_a q_target(s', a)

Everything runs in csrc/maze_net.cu through the C ABI (maze_dqn_forward / _backward / _adamw): tcgen05 GEMMs with
TMA-staged bf16 operands for the conv (implicit GEMM) and the two big Linear layers, fp32 master weights.
`state_dict()` / `load_state_dict()` speak the reference module's names (conv.0.weight, fc.0.weight, ...), so
weights move between this class and the reference's `DQN` nn.Module unchanged.  Dropout (between the conv's
LeakyReLU and its max-pool) is active in training mode (`train()`, the default: the reference never calls eval())
and off after `eval()`.  Its masks come from a counter stream keyed by `dropout_seed` (include/maze_b200.h): every
forward, features and backward call advances the net's draw counter, so two nets built alike and called alike
produce identical bits.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import cabi

_SHAPES = (("conv.0.weight", cabi.NET_OFF_CONV_W, (32, 3, 3, 3)), ("conv.0.bias", cabi.NET_OFF_CONV_B, (32,)),
           ("fc.0.weight", cabi.NET_OFF_W1, (cabi.NET_H1, cabi.NET_IN)), ("fc.0.bias", cabi.NET_OFF_B1, (cabi.NET_H1,)),
           ("fc.2.weight", cabi.NET_OFF_W2, (cabi.NET_H2, cabi.NET_H1)), ("fc.2.bias", cabi.NET_OFF_B2, (cabi.NET_H2,)),
           ("fc.4.weight", cabi.NET_OFF_W3, (4, cabi.NET_H2)), ("fc.4.bias", cabi.NET_OFF_B3, (4,)))


def _views(flat: torch.Tensor):
    out = {}
    for name, off, shape in _SHAPES:
        n = math.prod(shape)
        out[name] = flat[off:off + n].view(shape)
    return out


class DQNNet:
    def __init__(self, device, max_batch: int = 8192, seed: int = 0, train: bool = True, dropout: float = 0.0, double_q: bool = True,
                 dropout_seed: int | None = None):
        """dropout: Dropout p in [0, 1) after the conv's LeakyReLU; double_q: the DDQN target (False: the DQN max target);
        dropout_seed: key of the mask stream (default: `seed`)."""
        if not 0.0 <= float(dropout) < 1.0:
            raise ValueError(f"dropout must be in [0, 1), got {dropout}")
        self.device = torch.device(device)
        self.ctx = cabi.Context.for_device(self.device)
        self.max_batch = int(max_batch)
        d, P = self.device, cabi.NET_PARAMS
        f32 = dict(dtype=torch.float32, device=d)
        self.params = torch.zeros(P, **f32)
        self.target = torch.zeros(P, **f32)
        self.grads = torch.zeros(P, **f32)
        self.adam_m = torch.zeros(P, **f32)
        self.adam_v = torch.zeros(P, **f32)
        bf = dict(dtype=torch.bfloat16, device=d)
        self.w1_bf16 = torch.zeros((cabi.NET_H1, cabi.NET_IN), **bf)
        self.w2_bf16 = torch.zeros((cabi.NET_H2, cabi.NET_H1), **bf)
        self.w1t_bf16 = torch.zeros((cabi.NET_IN, cabi.NET_H1), **bf)
        self.w2t_bf16 = torch.zeros((cabi.NET_H1, cabi.NET_H2), **bf)
        self.tw1_bf16 = torch.zeros((cabi.NET_H1, cabi.NET_IN), **bf)
        self.tw2_bf16 = torch.zeros((cabi.NET_H2, cabi.NET_H1), **bf)
        nbytes = cabi.lib().maze_dqn_net_workspace_bytes(self.max_batch)
        self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=d)
        ws_ptr = (self.workspace.data_ptr() + 255) & ~255
        self.loss = torch.zeros(1, **f32)
        self.step_count = 0
        self._c = cabi.MazeDqnNet(
            params=self.params.data_ptr(), target=self.target.data_ptr(), grads=self.grads.data_ptr(), adam_m=self.adam_m.data_ptr(),
            adam_v=self.adam_v.data_ptr(), w1_bf16=self.w1_bf16.data_ptr(), w2_bf16=self.w2_bf16.data_ptr(),
            w1t_bf16=self.w1t_bf16.data_ptr(), w2t_bf16=self.w2t_bf16.data_ptr(), tw1_bf16=self.tw1_bf16.data_ptr(),
            tw2_bf16=self.tw2_bf16.data_ptr(), workspace=ws_ptr, loss=self.loss.data_ptr(), max_batch=self.max_batch, reserved=0,
            dropout=float(dropout), update=0 if double_q else 1, eval=0 if train else 1, reserved2=0,
            dropout_seed=int(seed if dropout_seed is None else dropout_seed) & (2 ** 64 - 1), draw=0)
        self.reset_parameters(seed)

    # ---- mode ---------------------------------------------------------------------------------------------------
    @property
    def dropout(self) -> float:
        return float(self._c.dropout)

    @property
    def double_q(self) -> bool:
        return self._c.update == 0

    @property
    def training(self) -> bool:
        return self._c.eval == 0

    def train(self, mode: bool = True):
        """Training mode (dropout active), as nn.Module.train()."""
        self._c.eval = 0 if mode else 1
        return self

    def eval(self):
        """Evaluation mode (no dropout), as nn.Module.eval()."""
        return self.train(False)

    @property
    def draw(self) -> int:
        """The draw counter the next forward / features / backward call uses (then advances by one)."""
        return int(self._c.draw)

    def _next_draw(self):
        """Each forward, features and backward call draws fresh dropout masks: the draw counter advances per call."""
        self._c.draw = (self._c.draw + 1) & (2 ** 64 - 1)

    # ---- parameters -------------------------------------------------------------------------------------------
    def reset_parameters(self, seed: int = 0):
        """torch's default Conv2d / Linear initialisation (kaiming_uniform(a = sqrt 5) = U(+-1/sqrt(fan_in)))."""
        gen = torch.Generator(device="cpu").manual_seed(int(seed))
        sd = {}
        for name, _, shape in _SHAPES:
            used = (cabi.NET_H1, cabi.NET_IN_USED) if name == "fc.0.weight" else shape
            layer = name.rsplit(".", 1)[0]
            fan_in = {"conv.0": 27, "fc.0": cabi.NET_IN_USED, "fc.2": cabi.NET_H1, "fc.4": cabi.NET_H2}[layer]
            bound = 1.0 / math.sqrt(fan_in)
            sd[name] = (torch.rand(used, generator=gen) * 2 - 1) * bound
        self.load_state_dict(sd)

    def state_dict(self, which: str = "source"):
        """Reference-shaped tensors (fc.0.weight is [1024, 1574]); clones."""
        v = _views(self.params if which == "source" else self.target)
        out = {k: t.clone() for k, t in v.items()}
        out["fc.0.weight"] = out["fc.0.weight"][:, :cabi.NET_IN_USED].contiguous()
        return out

    def load_state_dict(self, sd, which: str = "both"):
        for flat in ([self.params, self.target] if which == "both" else [self.params if which == "source" else self.target]):
            v = _views(flat)
            for name, _, shape in _SHAPES:
                src = sd[name].detach().to(device=self.device, dtype=torch.float32)
                if name == "fc.0.weight":
                    v[name].zero_()
                    v[name][:, :cabi.NET_IN_USED] = src
                else:
                    v[name].copy_(src.view(shape))
        self.refresh(0)
        self.refresh(1)

    def refresh(self, which: int):
        rc = cabi.lib().maze_dqn_net_refresh(self.ctx.handle, C.byref(self._c), int(which), cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_dqn_net_refresh")

    def update_target(self):
        """target_net.load_state_dict(source_net.state_dict()) (ddqn_agent.py:161-162)."""
        self.target.copy_(self.params)
        self.refresh(1)   # the target net's bf16 operands: fc1 / fc2 weights and the conv weight image

    # ---- compute ----------------------------------------------------------------------------------------------
    def forward(self, vec: torch.Tensor, win: torch.Tensor, which: int = 0, out: torch.Tensor | None = None) -> torch.Tensor:
        n = vec.shape[0]
        if out is None:
            out = torch.empty((n, 4), dtype=torch.float32, device=self.device)
        rc = cabi.lib().maze_dqn_forward(self.ctx.handle, C.byref(self._c), int(which), cabi.ptr(vec), cabi.ptr(win), n, cabi.ptr(out),
                                         cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_dqn_forward")
        self._next_draw()
        return out

    def features(self, vec, win, which: int = 0, save_idx: bool = False):
        n = vec.shape[0]
        X = torch.empty((n, cabi.NET_IN), dtype=torch.bfloat16, device=self.device)
        idx = torch.empty((n, 1568), dtype=torch.uint8, device=self.device) if save_idx else None
        rc = cabi.lib().maze_dqn_features(self.ctx.handle, C.byref(self._c), int(which), cabi.ptr(vec), cabi.ptr(win), n, cabi.ptr(X),
                                          cabi.ptr(idx), cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_dqn_features")
        self._next_draw()
        return (X, idx) if save_idx else X

    def backward(self, vec, win, next_vec, next_win, action, reward, gamma: float, qsa_out: torch.Tensor | None = None,
                 fc_ready: torch.cuda.Event | None = None):
        """Accumulate d loss / d params into self.grads; the loss lands in self.loss (no sync).  fc_ready: an event that
        is recorded as soon as self.grads[NET_OFF_W1:] (everything but the conv layer) is final."""
        n = vec.shape[0]
        ev = None if fc_ready is None else C.c_void_p(fc_ready.cuda_event)
        rc = cabi.lib().maze_dqn_backward(self.ctx.handle, C.byref(self._c), cabi.ptr(vec), cabi.ptr(win), cabi.ptr(next_vec),
                                          cabi.ptr(next_win), cabi.ptr(action), cabi.ptr(reward), n, float(gamma), cabi.ptr(qsa_out),
                                          ev, cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_dqn_backward")
        self._next_draw()
        return self.loss

    def profile(self, enable: bool):
        """Switch the in-situ launch timing of backward() on or off (one CUDA event after every launch)."""
        self.ctx.check(cabi.lib().maze_dqn_net_profile(self.ctx.handle, int(bool(enable))), "maze_dqn_net_profile")

    def profile_read(self):
        """[(label, ms)] of the last backward() call, in launch order (waits for it to finish)."""
        cap, nb = 96, 64
        ms = (C.c_float * cap)()
        labels = C.create_string_buffer(cap * nb)
        count = C.c_int(0)
        rc = cabi.lib().maze_dqn_net_profile_read(self.ctx.handle, ms, labels, nb, cap, C.byref(count))
        self.ctx.check(rc, "maze_dqn_net_profile_read")
        return [(labels.raw[i * nb:(i + 1) * nb].split(b"\0", 1)[0].decode(), float(ms[i])) for i in range(count.value)]

    def adamw(self, lr: float, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2, grad_scale: float = 1.0,
              clamp: float = 1.0):
        self.step_count += 1
        rc = cabi.lib().maze_dqn_adamw(self.ctx.handle, C.byref(self._c), float(lr), float(betas[0]), float(betas[1]), float(eps),
                                       float(weight_decay), self.step_count, float(grad_scale), float(clamp),
                                       cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_dqn_adamw")

    def train_step(self, vec, win, next_vec, next_win, action, reward, gamma: float, lr: float, all_reduce=None, world: int = 1, **adam):
        """optimize_model (ddqn_agent.py:113-152).  `all_reduce(tensor)` sums the flat gradient over ranks (NCCL)."""
        self.backward(vec, win, next_vec, next_win, action, reward, gamma)
        if all_reduce is not None and world > 1:
            all_reduce(self.grads)
        self.adamw(lr, grad_scale=1.0 / world, **adam)
        return self.loss

    def train_step_overlapped(self, vec, win, next_vec, next_win, action, reward, gamma: float, lr: float, world: int, group=None, **adam):
        """train_step for world > 1 with the gradient all-reduce hidden behind the tail of the backward pass: the fc
        gradients (99.96 % of the buffer) are reduced on a side stream from the moment they are final, while the
        backward-data GEMM and the conv weight gradient still run; the 896 conv floats follow at the end."""
        import torch.distributed as dist
        if getattr(self, "_fc_ready", None) is None:
            self._fc_ready = torch.cuda.Event()
            self._fc_ready.record(torch.cuda.current_stream(self.device))    # materialises the cudaEvent_t
            self._side = torch.cuda.Stream(self.device)
        main = torch.cuda.current_stream(self.device)
        self.backward(vec, win, next_vec, next_win, action, reward, gamma, fc_ready=self._fc_ready)
        with torch.cuda.stream(self._side):
            self._side.wait_event(self._fc_ready)
            work = dist.all_reduce(self.grads[cabi.NET_OFF_W1:], group=group, async_op=True)
        dist.all_reduce(self.grads[:cabi.NET_OFF_W1], group=group)
        work.wait()                       # the current (main) stream waits for the side all-reduce; the host does not
        main.wait_stream(self._side)
        self.adamw(lr, grad_scale=1.0 / world, **adam)
        return self.loss


def gemm_bf16(A: torch.Tensor, B: torch.Tensor, C_out: torch.Tensor, epilogue: int = 0, act: int = 0, bias=None, aux=None,
              tile_n: int = 256, splits: int = 1):
    """C = A . B^T through maze_dqn_gemm_bf16 (test / benchmark hook); epilogue 3: C += A^T . B with A [K, M], B [K, N]."""
    ctx = cabi.Context.for_device(A.device)
    if epilogue == 3:
        K, M = A.shape
        N = B.shape[1]
    else:
        M, K = A.shape
        N = B.shape[0]
    rc = cabi.lib().maze_dqn_gemm_bf16(ctx.handle, cabi.ptr(A), A.stride(0), cabi.ptr(B), B.stride(0), cabi.ptr(C_out), C_out.stride(0), M, N, K,
                                       int(epilogue), int(act), cabi.ptr(bias), cabi.ptr(aux), aux.stride(0) if aux is not None else 0,
                                       int(tile_n), int(splits), cabi.current_stream(A.device))
    ctx.check(rc, "maze_dqn_gemm_bf16")
    return C_out
