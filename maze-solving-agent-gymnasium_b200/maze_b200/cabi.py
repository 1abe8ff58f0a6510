"""ctypes binding of include/maze_b200.h (the drop-in boundary; see INTEGRATION.md)."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

ABI_VERSION = 14
BATCH_BORDERED = 1

# constants mirrored from include/maze_b200.h
META_WORDS = 8
META_H, META_W, META_START, META_GOAL, META_MAX_STEPS, META_FLAGS, META_SOL_LEN, META_SPARE = range(8)
FLAG_TOROIDAL = 1
TAB_OPEN, TAB_CODE_SHIFT, TAB_D4_SHIFT = 0x01, 1, 4
ST_NEEDS_RESET, ST_WON, ST_MOVE_SHIFT, ST_NMOVES_SHIFT = 0x01, 0x02, 2, 4
STEP_AUTORESET, STEP_WIN_NEXT, STEP_WIN_QUEUE, STEP_PACKED, STEP_NO_WIDE = 0x01, 0x02, 0x04, 0x08, 0x10
REC_CODE_SHIFT, REC_TERM_SHIFT, REC_TRUNC_SHIFT, REC_KIND_SHIFT, REC_INDEX_SHIFT = 16, 19, 20, 21, 23
ALGO_RPRIM, ALGO_DFS, ALGO_PRIMKILL = 0, 1, 2
MAX_DIM, GEN_MAX_DIM, WINDOW = 255, 131, 15
METRIC_WORDS = 8
METRIC_NAMES = ("difficulty", "complexity", "L", "DE", "D", "sol_len", "de_count")
PACK_BITMAP, PACK_WALLS = 0, 1
RENDER_TILE = 16
METRIC_EXT_WORDS = 20
METRIC_EXT_NAMES = ("density", "T", "J", "CR", "AC", "FDE", "BDE", "L_DE", "T_DE_AC", "T_DE_FDE", "T_DE_BDE",
                    "D_sharp_AC", "D_sharp_FDE", "D_sharp_BDE", "L_sharp_AC", "L_sharp_FDE", "L_sharp_BDE")
E_NULL, E_RANGE, E_SHAPE, E_ALGO, E_ALIGN = -1, -2, -3, -4, -5


class MazeEnvBatch(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32), ("num_mazes", C.c_int32), ("slot", C.c_int32), ("pool_stride", C.c_int32),
        ("meta", C.c_void_p), ("table", C.c_void_p), ("env_maze", C.c_void_p), ("state", C.c_void_p),
        ("visits", C.c_void_p), ("agent", C.c_void_p), ("target", C.c_void_p), ("best_dir", C.c_void_p),
        ("reward", C.c_void_p), ("terminated", C.c_void_p), ("truncated", C.c_void_p),
        ("ep_return", C.c_void_p), ("stats", C.c_void_p), ("stats_return", C.c_void_p),
        ("queue", C.c_void_p), ("queue_count", C.c_void_p),
        ("visit_cell_stride", C.c_int64), ("visit_env_stride", C.c_int64),
        ("visit_tiled", C.c_int32), ("visit_slot", C.c_int32),
        ("target_dirty", C.c_void_p), ("packed", C.c_void_p),
        ("visit_bits", C.c_void_p), ("visit_bits_pitch", C.c_int32), ("visit_bits_stride", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32),
    ]


class MazeQAgent(C.Structure):
    _fields_ = [
        ("capacity", C.c_int64), ("keys", C.c_void_p), ("q_a", C.c_void_p), ("q_b", C.c_void_p), ("overflow", C.c_void_p),
        ("envs_per_agent", C.c_int32), ("eps_len", C.c_int32), ("eps_lut", C.c_void_p), ("gamma", C.c_void_p),
        ("lr", C.c_double), ("eta", C.c_double),
        ("slot", C.c_void_p), ("steps_done", C.c_void_p), ("last_action", C.c_void_p), ("ep_return", C.c_void_p),
        ("seed", C.c_uint64), ("env_id_base", C.c_int64),
        ("u_tape", C.c_void_p), ("a_tape", C.c_void_p), ("tape_pos", C.c_void_p), ("u_len", C.c_int32), ("a_len", C.c_int32),
    ]


class MazeReplay(C.Structure):
    _fields_ = [
        ("capacity", C.c_int64), ("pushed", C.c_void_p), ("vec", C.c_void_p), ("next_vec", C.c_void_p),
        ("win", C.c_void_p), ("next_win", C.c_void_p), ("action", C.c_void_p), ("reward", C.c_void_p),
        ("stage_vec", C.c_void_p), ("stage_win", C.c_void_p), ("without_replacement", C.c_int32), ("reserved", C.c_int32),
    ]


WINDOW_WORDS = 24
Q_EMPTY = 0xffffffffffffffff
Q_NO_SLOT = 0xffffffff


class MazeStepTrace(C.Structure):
    _fields_ = [("agent", C.c_void_p), ("best_dir", C.c_void_p), ("reward", C.c_void_p), ("terminated", C.c_void_p),
                ("truncated", C.c_void_p)]


class MazeDqnNet(C.Structure):
    _fields_ = [("params", C.c_void_p), ("target", C.c_void_p), ("grads", C.c_void_p), ("adam_m", C.c_void_p), ("adam_v", C.c_void_p),
                ("w1_bf16", C.c_void_p), ("w2_bf16", C.c_void_p), ("w1t_bf16", C.c_void_p), ("w2t_bf16", C.c_void_p),
                ("tw1_bf16", C.c_void_p), ("tw2_bf16", C.c_void_p), ("workspace", C.c_void_p), ("loss", C.c_void_p),
                ("max_batch", C.c_int32), ("reserved", C.c_int32), ("dropout", C.c_float), ("update", C.c_int32), ("eval", C.c_int32),
                ("reserved2", C.c_int32), ("dropout_seed", C.c_uint64), ("draw", C.c_uint64)]


# flat parameter layout of the DQN / DDQN net (include/maze_b200.h MAZE_NET_*)
NET_IN, NET_IN_USED, NET_H1, NET_H2 = 1600, 1574, 1024, 512
NET_OFF_CONV_W, NET_OFF_CONV_B, NET_OFF_W1 = 0, 864, 896
NET_OFF_B1 = NET_OFF_W1 + NET_H1 * NET_IN
NET_OFF_W2 = NET_OFF_B1 + NET_H1
NET_OFF_B2 = NET_OFF_W2 + NET_H2 * NET_H1
NET_OFF_W3 = NET_OFF_B2 + NET_H2
NET_OFF_B3 = NET_OFF_W3 + 4 * NET_H2
NET_PARAMS = NET_OFF_B3 + 4


class MazeError(RuntimeError):
    pass


_lib = None

# name -> (restype, argtypes); every symbol declared in include/maze_b200.h
SIGNATURES = {
    "maze_abi_version": (C.c_int, []),
    "maze_ctx_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "maze_ctx_destroy": (None, [C.c_void_p]),
    "maze_last_error": (C.c_char_p, [C.c_void_p]),
    "maze_reward_lut": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double)]),
    "maze_fields": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "maze_step": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_void_p, C.c_uint32, C.c_void_p]),
    "maze_step_decode_host": (C.c_int, [C.c_void_p, C.c_int64] + [C.c_void_p] * 7),
    "maze_bench_scatter_rmw": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_uint32,
                                         C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "maze_step_many": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_void_p, C.c_int, C.c_uint32, C.POINTER(MazeStepTrace),
                                 C.c_int, C.c_void_p]),
    "maze_reset": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_void_p, C.c_void_p]),
    "maze_generate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "maze_curriculum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 8 + [C.c_void_p]),
    "maze_window": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "maze_direction_mask": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_int, C.c_void_p, C.c_void_p]),
    "maze_q_epsilon_lut": (C.c_int, [C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double), C.c_int]),
    "maze_q_act": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.POINTER(MazeQAgent), C.c_void_p, C.c_void_p]),
    "maze_q_update": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.POINTER(MazeQAgent), C.c_void_p]),
    "maze_q_rollout": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.POINTER(MazeQAgent), C.c_int, C.c_uint32, C.c_void_p]),
    "maze_dqn_observe": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.POINTER(MazeReplay), C.c_void_p]),
    "maze_dqn_push": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.POINTER(MazeReplay), C.c_void_p, C.c_void_p]),
    "maze_dqn_sample": (C.c_int, [C.c_void_p, C.POINTER(MazeReplay), C.c_int, C.c_uint64, C.c_uint64] + [C.c_void_p] * 7),
    "maze_dqn_select": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                  C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p]),
    "maze_difficulty": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p]),
    "maze_dqn_net_workspace_bytes": (C.c_int64, [C.c_int]),
    "maze_dqn_net_refresh": (C.c_int, [C.c_void_p, C.POINTER(MazeDqnNet), C.c_int, C.c_void_p]),
    "maze_dqn_forward": (C.c_int, [C.c_void_p, C.POINTER(MazeDqnNet), C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "maze_dqn_features": (C.c_int, [C.c_void_p, C.POINTER(MazeDqnNet), C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "maze_dqn_backward": (C.c_int, [C.c_void_p, C.POINTER(MazeDqnNet)] + [C.c_void_p] * 6 + [C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "maze_dqn_adamw": (C.c_int, [C.c_void_p, C.POINTER(MazeDqnNet)] + [C.c_float] * 5 + [C.c_int64, C.c_float, C.c_float, C.c_void_p]),
    "maze_regen_swap": (C.c_int, [C.c_void_p] + [C.c_void_p] * 7 + [C.c_int] + [C.c_void_p] * 2 + [C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.c_int]
                        + [C.c_void_p] * 5),
    "maze_regen_prepare": (C.c_int, [C.c_void_p] + [C.c_void_p] * 3 + [C.c_int] * 7 + [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 2 + [C.c_int]
                           + [C.c_void_p] * 3),
    "maze_regen_publish": (C.c_int, [C.c_void_p] + [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 2 + [C.c_int, C.c_void_p]),
    "maze_dqn_net_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "maze_dqn_net_profile_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "maze_dqn_sample_packed": (C.c_int, [C.c_void_p, C.POINTER(MazeReplay), C.c_int, C.c_uint64, C.c_uint64] + [C.c_void_p] * 7),
    "maze_dqn_gemm_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "maze_sizeof": (C.c_int, [C.c_int]),
    "maze_render": (C.c_int, [C.c_void_p, C.POINTER(MazeEnvBatch), C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "maze_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                            C.c_void_p]),
    "maze_unpack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                              C.c_void_p]),
    "maze_collection_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p]),
    "maze_difficulty_ext": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
}


def lib():
    """The loaded C-ABI library.  No fallback: a missing library is a hard error."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MazeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        if l.maze_abi_version() != ABI_VERSION:
            raise MazeError(f"ABI mismatch: library {l.maze_abi_version()} vs binding {ABI_VERSION}; rebuild")
        _lib = l
    return _lib


class Context:
    """One maze_ctx per (process, device)."""

    _by_device: dict = {}

    def __init__(self, device_index: int):
        self.device_index = int(device_index)
        self._h = C.c_void_p()
        rc = lib().maze_ctx_create(C.byref(self._h), self.device_index)
        if rc != 0:
            raise MazeError(f"maze_ctx_create(device={device_index}) failed with code {rc} "
                            "(a CUDA device is required; there is no CPU fallback)")

    @classmethod
    def for_device(cls, device) -> "Context":
        import torch
        dev = torch.device(device)
        if dev.type != "cuda":
            raise MazeError(f"device {dev} is not CUDA: the maze kernels are sm_100a only, there is no CPU path")
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        if idx not in cls._by_device:
            cls._by_device[idx] = cls(idx)
        return cls._by_device[idx]

    @property
    def handle(self):
        return self._h

    def check(self, rc: int, what: str):
        if rc != 0:
            msg = lib().maze_last_error(self._h)
            raise MazeError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")


def reward_lut(kind: int):
    """Host copy of a reward LUT (works without a GPU)."""
    import numpy as np
    out = (C.c_double * 256)()
    rc = lib().maze_reward_lut(None, kind, out)
    if rc != 0:
        raise MazeError(f"maze_reward_lut({kind}) -> {rc}")
    return np.array(out, dtype=np.float64)


def reward_table():
    """float64 [4, 256]: reward = table[kind, index] of a packed step record (include/maze_b200.h MAZE_REC_*)."""
    import numpy as np
    t = np.zeros((4, 256), dtype=np.float64)
    t[0], t[1] = reward_lut(0), reward_lut(1)
    t[2, :3] = reward_lut(2)[:3]
    t[3, :3] = (0.0, 1.0, -1.0)
    return t


def decode_records(records, shape=None, toroidal=None):
    """Packed step records (uint32 [n]) -> dict(agent [n, 2] int32, best_dir [n, 2] int32, reward [n] float64,
    terminated / truncated [n] bool), bit-identical to maze_step's wide outputs.  Runs the library's host-side C loop
    (maze_step_decode_host); shape [n, 2] int32 and toroidal [n] uint8 are needed for toroidal envs only."""
    import numpy as np
    rec = np.ascontiguousarray(records).view(np.uint32).reshape(-1)
    n = rec.shape[0]
    out = dict(agent=np.empty((n, 2), np.int32), best_dir=np.empty((n, 2), np.int32), reward=np.empty(n, np.float64),
               terminated=np.empty(n, np.uint8), truncated=np.empty(n, np.uint8))
    sh = None if shape is None else np.ascontiguousarray(shape, dtype=np.int32)
    to = None if toroidal is None else np.ascontiguousarray(toroidal, dtype=np.uint8)
    rc = lib().maze_step_decode_host(rec.ctypes.data, n, None if sh is None else sh.ctypes.data, None if to is None else to.ctypes.data,
                                     out["agent"].ctypes.data, out["best_dir"].ctypes.data, out["reward"].ctypes.data,
                                     out["terminated"].ctypes.data, out["truncated"].ctypes.data)
    if rc != 0:
        raise MazeError(f"maze_step_decode_host -> {rc}")
    out["terminated"], out["truncated"] = out["terminated"].view(np.bool_), out["truncated"].view(np.bool_)
    return out


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream(device):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
