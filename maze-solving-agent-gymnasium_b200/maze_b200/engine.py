"""Host-side engine: device-resident maze pool + structure-of-arrays env batch.

PyTorch is used for device memory and streams only; all compute goes through the C ABI.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import cabi

ALGO_IDS = {"r-prim": cabi.ALGO_RPRIM, "dfs": cabi.ALGO_DFS, "prim&kill": cabi.ALGO_PRIMKILL}
ALGO_NAMES = {v: k for k, v in ALGO_IDS.items()}


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def check_shape(shape, limit=cabi.MAX_DIM):
    H, W = int(shape[0]), int(shape[1])
    if H % 2 == 0 or W % 2 == 0:
        # the reference crashes with IndexError on even shapes (lib/maze_generation.py:197,203)
        raise ValueError(f"maze block shape must be odd (2N+1), got {(H, W)}")
    if H < 5 or W < 5 or H > limit or W > limit:
        raise ValueError(f"maze block shape {(H, W)} outside [5, {limit}]")
    return H, W


class MazePool:
    """M maze slots on one GPU: block grids, metadata records and step tables."""

    def __init__(self, num_mazes: int, max_shape, device="cuda"):
        self.device = torch.device(device)
        self.ctx = cabi.Context.for_device(self.device)
        self.max_shape = check_shape(max_shape)
        self.num_mazes = int(num_mazes)
        self.slot = _round_up(self.max_shape[0] * self.max_shape[1], 16)
        d = self.device
        self.grids = torch.zeros((self.num_mazes, self.slot), dtype=torch.uint8, device=d)
        self.table = torch.zeros((self.num_mazes, self.slot), dtype=torch.uint8, device=d)
        self.meta = torch.zeros((self.num_mazes, cabi.META_WORDS), dtype=torch.int32, device=d)
        # host-side knowledge "some slot may be toroidal" (conservative: set by every path that writes slot records, cleared only
        # when all slots are reconfigured as bordered): batches derive MAZE_BATCH_BORDERED from it without a device read
        self.any_toroidal = False

    # -- construction from host block grids (parity tests, reference-generated mazes)
    @classmethod
    def from_grids(cls, grids: Sequence[np.ndarray], starts, goals, toroidal, device="cuda", max_shape=None):
        M = len(grids)
        tor = [bool(toroidal)] * M if isinstance(toroidal, (bool, int)) else [bool(t) for t in toroidal]
        shapes = [np.asarray(g).shape for g in grids]
        if max_shape is None:
            max_shape = (max(s[0] for s in shapes), max(s[1] for s in shapes))
        pool = cls(M, max_shape, device)
        pool.upload(range(M), grids, starts, goals, tor)
        return pool

    def upload(self, ids, grids, starts, goals, toroidal):
        ids = list(ids)
        hg = np.zeros((len(ids), self.slot), dtype=np.uint8)
        hm = np.zeros((len(ids), cabi.META_WORDS), dtype=np.int32)
        toroidal = list(toroidal)
        self.any_toroidal = self.any_toroidal or any(bool(t) for t in toroidal)
        for k, (g, s, t, tor) in enumerate(zip(grids, starts, goals, toroidal)):
            g = np.asarray(g, dtype=np.uint8)
            H, W = check_shape(g.shape)
            if H * W > self.slot:
                raise ValueError(f"maze {g.shape} does not fit slot of {self.slot} bytes")
            hg[k, :H * W] = g.reshape(-1)
            hg[k, int(t[0]) * W + int(t[1])] = 2   # the goal block carries 2 (lib/maze_generation.py:33)
            hm[k, cabi.META_H], hm[k, cabi.META_W] = H, W
            hm[k, cabi.META_START] = int(s[0]) | (int(s[1]) << 16)
            hm[k, cabi.META_GOAL] = int(t[0]) | (int(t[1]) << 16)
            hm[k, cabi.META_FLAGS] = cabi.FLAG_TOROIDAL if tor else 0
        idx = torch.as_tensor(ids, dtype=torch.long, device=self.device)
        self.grids[idx] = torch.from_numpy(hg).to(self.device)
        self.meta[idx] = torch.from_numpy(hm).to(self.device)
        self.compute_fields(ids)

    def compute_fields(self, ids=None):
        """Step table + step budget for the given slots (all if None)."""
        if ids is None:
            ids_t, n = None, self.num_mazes
        else:
            ids_t = torch.as_tensor(list(ids), dtype=torch.int32, device=self.device)
            n = ids_t.numel()
        rc = cabi.lib().maze_fields(self.ctx.handle, cabi.ptr(self.grids), cabi.ptr(self.meta), cabi.ptr(self.table),
                                    cabi.ptr(ids_t), n, self.slot, cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_fields")

    def generate(self, ids=None, shapes=None, algorithms="r-prim", toroidal=False, seed=0, slot_id_base=0,
                 count_dev=None, configure=True, candidates=1, difficulty_out=None):
        """Generate mazes on the device into the given slots (all if None).

        shapes / algorithms / toroidal may be scalars or per-slot sequences.  With configure=False
        the per-slot meta (H, W, FLAGS) already on the device is reused (regeneration).
        candidates=6 reproduces BaseMazeEnv.generate_maze (keep the least difficult of six draws);
        difficulty_out: optional float64 [n] device tensor receiving the kept maze's difficulty."""
        if ids is None:
            ids_list = list(range(self.num_mazes))
            ids_t = None
        elif isinstance(ids, torch.Tensor):
            ids_list, ids_t = None, ids.to(device=self.device, dtype=torch.int32).contiguous()
        else:
            ids_list = [int(i) for i in ids]
            ids_t = torch.as_tensor(ids_list, dtype=torch.int32, device=self.device)
        n = self.num_mazes if ids_t is None else ids_t.numel()
        max_h, max_w = self.max_shape
        if configure:
            assert ids_list is not None
            k = len(ids_list)
            if shapes is None:
                shapes = self.max_shape
            def record(shape, a, t):
                H, W = check_shape(shape, cabi.GEN_MAX_DIM - 2 - (2 if t else 0))   # toroidal mazes are generated at shape + 2
                if H * W > self.slot:
                    raise ValueError(f"shape {(H, W)} does not fit the pool slot")
                if isinstance(a, str):
                    if a not in ALGO_IDS:
                        raise ValueError(f"unknown maze generation algorithm {a!r} (expected one of {list(ALGO_IDS)})")
                    a = ALGO_IDS[a]
                elif a not in ALGO_NAMES:
                    raise ValueError(f"unknown maze generation algorithm id {a}")
                return (H, W, (cabi.FLAG_TOROIDAL if t else 0) | (int(a) << 8))

            uniform = (isinstance(shapes[0], (int, np.integer)) and isinstance(algorithms, (str, int))
                       and isinstance(toroidal, (bool, int)))
            if uniform:   # one record for every slot: no per-slot host work
                hm = np.tile(np.array(record(shapes, algorithms, toroidal), dtype=np.int32), (k, 1))
            else:
                shp = [shapes] * k if isinstance(shapes[0], (int, np.integer)) else list(shapes)
                alg = [algorithms] * k if isinstance(algorithms, (str, int)) else list(algorithms)
                tor = [toroidal] * k if isinstance(toroidal, (bool, int)) else list(toroidal)
                cache = {}
                hm = np.zeros((k, 3), dtype=np.int32)
                for q in range(k):
                    key = (tuple(shp[q]), alg[q], bool(tor[q]))
                    if key not in cache:
                        cache[key] = record(*key)
                    hm[q] = cache[key]
            some_tor = bool((hm[:, 2] & cabi.FLAG_TOROIDAL).any())
            self.any_toroidal = some_tor if len(ids_list) == self.num_mazes and len(set(ids_list)) == self.num_mazes else (self.any_toroidal or some_tor)
            cfg = torch.from_numpy(hm).to(self.device)
            idx = torch.as_tensor(ids_list, dtype=torch.long, device=self.device)
            self.meta[idx, cabi.META_H] = cfg[:, 0]
            self.meta[idx, cabi.META_W] = cfg[:, 1]
            self.meta[idx, cabi.META_FLAGS] = cfg[:, 2]
        rc = cabi.lib().maze_generate(self.ctx.handle, cabi.ptr(self.grids), cabi.ptr(self.meta), cabi.ptr(self.table),
                                      cabi.ptr(ids_t), cabi.ptr(count_dev), n, self.slot, max_h, max_w,
                                      int(seed) & (2**64 - 1), int(slot_id_base), int(candidates),
                                      cabi.ptr(difficulty_out), cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_generate")

    def curriculum(self, ids, count_dev, wins: torch.Tensor, grow: int = 0, schedule=((5, "prim&kill"), (10, "dfs"))):
        """Advance the curriculum of the queued slots on the device (see maze_curriculum): wins += 1,
        shape += grow while it fits the pool, generator switched by the win thresholds of `schedule`
        (None / () keeps the generator)."""
        sched = list(schedule or ())
        (wa, aa), (wb, ab) = (sched + [(0, None), (0, None)])[:2]
        code = lambda a: -1 if a is None else (ALGO_IDS[a] if isinstance(a, str) else int(a))  # noqa: E731
        ids_t = ids.to(device=self.device, dtype=torch.int32).contiguous()
        rc = cabi.lib().maze_curriculum(self.ctx.handle, cabi.ptr(self.meta), cabi.ptr(wins), cabi.ptr(ids_t), cabi.ptr(count_dev),
                                        ids_t.numel(), int(grow), self.max_shape[0], self.max_shape[1], int(wa), code(aa),
                                        int(wb), code(ab), cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_curriculum")

    def difficulty(self, ids=None, extended: bool = False):
        """float64 [n, 8] metric records (cabi.METRIC_NAMES) of the given slots (all if None):
        McClendon difficulty / complexity, Kim-Crawfis L / DE / D, solution length, dead-end count.
        extended=True returns (records, ext) with ext float64 [n, 20] (cabi.METRIC_EXT_NAMES): the
        Kim-Crawfis metrics nothing in the reference calls (density, T, J, CR, AC / FDE / BDE, L_DE and the
        per-type T_DE / D_sharp / L_sharp sums)."""
        if ids is None:
            ids_t, n = None, self.num_mazes
        else:
            ids_t = torch.as_tensor(ids, dtype=torch.int32, device=self.device).contiguous()
            n = ids_t.numel()
        out = torch.empty((n, cabi.METRIC_WORDS), dtype=torch.float64, device=self.device)
        if extended:
            ext = torch.empty((n, cabi.METRIC_EXT_WORDS), dtype=torch.float64, device=self.device)
            rc = cabi.lib().maze_difficulty_ext(self.ctx.handle, cabi.ptr(self.grids), cabi.ptr(self.meta), cabi.ptr(ids_t), n,
                                                self.slot, self.max_shape[0], self.max_shape[1], cabi.ptr(out), cabi.ptr(ext),
                                                cabi.current_stream(self.device))
            self.ctx.check(rc, "maze_difficulty_ext")
            return out, ext
        rc = cabi.lib().maze_difficulty(self.ctx.handle, cabi.ptr(self.grids), cabi.ptr(self.meta), cabi.ptr(ids_t), n,
                                        self.slot, self.max_shape[0], self.max_shape[1], cabi.ptr(out),
                                        cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_difficulty")
        return out

    # -- checkpoint / resume (SURVEY.md section 5: the reference keeps no checkpoints; env state here is a
    #    handful of SoA tensors, so a state dict of them is a complete checkpoint)
    def state_dict(self):
        return {"max_shape": tuple(self.max_shape), "grids": self.grids, "table": self.table, "meta": self.meta}

    def load_state_dict(self, sd):
        if tuple(sd["max_shape"]) != tuple(self.max_shape) or sd["grids"].shape != self.grids.shape:
            raise ValueError("checkpoint was taken from a pool of another size / shape")
        for k in ("grids", "table", "meta"):
            getattr(self, k).copy_(sd[k])
        self.any_toroidal = bool((self.meta[:, cabi.META_FLAGS] & cabi.FLAG_TOROIDAL).any().item())

    # -- host views (tests, facade)
    def meta_host(self):
        return self.meta.cpu().numpy()

    def grid_host(self, m: int) -> np.ndarray:
        mh = self.meta[m].cpu().numpy()
        H, W = int(mh[cabi.META_H]), int(mh[cabi.META_W])
        return self.grids[m, :H * W].cpu().numpy().reshape(H, W)

    def table_host(self, m: int) -> np.ndarray:
        mh = self.meta[m].cpu().numpy()
        H, W = int(mh[cabi.META_H]), int(mh[cabi.META_W])
        return self.table[m, :H * W].cpu().numpy().reshape(H, W)


class MazeBatch:
    """B environments over a MazePool; the SoA buffers of `maze_env_batch`."""

    def __init__(self, pool: MazePool, num_envs: int, env_maze=None, stats: bool = False, pool_stride: int = 1,
                 queue: bool = False, visit_layout: str = "cell", visit_bits: bool = False):
        """visit_layout: "cell" = [slot, B] (best for the -v0 step: envs sharing a block share lines),
        "tile" = env-major with 4x4 block tiles per 32-byte sector (a walking agent stays in a sector).
        visit_bits: also keep the one-bit-per-block "visited this episode" map (1 KB per env at 81 x 81) that the -v1
        window and the replay encode read their non_visited channel from."""
        if visit_layout not in ("cell", "tile"):
            raise ValueError("visit_layout must be 'cell' or 'tile'")
        self.visit_layout = visit_layout
        self.pool = pool
        self.device = pool.device
        self.ctx = pool.ctx
        B = self.num_envs = int(num_envs)
        d = self.device
        if env_maze is None:
            env_maze = torch.arange(B, dtype=torch.int32, device=d) % pool.num_mazes
        self.env_maze = torch.as_tensor(env_maze, dtype=torch.int32, device=d).contiguous()
        assert self.env_maze.shape == (B,)
        self.state = torch.zeros(B, dtype=torch.int64, device=d)
        mh, mw = pool.max_shape
        self.visit_slot = pool.slot if visit_layout != "tile" else _round_up(16 * ((mh + 3) // 4) * ((mw + 3) // 4), 16)
        self.visits = torch.zeros((self.visit_slot, B) if visit_layout == "cell" else (B, self.visit_slot),
                                  dtype=torch.int16, device=d)
        self.window = None       # float32 [B, 3, 15, 15], allocated by window()
        self.agent_norm = None   # float64 [B, 2]
        self.target_norm = None
        self.dir_mask = None     # float32 [B, 4]
        self.agent = torch.zeros((B, 2), dtype=torch.int32, device=d)
        self.target = torch.zeros((B, 2), dtype=torch.int32, device=d)
        self.best_dir = torch.zeros((B, 2), dtype=torch.int32, device=d)
        self.reward = torch.zeros(B, dtype=torch.float64, device=d)
        self.terminated = torch.zeros(B, dtype=torch.uint8, device=d)
        self.truncated = torch.zeros(B, dtype=torch.uint8, device=d)
        self.ep_return = torch.zeros(B, dtype=torch.float64, device=d) if stats else None
        self.stats = torch.zeros(4, dtype=torch.int64, device=d) if stats else None
        self.stats_return = torch.zeros(1, dtype=torch.float64, device=d) if stats else None
        self.queue = torch.zeros(B, dtype=torch.int32, device=d) if queue else None
        self.queue_count = torch.zeros(1, dtype=torch.int32, device=d) if queue else None
        self.target_dirty = torch.zeros(1, dtype=torch.int32, device=d)   # set by launches that write `target`
        self.packed = torch.zeros(B, dtype=torch.int32, device=d)         # packed step records (cabi.STEP_PACKED)
        self.visit_bits_pitch = (mw + 31) // 32
        self.visit_bits_stride = _round_up(mh * self.visit_bits_pitch, 4)
        self.visit_bits = torch.zeros((B, self.visit_bits_stride), dtype=torch.int32, device=d) if visit_bits else None
        self.pool_stride = int(pool_stride)
        self._c = self._make_struct()

    _CKPT = ("env_maze", "state", "visits", "agent", "target", "best_dir", "reward", "terminated", "truncated",
             "ep_return", "stats", "stats_return", "queue", "queue_count", "target_dirty", "visit_bits")

    def state_dict(self):
        """Everything a later step depends on (the visit counters included: [slot, B] int16, by far the largest
        entry).  Tensors are references, not copies: clone or torch.save them before stepping on."""
        sd = {k: getattr(self, k) for k in self._CKPT if getattr(self, k) is not None}
        sd["visit_layout"] = self.visit_layout
        return sd

    def load_state_dict(self, sd):
        if sd["visit_layout"] != self.visit_layout or sd["state"].shape != self.state.shape:
            raise ValueError("checkpoint was taken from a batch of another size / visit layout")
        for k in self._CKPT:
            if getattr(self, k) is not None and k in sd:
                getattr(self, k).copy_(sd[k])
        self.target_dirty.fill_(1)   # host mirrors of `target` must be refreshed after a restore

    def _make_struct(self) -> cabi.MazeEnvBatch:
        p = self.pool
        return cabi.MazeEnvBatch(
            num_envs=self.num_envs, num_mazes=p.num_mazes, slot=p.slot, pool_stride=self.pool_stride,
            meta=p.meta.data_ptr(), table=p.table.data_ptr(), env_maze=self.env_maze.data_ptr(),
            state=self.state.data_ptr(), visits=self.visits.data_ptr(), agent=self.agent.data_ptr(),
            target=self.target.data_ptr(), best_dir=self.best_dir.data_ptr(), reward=self.reward.data_ptr(),
            terminated=self.terminated.data_ptr(), truncated=self.truncated.data_ptr(),
            ep_return=None if self.ep_return is None else self.ep_return.data_ptr(),
            stats=None if self.stats is None else self.stats.data_ptr(),
            stats_return=None if self.stats_return is None else self.stats_return.data_ptr(),
            queue=None if self.queue is None else self.queue.data_ptr(),
            queue_count=None if self.queue_count is None else self.queue_count.data_ptr(),
            visit_cell_stride=self.num_envs if self.visit_layout == "cell" else 1,
            visit_env_stride=1 if self.visit_layout == "cell" else self.visit_slot,
            visit_tiled=1 if self.visit_layout == "tile" else 0, visit_slot=self.visit_slot,
            target_dirty=self.target_dirty.data_ptr(), packed=self.packed.data_ptr(),
            visit_bits=None if self.visit_bits is None else self.visit_bits.data_ptr(),
            visit_bits_pitch=self.visit_bits_pitch, visit_bits_stride=self.visit_bits_stride,
            flags=0 if p.any_toroidal else cabi.BATCH_BORDERED, reserved=0)   # kept current by sync_flags()

    def sync_flags(self):
        """MAZE_BATCH_BORDERED follows the pool (a pool may be reconfigured after the batch was built); host-only, no device read.
        Called before the launches that read the flag (maze_window, maze_dqn_observe / _push)."""
        want = 0 if self.pool.any_toroidal else cabi.BATCH_BORDERED
        if self._c.flags != want:
            self._c.flags = want

    def view_struct(self, lo: int, hi: int) -> cabi.MazeEnvBatch:
        """maze_env_batch over the envs [lo, hi) of this batch: the same buffers with every per-env pointer advanced by
        lo (the visit array by lo env strides), so that a launch on the view touches exactly those envs.  The shared
        fields (statistics, regeneration queue, target_dirty) stay shared."""
        if not 0 <= lo < hi <= self.num_envs:
            raise ValueError("env range outside the batch")
        c = cabi.MazeEnvBatch.from_buffer_copy(self._c)
        c.num_envs = hi - lo
        for name, per_env_bytes in (("env_maze", 4), ("state", 8), ("agent", 8), ("target", 8), ("best_dir", 8), ("reward", 8),
                                    ("terminated", 1), ("truncated", 1), ("ep_return", 8), ("packed", 4)):
            base = getattr(self._c, name)
            if base:
                setattr(c, name, base + lo * per_env_bytes)
        c.visits = self._c.visits + lo * self._c.visit_env_stride * 2
        if self._c.visit_bits:
            c.visit_bits = self._c.visit_bits + lo * self.visit_bits_stride * 4
        return c

    def step_view(self, view: cabi.MazeEnvBatch, actions_ptr, mode: int, stream):
        """maze_step on a view_struct(); actions_ptr points at the view's first action; `stream` is a raw cudaStream_t."""
        rc = cabi.lib().maze_step(self.ctx.handle, C.byref(view), actions_ptr, mode, stream)
        self.ctx.check(rc, "maze_step")

    def reset(self, mask: Optional[torch.Tensor] = None):
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        rc = cabi.lib().maze_reset(self.ctx.handle, C.byref(self._c), cabi.ptr(mask), cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_reset")

    def step(self, actions: torch.Tensor, mode: int = 0):
        """actions: uint8 [B] on the device."""
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        assert actions.numel() == self.num_envs
        rc = cabi.lib().maze_step(self.ctx.handle, C.byref(self._c), cabi.ptr(actions), mode,
                                  cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_step")

    def step_many(self, actions: torch.Tensor, mode: int = 0, trace: bool = False, chunk_envs: int = 0):
        """K consecutive transitions for action sequences known in advance: actions uint8 [K, B] on the
        device.  Bit-identical to K step() calls; with trace=True returns the per-step outputs
        dict(agent [K,B,2], best_dir [K,B,2], reward [K,B], terminated [K,B], truncated [K,B])."""
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        K = actions.shape[0]
        assert actions.shape == (K, self.num_envs)
        out, tr = None, None
        if trace:
            d, B = self.device, self.num_envs
            out = dict(agent=torch.empty((K, B, 2), dtype=torch.int32, device=d), best_dir=torch.empty((K, B, 2), dtype=torch.int32, device=d),
                       reward=torch.empty((K, B), dtype=torch.float64, device=d), terminated=torch.empty((K, B), dtype=torch.uint8, device=d),
                       truncated=torch.empty((K, B), dtype=torch.uint8, device=d))
            tr = cabi.MazeStepTrace(**{k: v.data_ptr() for k, v in out.items()})
        rc = cabi.lib().maze_step_many(self.ctx.handle, C.byref(self._c), cabi.ptr(actions), int(K), int(mode),
                                       C.byref(tr) if tr is not None else None, int(chunk_envs), cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_step_many")
        return out

    def compute_window(self):
        """Enriched observation of the current positions: fills self.window [B,3,15,15] float32 and
        self.agent_norm / self.target_norm [B,2] float64 (agent / maze_shape, target / maze_shape)."""
        if self.window is None:
            d, B = self.device, self.num_envs
            self.window = torch.empty((B, 3, cabi.WINDOW, cabi.WINDOW), dtype=torch.float32, device=d)
            self.agent_norm = torch.empty((B, 2), dtype=torch.float64, device=d)
            self.target_norm = torch.empty((B, 2), dtype=torch.float64, device=d)
        self.sync_flags()
        rc = cabi.lib().maze_window(self.ctx.handle, C.byref(self._c), cabi.ptr(self.window), cabi.ptr(self.agent_norm),
                                    cabi.ptr(self.target_norm), cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_window")
        return self.window

    def render(self, env_ids=None) -> torch.Tensor:
        """uint8 [n, 16 H, 16 W, 3] frames of the given envs (all if None -- 5 MB per 81 x 81 env): the
        picture MazeViewTemplate keeps on its surface (lib/maze_view.py:88-104,148-152)."""
        ids_t = None if env_ids is None else torch.as_tensor(list(env_ids), dtype=torch.int32, device=self.device)
        n = self.num_envs if ids_t is None else ids_t.numel()
        H, W = self.pool.max_shape
        out = torch.empty((n, H * cabi.RENDER_TILE, W * cabi.RENDER_TILE, 3), dtype=torch.uint8, device=self.device)
        rc = cabi.lib().maze_render(self.ctx.handle, C.byref(self._c), cabi.ptr(ids_t), n, cabi.ptr(out), out.shape[1], out.shape[2],
                                    cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_render")
        return out

    def direction_mask(self, probs: bool = False):
        """float32 [B, 4] get_mask_direction of every env (action order down, up, right, left)."""
        if self.dir_mask is None:
            self.dir_mask = torch.empty((self.num_envs, 4), dtype=torch.float32, device=self.device)
        rc = cabi.lib().maze_direction_mask(self.ctx.handle, C.byref(self._c), int(bool(probs)), cabi.ptr(self.dir_mask),
                                            cabi.current_stream(self.device))
        self.ctx.check(rc, "maze_direction_mask")
        return self.dir_mask

    def state_host(self):
        s = self.state.cpu().numpy().view(np.uint64)
        return dict(r=(s & 0xff).astype(int), c=((s >> 8) & 0xff).astype(int), consec=((s >> 16) & 0xff).astype(int),
                    flags=((s >> 24) & 0xff).astype(int), steps=((s >> 32) & 0xffff).astype(int),
                    epoch=((s >> 48) & 0xff).astype(int), tab=((s >> 56) & 0xff).astype(int))
