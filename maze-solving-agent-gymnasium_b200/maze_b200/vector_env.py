"""MazeVectorEnv: thousands to millions of maze environments per GPU behind the gymnasium
VectorEnv protocol (reset / step / autoreset), backed by the sm_100a kernels.

Semantics per env are the reference's (gymnasium_env/envs/base_maze_env.py): same observation
dict keys and values, same reward, same termination / truncation rules.  `step` returns the
standard gymnasium order (obs, reward, terminated, truncated, info); `reference_order=True`
returns the reference's swapped order (obs, reward, truncated, terminated, info)
(base_maze_env.py:210).

Autoreset is gymnasium 1.x "next-step": the step after an episode ends ignores the action and
returns the reset observation with reward 0.  What happens to the maze on that reset follows the
reference's trainers (lib/trainers/off_policy_trainer.py:60-71): a truncated episode replays the
same maze; after a win `on_win` decides: "keep" (BaseMazeEnv.reset never changes the maze),
"next" (move to the next maze of the pool) or "regenerate" (a fresh maze is generated on the
device into the env's own slot, the analogue of update_maze()).
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Optional

import numpy as np
import torch

from . import cabi
from .engine import ALGO_IDS, MazeBatch, MazePool

from . import _gym as _gymshim

_gym = None
if _gymshim.HAVE_GYMNASIUM:  # pragma: no cover - gymnasium is absent from the build image
    import gymnasium as _gym
_VectorBase = _gymshim.VectorEnv


class _LazyInfo(dict):
    """info dict whose 'distance' (base_maze_env.py:124-134) is computed on first access."""

    def __init__(self, env):
        super().__init__()
        self._env = env

    def __missing__(self, key):
        if key == "distance":
            b = self._env.batch
            v = (b.agent - b.target).abs().sum(dim=1).to(torch.float64)
            self[key] = v
            return v
        raise KeyError(key)

    def __contains__(self, key):
        return key == "distance" or super().__contains__(key)


class _ActionSpace:
    def __init__(self, n, num_envs=None, seed=None):
        self.n = n
        self._num = num_envs
        self._rng = np.random.default_rng(seed)

    def sample(self):
        if self._num is None:
            return int(self._rng.integers(self.n))
        return self._rng.integers(0, self.n, size=self._num).astype(np.uint8)


class MazeVectorEnv(_VectorBase):
    def __init__(self, num_envs: int, shape=(81, 81), topology: str = "euclid", algorithms="r-prim",
                 num_mazes: Optional[int] = None, device="cuda", seed: int = 0, autoreset: bool = True,
                 on_win: str = "keep", reference_order: bool = False, stats: bool = True,
                 slot_id_base: int = 0, pool: Optional[MazePool] = None, env_maze=None, enrich: bool = False,
                 candidates: int = 1, start_shape=None, grow: int = 0, algorithm_schedule=None, visit_layout=None,
                 regenerate_ahead: Optional[int] = None):
        """enrich=True gives the -v1 observation (normalised agent / target, 15x15 window);
        candidates=6 makes every generated maze the least difficult of six (generate_maze).
        Curriculum (on_win="regenerate"): `shape` is the maximum block shape; mazes start at
        `start_shape` (one shape or one per maze) and grow by `grow` blocks per win
        (variable-size envs: START_SHAPE and +(4, 4), simple_variable_maze_env.py:17,97);
        `algorithm_schedule` = ((wins, algorithm), ...) switches a slot's generator by its win count
        (off_policy_trainer.py:302-310: ((5, "prim&kill"), (10, "dfs"))).
        regenerate_ahead (on_win="regenerate", with or without a curriculum; None = the default, 3; 0 turns it off): keep
        the next k mazes of every slot in a shadow ring that a side stream refills, so that a win costs a 13 KB copy
        instead of the generator's latency (include/maze_b200.h: maze_regen_swap).  Same mazes either way; k x 13 KB per slot.
        visit_layout: "cell" (default; best for one launch per step), "tile" (env-major in 4 x 4 block tiles:
        best for the fused multi-step paths -- step_many, the Q-learning rollout -- and the default with
        enrich, where the 15 x 15 window then reads <= 25 whole sectors per env)."""
        if topology not in ("euclid", "toroidal"):
            raise ValueError("topology must be 'euclid' or 'toroidal'")
        if on_win not in ("keep", "next", "regenerate"):
            raise ValueError("on_win must be 'keep', 'next' or 'regenerate'")
        self.num_envs = int(num_envs)
        self.device = torch.device(device)
        self.topology = topology
        self.shape = (int(shape[0]), int(shape[1]))
        self.seed = int(seed)
        self.autoreset = bool(autoreset)
        self.on_win = on_win
        self.reference_order = bool(reference_order)
        self.slot_id_base = int(slot_id_base)
        self.enrich = bool(enrich)
        self.candidates = int(candidates)
        if self.enrich and self.shape[0] != self.shape[1]:
            raise ValueError("the enriched observation needs square mazes: the reference clamps the window's columns with the "
                             "row count (lib/maze_handler.py:21-29)")
        if self.enrich and min(self.shape) < cabi.WINDOW:
            raise ValueError(f"the enriched observation needs mazes of at least {cabi.WINDOW} x {cabi.WINDOW} blocks")
        if pool is None:
            M = self.num_envs if num_mazes is None else int(num_mazes)
            pool = MazePool(M, self.shape, self.device)
            algos = algorithms
            if not isinstance(algorithms, str):
                algos = [algorithms[i % len(algorithms)] for i in range(M)]
            shapes0 = self.shape if start_shape is None else start_shape
            if not isinstance(shapes0[0], (int, np.integer)):
                shapes0 = [tuple(shapes0[i % len(shapes0)]) for i in range(M)]
            pool.generate(shapes=shapes0, algorithms=algos, toroidal=(topology == "toroidal"),
                          seed=self.seed, slot_id_base=self.slot_id_base, candidates=self.candidates)
        self.pool = pool
        if on_win == "regenerate" and pool.num_mazes != self.num_envs:
            raise ValueError("on_win='regenerate' needs one maze slot per env (num_mazes == num_envs)")
        self.grow = int(grow)
        self.algorithm_schedule = tuple(algorithm_schedule) if algorithm_schedule else ()
        if (self.grow or self.algorithm_schedule) and on_win != "regenerate":
            raise ValueError("grow / algorithm_schedule act when a maze is regenerated: use on_win='regenerate'")
        self.wins = torch.zeros(pool.num_mazes, dtype=torch.int32, device=self.device)
        if regenerate_ahead is None:
            regenerate_ahead = 3
        self.regenerate_depth = min(8, int(regenerate_ahead))   # True -> 1
        self.regenerate_ahead = self.regenerate_depth > 0 and on_win == "regenerate"
        self._ahead = None   # built on the first drain (and again after load_state_dict)
        if env_maze is None:
            # contiguous envs share a maze: table reads of a warp hit the same lines
            per = max(1, self.num_envs // pool.num_mazes)
            env_maze = (torch.arange(self.num_envs, device=self.device, dtype=torch.int32) // per).clamp_(max=pool.num_mazes - 1)
        self.batch = MazeBatch(pool, self.num_envs, env_maze=env_maze, stats=stats, queue=(on_win == "regenerate"),
                               visit_layout=visit_layout or ("tile" if self.enrich else "cell"), visit_bits=self.enrich)
        self._mode = ((cabi.STEP_AUTORESET if self.autoreset else 0)
                      | (cabi.STEP_WIN_NEXT if on_win == "next" else 0)
                      | (cabi.STEP_WIN_QUEUE if on_win == "regenerate" else 0))
        # spaces: gymnasium's when it is installed, the package's own stand-ins (maze_b200/_gym.py) otherwise, so that
        # single_observation_space / observation_space are never None.  They describe the PRODUCED observations
        # (base_maze_env.py:116-122; -v1: simple_maze_env.py:151-158), not the reference's declared ones, which disagree
        # with what its envs return (SURVEY.md section 8(a) E3).
        sp = _gymshim.spaces
        hi = max(self.pool.max_shape)
        if self.enrich:
            single = {"agent": sp.Box(0.0, 1.0, shape=(2,), dtype=np.float64), "target": sp.Box(0.0, 1.0, shape=(2,), dtype=np.float64),
                      "best dir": sp.Box(-hi, hi, shape=(2,), dtype=np.int32),
                      "window": sp.Box(0.0, 1.0, shape=(3, cabi.WINDOW, cabi.WINDOW), dtype=np.float32)}
        else:
            single = {"agent": sp.Box(0, hi, shape=(2,), dtype=np.int32), "target": sp.Box(0, hi, shape=(2,), dtype=np.int32),
                      "best dir": sp.Box(-hi, hi, shape=(2,), dtype=np.int32)}
        self.single_observation_space = sp.Dict(single)
        self.observation_space = sp.Dict({k: sp.Box(v.low if np.isscalar(v.low) else float(np.min(v.low)), v.high if np.isscalar(v.high) else float(np.max(v.high)),
                                                    shape=(self.num_envs,) + tuple(v.shape), dtype=v.dtype) for k, v in single.items()})
        if _gym is not None:  # pragma: no cover
            self.single_action_space = sp.Discrete(4)
            self.action_space = sp.MultiDiscrete([4] * self.num_envs)
        else:
            self.single_action_space = _ActionSpace(4)
            self.action_space = _ActionSpace(4, self.num_envs, seed)
        # pinned staging for the host-buffer path
        self._h_actions = None
        self._d_actions = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
        self._h_out = None
        self._h_flag = None
        self._h_packed = None
        self._h_shape_valid = False
        shapes = self.pool.meta[:, :2]   # one shape and topology for every slot -> the per-env mirrors never go stale
        self._pool_is_uniform = bool((shapes == shapes[0]).all().item()) and not self.grow
        self._h_bytes, self._h_calls = 0, 0

    # ------------------------------------------------------------------------------------------
    def _obs(self):
        b = self.batch
        if self.enrich:
            b.compute_window()
            return {"agent": b.agent_norm, "target": b.target_norm, "best dir": b.best_dir, "window": b.window}
        return {"agent": b.agent, "target": b.target, "best dir": b.best_dir}

    def step_many(self, actions, trace: bool = True):
        """K consecutive steps for an action tape known in advance (uint8 [K, B] device tensor): the same
        transitions as K step() calls, one launch.  Returns the per-step outputs (see MazeBatch.step_many).
        Not available with on_win='regenerate'."""
        if self.on_win == "regenerate":
            raise cabi.MazeError("step_many cannot regenerate mazes between its fused steps")
        return self.batch.step_many(actions, self._mode, trace=trace)

    def get_mask_direction(self, probs: bool = False):
        """float32 [B, 4] direction mask of every env (env.get_mask_direction of the reference)."""
        return self.batch.direction_mask(probs)

    def reset(self, seed: Optional[int] = None, options: Optional[dict] = None):
        """seed is accepted and ignored, like the reference (base_maze_env.py:136)."""
        self.batch.reset()
        return self._obs(), _LazyInfo(self)

    def _device_actions(self, actions):
        if isinstance(actions, torch.Tensor):
            if actions.device == self.device and actions.dtype == torch.uint8 and actions.is_contiguous():
                return actions
            self._d_actions.copy_(actions.reshape(-1), non_blocking=True)
            return self._d_actions
        a = np.ascontiguousarray(actions, dtype=np.uint8).reshape(-1)
        if self._h_actions is None:
            self._h_actions = torch.empty(self.num_envs, dtype=torch.uint8, pin_memory=True)
        self._h_actions.numpy()[:] = a
        self._d_actions.copy_(self._h_actions, non_blocking=True)
        return self._d_actions

    def drain_regeneration(self):
        """Regenerate the maze slots whose env won on the previous step (the analogue of update_maze(),
        off_policy_trainer.py:60-71 / :190-214).  It runs at the START of the next step(), right before the kernel
        that autoresets those envs: everything the caller does with the terminal step in between -- the terminal
        observation and window, DeviceReplay.push, maze_q_update -- still sees the maze the episode was played on, as
        in the reference, where next_obs comes from env.step() before update_maze().  The three launches are
        device-side no-ops when the queue is empty (its length is read on the device)."""
        b = self.batch
        if self.regenerate_ahead:
            return self._drain_ahead()
        if self.grow or self.algorithm_schedule:
            self.pool.curriculum(b.queue, b.queue_count, self.wins, self.grow, self.algorithm_schedule)
        self.pool.generate(ids=b.queue, count_dev=b.queue_count, configure=False, seed=self.seed,
                           slot_id_base=self.slot_id_base, candidates=self.candidates)
        b.queue_count.zero_()

    # -- regeneration ahead of time (include/maze_b200.h: maze_regen_swap / _prepare / _publish) -------------------
    def _curriculum_rule(self):
        sched = list(self.algorithm_schedule or ())
        (wa, aa), (wb, ab) = (sched + [(0, None), (0, None)])[:2]
        code = lambda a: -1 if a is None else (ALGO_IDS[a] if isinstance(a, str) else int(a))  # noqa: E731
        return (int(self.grow), self.pool.max_shape[0], self.pool.max_shape[1], int(wa), code(aa), int(wb), code(ab))

    def _build_ahead(self):
        pool, dev, M, K = self.pool, self.device, self.pool.num_mazes, self.regenerate_depth
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        i32 = dict(dtype=torch.int32, device=dev)
        grids = torch.zeros((K, M, pool.slot), dtype=torch.uint8, device=dev)
        table = torch.zeros((K, M, pool.slot), dtype=torch.uint8, device=dev)
        meta = torch.zeros((K, M, cabi.META_WORDS), **i32)
        ctx = cabi.Context(idx)   # own work counter / scratch: the refills run beside the live pool's generator
        ring = []
        for j in range(K):   # ring entry j holds M(m, g) for the g in [live, live + K) with g % K == j
            sh = MazePool.__new__(MazePool)
            sh.device, sh.ctx, sh.max_shape, sh.num_mazes, sh.slot = dev, ctx, pool.max_shape, M, pool.slot
            sh.grids, sh.table, sh.meta, sh.any_toroidal = grids[j], table[j], meta[j], pool.any_toroidal
            ring.append(sh)
        curriculum = bool(self.grow or self.algorithm_schedule)
        a = SimpleNamespace(ring=ring, grids=grids, table=table, meta=meta, ctx=ctx, ready=torch.zeros((K, M), **i32),
                 # the slot records and win counts now, with nothing in flight: what maze_regen_prepare derives every later
                 # configuration from (reading the live records there would race with maze_regen_swap)
                 base_meta=pool.meta.clone(), base_wins=self.wins.clone() if curriculum else None, curriculum=curriculum,
                 refill=[torch.arange(M, **i32), torch.zeros(M, **i32)], refill_count=[torch.full((1,), M, **i32), torch.zeros(1, **i32)],
                 tag=torch.full((M,), -1, **i32), slow=torch.zeros(M, **i32), slow_count=torch.zeros(1, **i32),
                 work=torch.zeros((K, M), **i32), work_count=torch.zeros(K, **i32), stats=torch.zeros(2, **i32),
                 side=torch.cuda.Stream(device=dev), side_done=torch.cuda.Event(), main_evt=torch.cuda.Event(), cur=0, batch=0, jobs=0)
        self._ahead = a
        self._refill_job(0)   # every slot, on the current stream: the ring starts complete
        for t in (grids, table, meta, a.ready, *a.refill, *a.refill_count, a.work, a.work_count, pool.meta, a.base_meta):
            t.record_stream(a.side)   # the side stream reads / writes them: the allocator must not recycle them under it
        if a.base_wins is not None:
            a.base_wins.record_stream(a.side)

    def _refill_job(self, cur):
        """prepare -> maze_generate per ring entry -> publish for refill queue `cur`, on the current stream."""
        a, pool, K = self._ahead, self.pool, self.regenerate_depth
        lib, p, ctx, M = cabi.lib(), cabi.ptr, a.ctx, pool.num_mazes
        stream = cabi.current_stream(self.device)
        rc = lib.maze_regen_prepare(ctx.handle, p(pool.meta), p(a.base_meta), p(a.base_wins), *self._curriculum_rule(), p(a.meta),
                                    p(a.ready), K, p(a.refill[cur]), p(a.refill_count[cur]), M, p(a.work), p(a.work_count), stream)
        ctx.check(rc, "maze_regen_prepare")
        for j, sh in enumerate(a.ring):
            sh.generate(ids=a.work[j], count_dev=a.work_count[j:j + 1], configure=False, seed=self.seed, slot_id_base=self.slot_id_base,
                        candidates=self.candidates)
        rc = lib.maze_regen_publish(ctx.handle, p(a.meta), p(a.ready), K, p(a.work), p(a.work_count), M, stream)
        ctx.check(rc, "maze_regen_publish")
        a.refill_count[cur].zero_()
        a.work_count.zero_()

    def _fit_ahead_depth(self):
        """The ring costs depth x (2 x slot + 36) bytes per maze slot (3 x 13 KB at 81 x 81): shrink the depth, down to in-place
        regeneration, rather than take more than half of the free device memory."""
        per_entry = self.pool.num_mazes * (2 * self.pool.slot + 4 * cabi.META_WORDS + 4)
        free, _ = torch.cuda.mem_get_info(self.device)
        depth = self.regenerate_depth
        while depth > 0 and depth * per_entry > free // 2:
            depth -= 1
        if depth != self.regenerate_depth:
            import warnings
            warnings.warn(f"regenerate_ahead={self.regenerate_depth} needs {self.regenerate_depth * per_entry / 2**30:.1f} GiB for {self.pool.num_mazes} maze slots; "
                          f"using depth {depth}" + (" (regeneration in place)" if depth == 0 else ""))
            self.regenerate_depth = depth
            self.regenerate_ahead = depth > 0
        return self.regenerate_ahead

    def _drain_ahead(self):
        if self._ahead is None:
            if not self._fit_ahead_depth():
                return self.drain_regeneration()   # no room for a ring: in place, as with regenerate_ahead=0
            self._build_ahead()
        a, b, pool, K = self._ahead, self.batch, self.pool, self.regenerate_depth
        cur, M = a.cur, pool.num_mazes
        lib, p = cabi.lib(), cabi.ptr
        a.slow_count.zero_()
        rc = lib.maze_regen_swap(pool.ctx.handle, p(pool.grids), p(pool.table), p(pool.meta), p(a.grids), p(a.table), p(a.meta), p(a.ready), K,
                                 p(b.queue), p(b.queue_count), M, pool.slot, p(a.refill[cur]), p(a.refill_count[cur]), p(a.tag), a.batch,
                                 p(a.slow), p(a.slow_count), p(a.stats), p(self.wins) if a.curriculum else None,
                                 cabi.current_stream(self.device))
        pool.ctx.check(rc, "maze_regen_swap")
        # slots whose ring entry was not ready (more wins than the ring is deep before a refill was published): drawn in place
        if a.curriculum:
            pool.curriculum(a.slow, a.slow_count, self.wins, self.grow, self.algorithm_schedule)
        pool.generate(ids=a.slow, count_dev=a.slow_count, configure=False, seed=self.seed, slot_id_base=self.slot_id_base,
                      candidates=self.candidates)
        b.queue_count.zero_()
        if a.side_done.query():   # the previous refill has finished: start the next one on what queued up meanwhile
            main, side = torch.cuda.current_stream(self.device), a.side
            a.main_evt.record(main)
            side.wait_event(a.main_evt)
            with torch.cuda.stream(side):
                self._refill_job(cur)
                a.side_done.record(side)
            a.cur, a.batch, a.jobs = cur ^ 1, a.batch + 1, a.jobs + 1

    def regeneration_statistics(self):
        """(slots installed from the shadow pool, slots drawn in place, refill jobs launched) since construction; one small D2H."""
        if self._ahead is None:
            return (0, 0, 0)
        fast, slow = (int(v) for v in self._ahead.stats.tolist())
        return (fast, slow, self._ahead.jobs)

    def _drop_ahead(self):
        if self._ahead is not None:
            self._ahead.side.synchronize()
            self._ahead = None

    def step(self, actions, extra_mode: int = 0, observe: bool = True):
        """observe=False skips building the observation dict (with enrich=True: the 2.7 KB-per-env float window) and
        returns None in its place -- for consumers that read the state another way, like the tensor-core DQN net, which
        takes the replay ring's bit-packed windows."""
        b = self.batch
        if self.on_win == "regenerate":
            self.drain_regeneration()
        b.step(self._device_actions(actions), self._mode | extra_mode)
        term, trunc = b.terminated.view(torch.bool), b.truncated.view(torch.bool)
        if not observe:
            return (None, b.reward, trunc, term, None) if self.reference_order else (None, b.reward, term, trunc, None)
        if self.reference_order:
            return self._obs(), b.reward, trunc, term, _LazyInfo(self)
        return self._obs(), b.reward, term, trunc, _LazyInfo(self)

    # -- host-buffer path: numpy in, numpy out, all copies through pinned memory ---------------
    def _host_out(self):
        if self._h_out is None:
            B = self.num_envs
            pin = dict(pin_memory=True)
            self._h_out = dict(agent=torch.empty((B, 2), dtype=torch.int32, **pin),
                               target=torch.empty((B, 2), dtype=torch.int32, **pin),
                               best_dir=torch.empty((B, 2), dtype=torch.int32, **pin),
                               reward=torch.empty(B, dtype=torch.float64, **pin),
                               terminated=torch.empty(B, dtype=torch.uint8, **pin),
                               truncated=torch.empty(B, dtype=torch.uint8, **pin))
            if self.enrich:
                self._h_out.update(window=torch.empty((B, 3, cabi.WINDOW, cabi.WINDOW), dtype=torch.float32, **pin),
                                   agent_norm=torch.empty((B, 2), dtype=torch.float64, **pin),
                                   target_norm=torch.empty((B, 2), dtype=torch.float64, **pin))
        return self._h_out

    def h2d_bytes_per_step(self):
        return self.num_envs

    def reset_host_counters(self):
        self._h_bytes, self._h_calls = 0, 0

    def d2h_bytes_per_step(self):
        """Average bytes step_host() has copied back per call so far (the target array travels only on the steps
        whose launch rewrote it); before the first call, the worst case."""
        if self._h_calls:
            return self._h_bytes / self._h_calls
        per = 3 * 8 + 8 + 1 + 1
        if self.enrich:
            per += 3 * cabi.WINDOW * cabi.WINDOW * 4 + 2 * 16
        return self.num_envs * per

    def pinned_actions(self) -> torch.Tensor:
        """A fresh uint8 [B] tensor in pinned host memory: actions written into it go to the device without the extra
        host-side staging copy that pageable numpy arrays need (4 MB per step at 4 M envs)."""
        return torch.zeros(self.num_envs, dtype=torch.uint8, pin_memory=True)

    def step_host_packed(self, actions, decode: bool = False, chunks: Optional[int] = None):
        """step_host() over the packed wire format: the actions go host -> device, the kernel writes a single uint32
        record per env instead of the 26 bytes of wide outputs (MAZE_STEP_PACKED | MAZE_STEP_NO_WIDE), the records come
        back to pinned host memory, one synchronisation.  With chunks > 1 (default 4 for batches of 256 k envs and more)
        the batch is cut into env ranges whose copy-in / kernel / copy-out run on alternating streams, so that the PCIe
        transfers of one range overlap the kernel of the next and the two directions overlap each other; the result is
        the same launch by launch (envs are independent).  Returns the pinned uint32 [B] record array (a view: the next
        call overwrites it); `decode=True` returns what step_host() returns, bit for bit, by running
        cabi.decode_records on it (a host-side C loop; `target` and the per-env shapes are refreshed from the device
        only on the steps whose launch changed a maze).  -v0 observations only."""
        if self.enrich:
            raise cabi.MazeError("the packed wire format carries the -v0 observation; use step_host() with enrich=True")
        b = self.batch
        B = self.num_envs
        if chunks is None:
            chunks = 4 if B >= 262144 else 1
        if self._h_packed is None:
            self._h_packed = torch.empty(B, dtype=torch.int32, pin_memory=True)
            self._h_flag = torch.ones(1, dtype=torch.int32, pin_memory=True)
            self._h_target = torch.empty((B, 2), dtype=torch.int32, pin_memory=True)
            self._h_shape = torch.empty((B, 2), dtype=torch.int32, pin_memory=True)
            self._h_tor = torch.empty(B, dtype=torch.uint8, pin_memory=True)
            self._h_actions = torch.empty(B, dtype=torch.uint8, pin_memory=True) if self._h_actions is None else self._h_actions
            self._side_streams = [torch.cuda.Stream(self.device) for _ in range(2)]
        stream = torch.cuda.current_stream(self.device)
        mode = self._mode | cabi.STEP_PACKED | cabi.STEP_NO_WIDE
        if chunks <= 1:
            self.step(actions, extra_mode=cabi.STEP_PACKED | cabi.STEP_NO_WIDE, observe=False)
            self._h_packed.copy_(b.packed, non_blocking=True)
        else:
            if self.on_win == "regenerate":
                self.drain_regeneration()
            if isinstance(actions, torch.Tensor) and actions.device.type == "cpu" and actions.is_pinned() and actions.dtype == torch.uint8:
                src = actions.reshape(-1)      # already in pinned host memory: copied to the device from where it is
            else:
                self._h_actions.numpy()[:] = np.ascontiguousarray(actions, dtype=np.uint8).reshape(-1)
                src = self._h_actions
            start = torch.cuda.Event()
            start.record(stream)
            bounds = [B * k // chunks // 512 * 512 for k in range(chunks)] + [B]    # whole CTAs per range
            for k in range(chunks):
                lo, hi = bounds[k], bounds[k + 1]
                side = self._side_streams[k % 2]
                side.wait_event(start)
                with torch.cuda.stream(side):
                    self._d_actions[lo:hi].copy_(src[lo:hi], non_blocking=True)
                    b.step_view(b.view_struct(lo, hi), self._d_actions.data_ptr() + lo, mode, side.cuda_stream)
                    self._h_packed[lo:hi].copy_(b.packed[lo:hi], non_blocking=True)
            for side in self._side_streams:
                stream.wait_stream(side)
        self._h_flag.copy_(b.target_dirty, non_blocking=True)
        stream.synchronize()
        nbytes = 4 * B + 4
        if int(self._h_flag[0]) != 0:   # a maze changed under some env: refresh the target (and shape / topology) mirrors
            b.target_dirty.zero_()
            self._h_target.copy_(b.target, non_blocking=True)
            nbytes += self.num_envs * 8
            if self._h_shape_valid is False or self.grow:   # shapes only change under the growing curriculum
                meta = self.pool.meta[b.env_maze.long()]
                self._h_shape.copy_(meta[:, :2].contiguous(), non_blocking=True)
                self._h_tor.copy_((meta[:, cabi.META_FLAGS] & cabi.FLAG_TOROIDAL).to(torch.uint8), non_blocking=True)
                nbytes += self.num_envs * (8 + 1)
                self._h_shape_valid = self._pool_is_uniform
            stream.synchronize()
        self._h_bytes += nbytes
        self._h_calls += 1
        rec = self._h_packed.numpy().view(np.uint32)
        if not decode:
            return rec
        d = cabi.decode_records(rec, self._h_shape.numpy(), self._h_tor.numpy())
        obs = {"agent": d["agent"], "target": self._h_target.numpy(), "best dir": d["best_dir"]}
        if self.reference_order:
            return obs, d["reward"], d["truncated"], d["terminated"], {}
        return obs, d["reward"], d["terminated"], d["truncated"], {}

    def step_host(self, actions: np.ndarray):
        """Same transition as step() with HOST buffers on both sides: actions are copied to the
        device, every output is copied back; returns numpy views of the pinned result buffers."""
        b = self.batch
        self.step(actions)
        h = self._host_out()
        if self._h_flag is None:
            self._h_flag = torch.ones(1, dtype=torch.int32, pin_memory=True)
        # `target` changes only when an env's maze does (reset, restart after a win): the kernels raise
        # batch.target_dirty when they write it, and only then is it copied again
        self._h_flag.copy_(b.target_dirty, non_blocking=True)
        nbytes = 4
        for k in h:
            if k != "target":
                h[k].copy_(getattr(b, k), non_blocking=True)
                nbytes += h[k].numel() * h[k].element_size()
        stream = torch.cuda.current_stream(self.device)
        stream.synchronize()
        if int(self._h_flag[0]) != 0:
            b.target_dirty.zero_()
            h["target"].copy_(b.target, non_blocking=True)
            nbytes += h["target"].numel() * h["target"].element_size()
            stream.synchronize()
        self._h_bytes += nbytes
        self._h_calls += 1
        obs = {"agent": h["agent"].numpy(), "target": h["target"].numpy(), "best dir": h["best_dir"].numpy()}
        if self.enrich:
            obs.update(agent=h["agent_norm"].numpy(), target=h["target_norm"].numpy(), window=h["window"].numpy())
        term, trunc = h["terminated"].numpy().view(np.bool_), h["truncated"].numpy().view(np.bool_)
        info = {}
        if self.reference_order:
            return obs, h["reward"].numpy(), trunc, term, info
        return obs, h["reward"].numpy(), term, trunc, info

    def state_dict(self):
        """Checkpoint of the whole env (pool, batch, curriculum win counts): load it into an env built with the
        same arguments and the following steps are bit-identical.  Values are references to the live tensors --
        `torch.save(env.state_dict(), path)` serialises them, `{k: v.clone()}` snapshots them in memory."""
        return {"pool": self.pool.state_dict(), "batch": self.batch.state_dict(), "wins": self.wins}

    def load_state_dict(self, sd):
        self._drop_ahead()   # the shadow pool is rebuilt from the loaded generation counts on the next drain
        self.pool.load_state_dict(sd["pool"])
        self.batch.load_state_dict(sd["batch"])
        self.wins.copy_(sd["wins"])

    def episode_statistics(self, reduce: bool = False):
        """Episodes / wins / truncations / return sum since construction (one small D2H); with
        reduce=True summed over all ranks of the torch.distributed job (the only collective of
        the env path: five float64 scalars at the end of a rollout)."""
        from . import dist as mdist
        b = self.batch
        if b.stats is None:
            return None
        vec = torch.cat([b.stats.to(torch.float64), b.stats_return])
        if reduce:
            vec = mdist.reduce_statistics(vec)
        return mdist.statistics_dict(vec)

    def close(self):
        pass
