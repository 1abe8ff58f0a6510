"""The reference's eight single-maze environment classes as batch-of-1 views of the device engine.

Same constructors, methods, attributes and return conventions as
gymnasium_env/envs/{simple,simple_variable,toroidal,toroidal_variable}_maze_env.py and
base_maze_env.py of the reference, so lib/trainers/* and agents/* of the reference run against
them unmodified (they reach the env through `RecordEpisodeStatistics(env).env`):

  step(a) -> (obs, reward, truncated, terminated, info)      # the reference's swapped order, :210
  reset() -> (obs, {"distance": L1(agent, target)})          # :136-161, seed ignored like the reference
  obs -v0 = {"agent": int32[2], "target": int32[2], "best dir": int64[2]}                :116-122
  obs -v1 = {"agent": f64[2] / shape, "target": f64[2] / shape, "best dir", "window": f32[3,15,15]}

Everything is computed by the CUDA kernels (maze_generate with candidates=6, maze_step,
maze_window, maze_direction_mask, maze_difficulty); this file only moves a few bytes per call.
Rendering (lib/maze_view.py) is out of scope: render() is a no-op.
"""
from __future__ import annotations

import random

import numpy as np
import torch

from . import cabi
from ._gym import Env, spaces
from .engine import ALGO_IDS, MazeBatch, MazePool, check_shape

WINDOW_DIM = cabi.WINDOW


class BaseMazeEnv(Env):
    """base_maze_env.py:10-309.  ALGORITHM is a class-level global shared by every env, as in the
    reference (:17,60-64)."""

    metadata = {"render.modes": ["human", "rgb_array"], "render_fps": 4}
    ALGORITHM = "r-prim"
    ACTIONS = {0: np.array([1, 0]), 1: np.array([-1, 0]), 2: np.array([0, 1]), 3: np.array([0, -1])}
    TOROIDAL = False
    ENRICH = False
    VARIABLE = False
    CANDIDATES = 6          # generate_maze keeps the least difficult of 1 + 5 mazes (:78-97)
    _seed_counter = [0]

    def __init__(self, maze_shape, render_mode: str = "human", max_shape=None, device="cuda", seed=None):
        self.render_mode = render_mode
        self.device = torch.device(device)
        self.max_shape = tuple(max_shape) if max_shape is not None else None
        pool_shape = self.max_shape if self.max_shape is not None else tuple(maze_shape)
        check_shape(pool_shape, cabi.GEN_MAX_DIM - 2)
        if seed is None:
            seed = random.getrandbits(62)   # the reference draws from the global `random`, so seeding it seeds us
        self._seed = int(seed)
        self._pool = MazePool(1, pool_shape, self.device)
        self._batch = MazeBatch(self._pool, 1, visit_layout="tile" if self.ENRICH else "cell")
        self._act = torch.zeros(1, dtype=torch.uint8, device=self.device)
        self._difficulty = torch.zeros(1, dtype=torch.float64, device=self.device)
        self.action_space = spaces.Discrete(4)
        self.maze_view = None
        self.cum_rew = 0
        self.mazes = []
        self.next = 0
        self.maze_shape = tuple(maze_shape)
        self._start_pos, goal_pos, self.maze_map = self.generate_maze(self.maze_shape)
        self._target_location = np.array(goal_pos, dtype=np.int32)
        self._agent_location = np.array(self._start_pos, dtype=np.int32)
        self.observation_space = self._make_observation_space()
        self.set_max_steps()
        self.mazes.append(self._maze_record())
        self.reset()

    # ---- reference API: algorithm / shape getters ----------------------------------------------
    def set_algorithm(self, algorithm: str):
        BaseMazeEnv.ALGORITHM = algorithm

    def get_algorithm(self):
        return BaseMazeEnv.ALGORITHM

    def get_maze_shape(self):
        return self.maze_shape

    def get_max_shape(self):
        return self.max_shape

    def _make_observation_space(self):
        hi = np.array(self.max_shape if self.VARIABLE else self.maze_shape)
        if self.ENRICH:
            return spaces.Dict({"agent": spaces.Box(0, 1, shape=(2,), dtype=int), "target": spaces.Box(0, 1, shape=(2,), dtype=int),
                                "best dir": spaces.Box(-1, 1, shape=(2,), dtype=int),
                                "window": spaces.Box(-1, 1, shape=(3, WINDOW_DIM, WINDOW_DIM), dtype=float)})
        return spaces.Dict({"agent": spaces.Box(low=np.array([0, 0]), high=hi, dtype=int),
                            "target": spaces.Box(low=np.array([0, 0]), high=hi, dtype=int),
                            "best dir": spaces.Box(-1, 1, shape=(2,), dtype=int)})

    # ---- maze lifecycle -------------------------------------------------------------------------
    def generate_maze(self, maze_shape):
        """base_maze_env.py:78-97 / toroidal_maze_env.py:40-54 on the device: six candidates, the least
        difficult one is kept.  Returns (start_pos, goal_pos, maze_map as a list of lists)."""
        algo = BaseMazeEnv.ALGORITHM
        if algo not in ALGO_IDS:
            raise ValueError(f"unknown maze generation algorithm {algo!r}")
        BaseMazeEnv._seed_counter[0] += 1
        self._pool.generate(ids=[0], shapes=tuple(maze_shape), algorithms=algo, toroidal=self.TOROIDAL,
                            seed=self._seed, slot_id_base=BaseMazeEnv._seed_counter[0], candidates=self.CANDIDATES,
                            difficulty_out=self._difficulty)
        meta = self._pool.meta_host()[0]
        start = (int(meta[cabi.META_START]) & 0xffff, int(meta[cabi.META_START]) >> 16)
        goal = (int(meta[cabi.META_GOAL]) & 0xffff, int(meta[cabi.META_GOAL]) >> 16)
        self._max_steps_device = int(meta[cabi.META_MAX_STEPS])
        return start, goal, self._pool.grid_host(0).astype(np.int64).tolist()

    def _maze_record(self):
        if self.VARIABLE:
            return [self._start_pos, self.maze_shape, self.maze_map]
        return [self._start_pos, self.maze_map]

    def _install(self, start, goal, maze_map, shape):
        """Upload a host maze (update_visited_maze) and recompute its fields on the device."""
        self._pool.upload([0], [np.asarray(maze_map, dtype=np.uint8)], [start], [goal], [self.TOROIDAL])
        self._max_steps_device = int(self._pool.meta_host()[0, cabi.META_MAX_STEPS])

    def set_max_steps(self):
        """simple_maze_env.py:52-58: ceil(((H-1)(W-1)-1) * len(path) / CE), computed by maze_fields."""
        self.max_steps_taken = self._max_steps_device

    def get_maze_difficulty(self):
        """McClendon difficulty of the current maze (base_maze_env.py:99-105)."""
        return float(self._pool.difficulty([0])[0, 0].item())

    def _after_new_maze(self, goal_pos):
        self._target_location = np.array(goal_pos, dtype=np.int32)
        self.set_max_steps()

    def update_maze(self):
        if self.VARIABLE:   # simple_variable_maze_env.py:93-112: grow by (4, 4) until max_shape, then shuffle
            shape = tuple(a + b for a, b in zip(self.maze_shape, (4, 4)))
            if not shape <= self.max_shape:
                random.shuffle(self.mazes)
                return
            self.maze_shape = shape
        self._start_pos, goal_pos, self.maze_map = self.generate_maze(self.maze_shape)
        self._after_new_maze(goal_pos)
        self.mazes.append(self._maze_record())
        self.reset()

    def update_visited_maze(self, remove: bool = True):
        rec = self.mazes[self.next]
        if self.VARIABLE:
            self._start_pos, self.maze_shape, self.maze_map = rec
        else:
            self._start_pos, self.maze_map = rec
        grid = np.asarray(self.maze_map)
        r, c = np.argwhere(grid == 2)[0]
        if remove:
            self.mazes.remove(rec)
        else:
            self.next += 1
        self._install(self._start_pos, (int(r), int(c)), self.maze_map, self.maze_shape)
        self._after_new_maze((int(r), int(c)))
        self.reset()

    def update_new_maze(self, shape=None):
        if shape is not None:
            self.maze_shape = tuple(shape)
        elif self.VARIABLE:   # simple_variable_maze_env.py:135-139
            self.maze_shape = random.sample([(a, a) for a in range(self.START_SHAPE[0], self.max_shape[0], 2)], 1)[0]
        self._start_pos, goal_pos, self.maze_map = self.generate_maze(self.maze_shape)
        self._after_new_maze(goal_pos)
        self.reset()

    # ---- observation / step ---------------------------------------------------------------------
    def _get_info(self):
        return {"distance": float(np.abs(self._agent_location.astype(np.int64) - self._target_location).sum())}

    def _get_obs(self):
        b = self._batch
        agent = b.agent.cpu().numpy()[0]
        self._agent_location = agent.astype(np.int32)
        best = b.best_dir.cpu().numpy()[0].astype(np.int64)
        if not self.ENRICH:
            return {"agent": self._agent_location, "target": self._target_location, "best dir": best}
        window = b.compute_window()[0].cpu()
        return {"agent": b.agent_norm.cpu().numpy()[0], "target": b.target_norm.cpu().numpy()[0], "best dir": best,
                "window": window}

    def reset(self, seed=None, options=None):
        self._batch.reset()
        self.steps_taken = 0
        self.cum_rew = 0
        obs = self._get_obs()
        return obs, self._get_info()

    def step(self, action):
        self._act.fill_(int(action) & 3)
        self._batch.step(self._act, mode=0)
        out = torch.stack([self._batch.reward, self._batch.terminated.to(torch.float64),
                           self._batch.truncated.to(torch.float64)]).cpu().numpy()[:, 0]
        reward, terminated, truncated = float(out[0]), bool(out[1]), bool(out[2])
        obs = self._get_obs()
        self.steps_taken += 1
        self.cum_rew += reward
        return obs, reward, truncated, terminated, self._get_info()

    def get_mask_direction(self, probs: bool = False):
        m = self._batch.direction_mask(probs).cpu().numpy()[0]
        if probs and (m == 0.25).any():
            return m.astype(np.float32)
        return m.astype(np.int32)

    def render(self, mode="human", close=False):
        """rgb frame uint8 [16 H, 16 W, 3] of the current maze (base_maze_env.py:212-222 returns
        maze_view.update(mode), the surface as an array); there is no window to update here."""
        if close:
            return None
        H, W = self.maze_shape
        return self._batch.render([0])[0, :H * 16, :W * 16].cpu().numpy()

    def close(self):
        pass


class SimpleMazeEnv(BaseMazeEnv):
    """gymnasium_env/envs/simple_maze_env.py:14-127"""

    def __init__(self, maze_shape, render_mode: str = "human", **kw):
        super().__init__(maze_shape, render_mode, **kw)


class SimpleEnrichMazeEnv(SimpleMazeEnv):
    """simple_maze_env.py:129-158"""
    ENRICH = True
    WINDOW_DIM = WINDOW_DIM


class ToroidalMazeEnv(BaseMazeEnv):
    """gymnasium_env/envs/toroidal_maze_env.py:15-156"""
    TOROIDAL = True

    def __init__(self, maze_shape, render_mode: str = "human", **kw):
        super().__init__(maze_shape, render_mode, **kw)


class ToroidalEnrichMazeEnv(ToroidalMazeEnv):
    """toroidal_maze_env.py:158-172"""
    ENRICH = True


class SimpleVariableMazeEnv(BaseMazeEnv):
    """gymnasium_env/envs/simple_variable_maze_env.py:16-147"""
    VARIABLE = True
    START_SHAPE = (15, 15)

    def __init__(self, max_shape, render_mode: str = "human", **kw):
        super().__init__(self.START_SHAPE, render_mode, max_shape=tuple(max_shape), **kw)


class SimpleEnrichVariableMazeEnv(SimpleVariableMazeEnv):
    """simple_variable_maze_env.py:150-179"""
    ENRICH = True
    WINDOW_DIM = WINDOW_DIM


class ToroidalVariableMazeEnv(BaseMazeEnv):
    """gymnasium_env/envs/toroidal_variable_maze_env.py:16-175"""
    TOROIDAL = True
    VARIABLE = True
    START_SHAPE = (29, 29)

    def __init__(self, max_shape, render_mode: str = "human", **kw):
        super().__init__(self.START_SHAPE, render_mode, max_shape=tuple(max_shape), **kw)


class ToroidalEnrichVariableMazeEnv(ToroidalVariableMazeEnv):
    """toroidal_variable_maze_env.py:177-194"""
    ENRICH = True


ENV_CLASSES = {c.__name__: c for c in (SimpleMazeEnv, SimpleEnrichMazeEnv, SimpleVariableMazeEnv, SimpleEnrichVariableMazeEnv,
                                       ToroidalMazeEnv, ToroidalEnrichMazeEnv, ToroidalVariableMazeEnv, ToroidalEnrichVariableMazeEnv)}
