"""Bit-exact model of the device generators' random stream (test infrastructure; see oracle/__init__.py).

`maze_generate` (csrc/maze_gen.cu) keys one PCG32 stream per (seed, global slot id, generation count,
candidate) from a Philox4x32-10 block and draws the start cell and every choice of the generator from
it.  This module replays that stream in plain Python, with lattice rows held as integers exactly as
the warp holds them, so that `stream_maze` returns the maze the device draws under a given key:

- Philox4x32-10 (maze_common.cuh, `Philox::refill`): key (seed lo, seed hi), counter
  (0, sub, seq lo, seq hi).
- `GenRng` (maze_gen.cu): PCG-XSH-RR 64/32, state = o1:o0, increment = (o3:o2) << 1 | 1, one output
  discarded at init, below(n) = (next() * n) >> 32.  Every pick draws, even among one choice.
- `pick_uniform` ranks the cells of a set LANE-major: lane l holds rows l and l + 32, so the order is
  row 0, row 32, row 1, row 33, ... (ascending column within a row).
- `pick_direction` takes the k-th set bit of the neighbour mask (0 up, 1 down, 2 left, 3 right).
"""
from __future__ import annotations

import numpy as np

from .generation import select_goal, strip_border

M32 = 0xFFFFFFFF
M64 = 0xFFFFFFFFFFFFFFFF
ALGO_IDS = {"r-prim": 0, "dfs": 1, "prim&kill": 2}


def philox4x32_10(key, ctr):
    """One Philox4x32-10 block: key (k0, k1), counter (c0, c1, c2, c3) -> four 32-bit words."""
    a, b = key[0] & M32, key[1] & M32
    x0, x1, x2, x3 = (c & M32 for c in ctr)
    for _ in range(10):
        p0 = 0xD2511F53 * x0
        p1 = 0xCD9E8D57 * x2
        x0, x1, x2, x3 = ((p1 >> 32) ^ x1 ^ a) & M32, p1 & M32, ((p0 >> 32) ^ x3 ^ b) & M32, p0 & M32
        a = (a + 0x9E3779B9) & M32
        b = (b + 0xBB67AE85) & M32
    return x0, x1, x2, x3


class GenRng:
    """maze_gen.cu `GenRng`: PCG-XSH-RR 64/32 seeded by Philox::init(seed, seq, sub) + refill()."""

    def __init__(self, seed: int, seq: int, sub: int):
        o0, o1, o2, o3 = philox4x32_10((seed & M32, (seed >> 32) & M32), (0, sub & M32, seq & M32, (seq >> 32) & M32))
        self.state = (o1 << 32) | o0
        self.inc = ((((o3 << 32) | o2) << 1) | 1) & M64
        self.next()

    def next(self) -> int:
        old = self.state
        self.state = (old * 6364136223846793005 + self.inc) & M64
        xs = (((old >> 18) ^ old) >> 27) & M32
        rot = old >> 59
        return ((xs >> rot) | (xs << (32 - rot))) & M32

    def below(self, n: int) -> int:
        return (self.next() * n) >> 32


def _kth_bit(w: int, k: int) -> int:
    for _ in range(k):
        w &= w - 1
    return (w & -w).bit_length() - 1


def lane_major_rows(nr: int):
    """Row order in which pick_uniform ranks set bits: lane 0 (rows 0, 32), lane 1 (rows 1, 33), ..."""
    return [r for lane in range(32) for r in (lane, lane + 32) if r < nr]


def pick_uniform(rows, order, rng):
    """Uniformly random set bit of the row sets `rows` (ranked in `order`) -> (i, j), or None if empty."""
    total = sum(rows[r].bit_count() for r in order)
    if total == 0:
        return None
    k = rng.below(total)
    for r in order:
        c = rows[r].bit_count()
        if k < c:
            return r, _kth_bit(rows[r], k)
        k -= c
    raise AssertionError("unreachable")


def neighbour_mask(rows, i, j, nr, nc, want):
    """Bit 0 up, 1 down, 2 left, 3 right: lattice neighbours of (i, j) whose bit equals `want`."""
    w = 1 if want else 0
    nb = 0
    if i > 0 and (rows[i - 1] >> j) & 1 == w:
        nb |= 1
    if i + 1 < nr and (rows[i + 1] >> j) & 1 == w:
        nb |= 2
    if j > 0 and (rows[i] >> (j - 1)) & 1 == w:
        nb |= 4
    if j + 1 < nc and (rows[i] >> (j + 1)) & 1 == w:
        nb |= 8
    return nb


def pick_direction(nb, rng):
    return _kth_bit(nb, rng.below(nb.bit_count()))


_DELTA = ((-1, 0), (1, 0), (0, -1), (0, 1))   # up, down, left, right


def _open_wall(E, S, i, j, d):
    if d == 0:
        S[i - 1] |= 1 << j
    elif d == 1:
        S[i] |= 1 << j
    elif d == 2:
        E[i] |= 1 << (j - 1)
    else:
        E[i] |= 1 << j


def _random_prim(E, S, nr, nc, si, sj, rng, order):
    colmask = (1 << nc) - 1
    inn = [0] * nr
    fr = [0] * nr

    def add_cell(i, j):
        bit = 1 << j
        inn[i] |= bit
        fr[i] &= ~bit
        fr[i] |= ((bit << 1) | (bit >> 1)) & ~inn[i] & colmask
        for r in (i - 1, i + 1):
            if 0 <= r < nr:
                fr[r] |= bit & ~inn[r]

    add_cell(si, sj)
    while True:
        p = pick_uniform(fr, order, rng)
        if p is None:
            return
        i, j = p
        _open_wall(E, S, i, j, pick_direction(neighbour_mask(inn, i, j, nr, nc, True), rng))
        add_cell(i, j)


def _depth_first(E, S, nr, nc, si, sj, rng, order):
    vis = [0] * nr
    back = {}
    vis[si] |= 1 << sj
    i, j = si, sj
    while True:
        nb = neighbour_mask(vis, i, j, nr, nc, False)
        if nb:
            d = pick_direction(nb, rng)
            i, j = i + _DELTA[d][0], j + _DELTA[d][1]
            _open_wall(E, S, i, j, d ^ 1)
            vis[i] |= 1 << j
            back[i, j] = d ^ 1
        else:
            if (i, j) == (si, sj):
                return
            d = back[i, j]
            i, j = i + _DELTA[d][0], j + _DELTA[d][1]


def _prim_and_kill(E, S, nr, nc, si, sj, rng, order):
    mk = [0] * nr
    mk[si] |= 1 << sj
    unmarked = nr * nc - 1
    i, j = si, sj
    while True:
        while True:
            nb = neighbour_mask(mk, i, j, nr, nc, False)
            if not nb:
                break
            d = pick_direction(nb, rng)
            i, j = i + _DELTA[d][0], j + _DELTA[d][1]
            _open_wall(E, S, i, j, d ^ 1)
            mk[i] |= 1 << j
            unmarked -= 1
        if unmarked == 0:
            return
        # marked cells with at least one unmarked lattice neighbour
        elig = [0] * nr
        for r in range(nr):
            for c in range(nc):
                if (mk[r] >> c) & 1 and neighbour_mask(mk, r, c, nr, nc, False):
                    elig[r] |= 1 << c
        i, j = pick_uniform(elig, order, rng)


_GENERATORS = {"r-prim": _random_prim, "dfs": _depth_first, "prim&kill": _prim_and_kill}


def stream_key(slot: int, gen_count: int = 0) -> int:
    """Philox sequence id of a slot: global slot id | generation count << 40."""
    return (int(slot) | (int(gen_count) << 40)) & M64


def draw_walls(algo, nr, nc, seed, seq, sub=0):
    """The device's generate_walls: start cell and wall planes (E[i] bit j = passage (i, j)-(i, j+1),
    S[i] bit j = passage (i, j)-(i+1, j)) of one nr x nc lattice -> (si, sj, E, S)."""
    rng = GenRng(int(seed) & M64, seq, sub)
    si = rng.below(nr)
    sj = rng.below(nc)
    E, S = [0] * nr, [0] * nr
    _GENERATORS[algo](E, S, nr, nc, si, sj, rng, lane_major_rows(nr))
    return si, sj, E, S


def walls_to_grid(nr, nc, E, S):
    """Bordered block grid (2 nr + 1) x (2 nc + 1) of the wall planes: cells and open passages 1."""
    g = np.zeros((2 * nr + 1, 2 * nc + 1), dtype=np.uint8)
    g[1::2, 1::2] = 1
    for i in range(nr):
        for j in range(nc):
            if (E[i] >> j) & 1:
                g[2 * i + 1, 2 * j + 2] = 1
            if (S[i] >> j) & 1:
                g[2 * i + 2, 2 * j + 1] = 1
    return g


def stream_maze(algo, shape, toroidal, seed, slot, gen_count=0, candidate=0):
    """The maze `maze_generate` draws for global slot id `slot` -> (start, goal, grid) as
    oracle.generation.gen_maze / gen_maze_no_border return them (block coordinates, goal block = 2).
    Toroidal mazes are drawn at shape + 2 and stripped of their border."""
    H, W = (shape, shape) if isinstance(shape, (int, np.integer)) else (int(shape[0]), int(shape[1]))
    Hb, Wb = (H + 2, W + 2) if toroidal else (H, W)
    nr, nc = (Hb - 1) // 2, (Wb - 1) // 2
    si, sj, E, S = draw_walls(algo, nr, nc, seed, stream_key(slot, gen_count), candidate)
    grid = walls_to_grid(nr, nc, E, S)
    start = (2 * si + 1, 2 * sj + 1)
    goal = select_goal(grid, start)
    grid[goal] = 2
    return strip_border(start, goal, grid) if toroidal else (start, goal, grid)
