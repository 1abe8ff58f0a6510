"""The generator models the device tests rest on, checked without a GPU:

- oracle.gen_stream's Philox4x32-10 against the Random123 known-answer vectors;
- oracle.gen_exact's enumeration of the generators' exact output distributions (total mass, support
  sizes, every outcome a perfect maze) against samples of the oracle generators (oracle.generation);
- the device stream model (oracle.gen_stream) against the enumeration;
- best_of_k against brute force over all draw sequences, with ties going to the first draw."""
import itertools
import random

import numpy as np
import pytest

from oracle.gen_exact import (best_candidate, best_of_k, chi_square, exact_outcomes, grid_outcome_id, n_edges,
                              outcome_grid, walls_outcome_id)
from oracle.gen_stream import draw_walls, lane_major_rows, philox4x32_10, stream_key, stream_maze
from oracle.generation import ALGORITHMS, check_perfect_maze, gen_maze, select_goal

P_MIN = 1e-6   # chi-square p-value floor; every sample below is drawn from a fixed seed


@pytest.mark.parametrize("key,ctr,want", [
    ((0, 0), (0, 0, 0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF, 0xFFFFFFFF), (0xFFFFFFFF,) * 4, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0xA4093822, 0x299F31D0), (0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(key, ctr, want):
    assert philox4x32_10(key, ctr) == want


def test_pick_order_is_lane_major():
    assert lane_major_rows(3) == [0, 1, 2]
    assert lane_major_rows(34)[:6] == [0, 32, 1, 33, 2, 3]
    assert lane_major_rows(64) == [r for lane in range(32) for r in (lane, lane + 32)]


# outcome counts over all start cells: r-prim reaches every spanning tree from every start
SUPPORT = {(2, 2): {"r-prim": 16, "dfs": 8, "prim&kill": 8},
           (3, 3): {"r-prim": 1728, "dfs": 108, "prim&kill": 424},
           (3, 4): {"r-prim": 28980, "dfs": 494, "prim&kill": 3934},
           (4, 3): {"r-prim": 28980, "dfs": 494, "prim&kill": 3934}}


@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("lattice", list(SUPPORT))
def test_enumeration_is_a_distribution_over_perfect_mazes(algo, lattice):
    nr, nc = lattice
    probs = exact_outcomes(algo, nr, nc)
    assert len(probs) == SUPPORT[lattice][algo]
    assert sum(probs.values()) == pytest.approx(1.0, abs=1e-12)
    assert min(probs.values()) > 0
    starts = set()
    for oid in probs:
        start, grid = outcome_grid(oid, nr, nc)
        ok, why = check_perfect_maze(grid)
        assert ok, (algo, lattice, oid, why)
        assert grid_outcome_id(grid, start) == oid
        starts.add(start)
    assert len(starts) == nr * nc
    # every start cell carries 1 / (nr nc)
    per_start = {}
    for oid, p in probs.items():
        s = oid >> n_edges(nr, nc)
        per_start[s] = per_start.get(s, 0.0) + p
    assert all(v == pytest.approx(1.0 / (nr * nc), abs=1e-12) for v in per_start.values())


def test_every_outcome_is_an_r_prim_outcome():
    """r-prim reaches every (start, spanning tree) pair; dfs and prim&kill reach a subset of them."""
    rp = exact_outcomes("r-prim", 3, 3)
    for algo in ("dfs", "prim&kill"):
        assert set(exact_outcomes(algo, 3, 3)) <= set(rp)


@pytest.mark.parametrize("algo", ALGORITHMS)
def test_enumeration_matches_oracle_generators(algo):
    """Chi-square of 20 000 oracle.generation samples at 7 x 7 against the exact distribution: the
    enumeration restates the same processes as the oracle does."""
    probs = exact_outcomes(algo, 3, 3)
    rng = random.Random(1234)
    counts = {}
    for _ in range(20000):
        start, goal, grid = gen_maze((7, 7), algo, rng)
        oid = grid_outcome_id(grid, start)
        counts[oid] = counts.get(oid, 0) + 1
    p, outside = chi_square(counts, probs)
    assert outside == 0
    assert p >= P_MIN, (algo, p)


@pytest.mark.parametrize("algo", ALGORITHMS)
def test_stream_model_matches_enumeration(algo):
    """Chi-square of 20 000 mazes of the device stream model (slot ids 0 .. 19 999 of seed 17) at 3 x 3."""
    probs = exact_outcomes(algo, 3, 3)
    counts = {}
    for slot in range(20000):
        oid = walls_outcome_id(3, 3, *draw_walls(algo, 3, 3, 17, stream_key(slot)))
        counts[oid] = counts.get(oid, 0) + 1
    p, outside = chi_square(counts, probs)
    assert outside == 0
    assert p >= P_MIN, (algo, p)


def test_chi_square_rejects_a_biased_sampler():
    """The test statistic has teeth: r-prim joined through the FIRST in-tree neighbour (a plausible kernel bug
    that still yields perfect mazes) is rejected at 20 000 samples."""
    probs = exact_outcomes("r-prim", 3, 3)
    rng = random.Random(5)
    counts = {}
    from oracle import generation as G

    def first_neighbour_prim(grid, start, rng):
        H, W = grid.shape
        grid[start] = 1
        frontier = list(G._cell_neighbours(*start, H, W))
        while frontier:
            f = frontier.pop(rng.randrange(len(frontier)))
            if grid[f]:
                continue
            n = [q for q in G._cell_neighbours(*f, H, W) if grid[q] == 1][0]
            grid[f] = 1
            grid[(f[0] + n[0]) // 2, (f[1] + n[1]) // 2] = 1
            frontier += [q for q in G._cell_neighbours(*f, H, W) if grid[q] == 0 and q not in frontier]

    for _ in range(20000):
        grid = np.zeros((7, 7), dtype=np.uint8)
        start = (rng.randrange(1, 6, 2), rng.randrange(1, 6, 2))
        first_neighbour_prim(grid, start, rng)
        oid = grid_outcome_id(grid, start)
        counts[oid] = counts.get(oid, 0) + 1
    p, _ = chi_square(counts, probs)
    assert p < 1e-12


@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("shape,toroidal", [(5, False), ((9, 129), False), ((129, 9), False), ((65, 7), False), (129, False),
                                            (63, True), (127, True)])
def test_stream_mazes_are_perfect(algo, shape, toroidal):
    """Structure of the model's mazes on the shapes the device tests compare bit for bit (rows past 31 in use)."""
    for slot in (0, 77):
        start, goal, grid = stream_maze(algo, shape, toroidal, 3, slot)
        H, W = (shape, shape) if isinstance(shape, int) else shape
        assert grid.shape == (H, W)
        if toroidal:
            grid, start, goal = np.pad(grid, 1), (start[0] + 1, start[1] + 1), (goal[0] + 1, goal[1] + 1)
        ok, why = check_perfect_maze(grid)
        assert ok, why
        g1 = grid.copy()
        g1[goal] = 1
        assert grid[goal] == 2 and select_goal(g1, start) == goal


def test_stream_keys_select_independent_mazes():
    base = stream_maze("r-prim", 21, False, 5, 3)[2]
    assert np.array_equal(stream_maze("r-prim", 21, False, 5, 3)[2], base)
    for kw in (dict(slot=4), dict(slot=3, gen_count=1), dict(slot=3, candidate=1)):
        args = dict(slot=3, gen_count=0, candidate=0)
        args.update(kw)
        assert not np.array_equal(stream_maze("r-prim", 21, False, 5, **args)[2], base)
    assert not np.array_equal(stream_maze("r-prim", 21, False, 6, 3)[2], base)


def test_best_of_k_against_brute_force():
    """All 5^3 draw sequences of a five-outcome distribution with a tie class of two (scores differing
    in the last bits) and an exact tie: kept = best_candidate, i.e. the first draw of the lowest class."""
    probs = {10: 0.1, 11: 0.25, 12: 0.3, 13: 0.15, 14: 0.2}
    scores = {10: 2.0, 11: 1.0, 12: 1.0 * (1 + 3e-16), 13: 3.0, 14: 2.0}
    want = {o: 0.0 for o in probs}
    ids = list(probs)
    for seq in itertools.product(ids, repeat=3):
        p = np.prod([probs[o] for o in seq])
        want[seq[best_candidate([scores[o] for o in seq])]] += p
    got = best_of_k(probs, scores, 3)
    assert sum(got.values()) == pytest.approx(1.0, abs=1e-15)
    for o in ids:
        assert got[o] == pytest.approx(want[o], abs=1e-15), o
    assert best_of_k(probs, scores, 1) == pytest.approx(probs)


def test_best_candidate_rule():
    assert best_candidate([3.0, 2.0, 2.0 * (1 - 1e-13), 2.5]) == 1       # within 1e-12: the earlier one stays
    assert best_candidate([3.0, 2.0, 2.0 * (1 - 1e-10), 2.5]) == 2       # genuinely lower
    assert best_candidate([0.0, 0.0, -1.0]) == 2
    assert best_candidate([5.0]) == 0
