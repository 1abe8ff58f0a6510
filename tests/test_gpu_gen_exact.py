"""Device generators (maze_generate) against their exact output distributions and against a bit-exact
model of the device random stream.

(a) Exact distribution.  On lattices of up to 12 cells the probability of every (start, spanning tree)
    outcome is known (oracle.gen_exact, checked against the oracle generators in
    test_gen_exact_cpu.py).  Millions of device mazes are encoded as outcome ids on the device and
    counted; no mass may fall outside the support, every outcome carries select_goal's goal, and a
    chi-square (bins expected below 5 pooled) must give p >= 1e-6.  The seeds are fixed, so the
    verdict is deterministic.  Power: 2^22 draws on 3 x 3 lattices and 2^24 on 3 x 4 / 4 x 3 put
    several hundred expected draws in the typical bin; a rule that moves a few percent of the mass
    between outcomes (first instead of a random tree neighbour, a restart set missing one direction,
    one dfs direction never taken) fails by hundreds of standard deviations, while none of these
    changes the five means test_generator_distribution_matches_reference looks at by enough to fail it.
    Best-of-6 is covered the same way at 7 x 7 and 7 x 9 through both scored paths, against
    best_of_k of the oracle's McClendon scores with ties going to the first candidate.
(b) Bit-exact.  The device grid, start, goal, step table, SOL_LEN, MAX_STEPS and generation count
    equal what oracle.gen_stream.stream_maze draws under the same key, on shapes around the lattice
    widths 32 and 64 (rows past 31 live in a lane's second word), non-square shapes, toroidal shapes,
    slot_id_base != 0 and regeneration; best-of-6 keeps exactly the candidate the shared tie rule
    (oracle.gen_exact.best_candidate) picks from the oracle's scores of the model's six candidates.
(c) Metrics on the smallest mazes: every enumerated 5 x 5, 7 x 7, 7 x 9 and 9 x 7 maze scored on the
    device equals the oracle.
"""
from functools import lru_cache

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle.env_port import MazeTables  # noqa: E402
from oracle.gen_exact import (TIE_REL, best_candidate, best_of_k, chi_square, edge_weights, exact_outcomes,  # noqa: E402
                              n_edges, outcome_grid)
from oracle.gen_stream import stream_maze  # noqa: E402
from oracle.generation import ALGORITHMS, select_goal  # noqa: E402
from oracle.metrics import kim_crawfis, mcclendon  # noqa: E402

POOL = 1 << 20    # slots per generate call of the distribution tests
P_MIN = 1e-6
KNIFE_REL = 1e-9  # device and oracle difficulties agree to this; closer genuine gaps cannot be judged


def _hw(shape):
    return (shape, shape) if isinstance(shape, int) else tuple(shape)


def _lattice(shape, toroidal):
    H, W = _hw(shape)
    if toroidal:   # drawn at shape + 2 (lib/maze_generation.py:48)
        H, W = H + 2, W + 2
    return (H - 1) // 2, (W - 1) // 2


def _unpack(v):
    return int(v) & 0xffff, int(v) >> 16


@lru_cache(maxsize=None)
def _lattice_scores(nr, nc):
    """Oracle metrics of every (start, tree) outcome of an nr x nc lattice (r-prim reaches them all):
    {outcome: (goal, mcclendon difficulty, complexity, kim_crawfis dict)}."""
    out = {}
    for oid in exact_outcomes("r-prim", nr, nc):
        start, grid = outcome_grid(oid, nr, nc)
        goal = select_goal(grid, start)
        grid[goal] = 2
        d, c = mcclendon(grid, start, goal)
        out[oid] = (goal, d, c, kim_crawfis(grid, start, goal))
    return out


def _device_outcomes(pool, n, shape, toroidal):
    """Outcome ids (oracle.gen_exact numbering) and goal cell indices of slots 0 .. n-1, on the device."""
    import maze_b200 as mb
    H, W = _hw(shape)
    nr, nc = _lattice(shape, toroidal)
    g = pool.grids[:n, :H * W].reshape(n, H, W)
    meta = pool.meta[:n]
    st, gl = meta[:, mb.cabi.META_START].long(), meta[:, mb.cabi.META_GOAL].long()
    sr, sc, gr, gc = st & 0xffff, st >> 16, gl & 0xffff, gl >> 16
    if toroidal:   # back to the bordered maze the generator drew
        b = torch.zeros((n, H + 2, W + 2), dtype=g.dtype, device=g.device)
        b[:, 1:-1, 1:-1] = g
        g, sr, sc, gr, gc = b, sr + 1, sc + 1, gr + 1, gc + 1
    wE, wS = (torch.from_numpy(w).to(g.device) for w in edge_weights(nr, nc))
    bits = ((g[:, 1::2, 2:-1:2] != 0).long() * wE).sum((1, 2)) + ((g[:, 2:-1:2, 1::2] != 0).long() * wS).sum((1, 2))
    cell = lambda r, c: ((r - 1) // 2) * nc + (c - 1) // 2   # noqa: E731
    return (cell(sr, sc) << n_edges(nr, nc)) | bits, cell(gr, gc)


def _sample(algo, shape, toroidal, total, candidates=1, queue=False):
    """Counts per outcome id of `total` device mazes (POOL slots per call, seeds 1, 2, ...) and the set of
    (outcome, goal cell) pairs seen.  queue=True draws through the regeneration path (device-side count,
    single kernel) instead of the bulk pipeline."""
    import maze_b200 as mb
    nr, nc = _lattice(shape, toroidal)
    cells = nr * nc
    counts = torch.zeros(cells << n_edges(nr, nc), dtype=torch.int64, device="cuda")
    pairs = set()
    pool = mb.MazePool(POOL, _hw(shape))
    ids = torch.arange(POOL, dtype=torch.int32, device="cuda")
    count = torch.tensor([POOL], dtype=torch.int32, device="cuda")
    for k in range(total // POOL):
        seed = 1 + k
        if queue:
            if k == 0:
                pool.generate(shapes=_hw(shape), algorithms=algo, toroidal=toroidal, seed=0)   # configure the slots
            pool.generate(ids=ids, count_dev=count, configure=False, seed=seed, candidates=candidates)
        else:
            pool.generate(shapes=_hw(shape), algorithms=algo, toroidal=toroidal, seed=seed, candidates=candidates)
        oid, goal = _device_outcomes(pool, POOL, shape, toroidal)
        counts += torch.bincount(oid, minlength=counts.numel())
        pairs.update(torch.unique(oid * cells + goal).tolist())
    return counts.cpu().numpy(), pairs


def _assert_distribution(counts, pairs, probs, nr, nc, tag):
    p, outside = chi_square(counts, probs)
    assert outside == 0, (tag, "draws outside the support", outside)
    cells = nr * nc
    seen = {}
    for pair in pairs:
        oid, goal = divmod(pair, cells)
        assert oid not in seen, (tag, "two goals for one maze", oid)
        seen[oid] = goal
    for oid, goal in seen.items():
        gr, gc = _lattice_scores(nr, nc)[oid][0]
        assert goal == ((gr - 1) // 2) * nc + (gc - 1) // 2, (tag, "goal is not select_goal's", oid)
    assert p >= P_MIN, (tag, "chi-square p", p)


DIST_CASES = [(5, False), (7, False), ((7, 9), False), ((9, 7), False), (5, True), ((5, 7), True), ((7, 5), True)]


@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("shape,toroidal", DIST_CASES)
def test_generator_matches_exact_distribution(algo, shape, toroidal):
    nr, nc = _lattice(shape, toroidal)
    total = (1 << 22) if nr * nc <= 9 else (1 << 24)
    counts, pairs = _sample(algo, shape, toroidal, total)
    _assert_distribution(counts, pairs, exact_outcomes(algo, nr, nc), nr, nc, (algo, shape, toroidal))


@pytest.mark.parametrize("queue", [False, True], ids=["bulk", "queue"])
@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("shape", [7, (7, 9)])
def test_best_of_six_matches_exact_distribution(shape, algo, queue):
    """Kept maze of best-of-6 against best_of_k of the exact distribution and the oracle's scores: ties
    (scores equal to 1e-12, of which 7 x 7 and 7 x 9 have many) must go to the first candidate."""
    nr, nc = _lattice(shape, False)
    probs = exact_outcomes(algo, nr, nc)
    scores = {o: v[1] for o, v in _lattice_scores(nr, nc).items()}
    counts, pairs = _sample(algo, shape, False, 1 << 22, candidates=6, queue=queue)
    _assert_distribution(counts, pairs, best_of_k(probs, scores, 6), nr, nc, (algo, shape, queue))


# ---- (b) bit-exact against the stream model ----------------------------------------------------

def _assert_slot(mb, pool, meta, m, algo, shape, toroidal, seed, slot, gen_count=0, maze=None):
    start, goal, grid = maze or stream_maze(algo, shape, toroidal, seed, slot, gen_count)
    tag = (algo, shape, toroidal, seed, slot, gen_count)
    np.testing.assert_array_equal(pool.grid_host(m), grid, err_msg=str(tag))
    assert _unpack(meta[m, mb.cabi.META_START]) == start, tag
    assert _unpack(meta[m, mb.cabi.META_GOAL]) == goal, tag
    t = MazeTables(grid, start, goal, toroidal)
    np.testing.assert_array_equal(pool.table_host(m), t.table, err_msg=str(tag))
    assert meta[m, mb.cabi.META_SOL_LEN] == int(t.dgoal[start]) + 1, tag
    assert meta[m, mb.cabi.META_MAX_STEPS] == t.max_steps, tag
    assert meta[m, mb.cabi.META_SPARE] == gen_count + 1, tag


BIT_EXACT_SHAPES = [5, 7, 9, 21, 63, 65, 67, 81, 127, 129, (9, 129), (129, 9), (65, 7)]


@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("shape", BIT_EXACT_SHAPES, ids=str)
def test_generator_matches_stream_model(algo, shape):
    import maze_b200 as mb
    n = 8 if max(_hw(shape)) <= 21 else 3
    pool = mb.MazePool(n, _hw(shape))
    pool.generate(shapes=_hw(shape), algorithms=algo, seed=2024)
    meta = pool.meta_host()
    for m in range(n):
        _assert_slot(mb, pool, meta, m, algo, shape, False, 2024, m)


@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("shape", [5, 61, 63, 65, 127])
def test_toroidal_generator_matches_stream_model(algo, shape):
    import maze_b200 as mb
    n = 6 if shape <= 21 else 2
    pool = mb.MazePool(n, (shape, shape))
    pool.generate(algorithms=algo, toroidal=True, seed=77)
    meta = pool.meta_host()
    for m in range(n):
        _assert_slot(mb, pool, meta, m, algo, shape, True, 77, m)


def test_slot_id_base_ids_and_regeneration_match_stream_model():
    """Slot m of a pool generated with slot_id_base b draws slot id b + m; a second generate of a subset
    draws generation count 1 for those slots and leaves the others as they were."""
    import maze_b200 as mb
    n, base, shapes = 12, 1 << 33, [(21, 21), (9, 129), (65, 7)] * 4
    algos = [ALGORITHMS[m % 3] for m in range(n)]
    pool = mb.MazePool(n, (129, 129))
    pool.generate(shapes=shapes, algorithms=algos, seed=5, slot_id_base=base)
    meta = pool.meta_host()
    for m in range(n):
        _assert_slot(mb, pool, meta, m, algos[m], shapes[m], False, 5, base + m)
    again = [1, 4, 11, 7]
    pool.generate(ids=again, configure=False, seed=5, slot_id_base=base)
    meta = pool.meta_host()
    for m in range(n):
        _assert_slot(mb, pool, meta, m, algos[m], shapes[m], False, 5, base + m, gen_count=int(m in again))


def _oracle_difficulty(maze, toroidal):
    start, goal, grid = maze
    if toroidal:   # scored on the bordered maze before stripping (lib/maze_generation.py:48-56)
        grid, start, goal = np.pad(grid, 1), (start[0] + 1, start[1] + 1), (goal[0] + 1, goal[1] + 1)
    return mcclendon(grid, start, goal)[0]


@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("shape,toroidal", [(5, False), (7, False), (21, False), (41, False), (81, False), (21, True)])
def test_best_of_six_matches_stream_model(algo, shape, toroidal):
    """Both scored paths keep the candidate oracle.gen_exact.best_candidate picks from the oracle's scores of
    the model's six candidates: the lowest score, the first of several equal ones.  Slots where two scores
    differ by more than the tie tolerance but less than the device / oracle agreement (1e-9) are knife-edge:
    they are skipped and counted."""
    import maze_b200 as mb
    n = {5: 64, 7: 64, 21: 32, 41: 12, 81: 6}[shape]
    seed = 300 + shape
    expect, knife = {}, 0
    for m in range(n):
        cands = [stream_maze(algo, shape, toroidal, seed, m, candidate=c) for c in range(6)]
        scores = [_oracle_difficulty(c, toroidal) for c in cands]
        gaps = [abs(a - b) / max(abs(a), abs(b)) for i, a in enumerate(scores) for b in scores[i + 1:] if a != b]
        if any(TIE_REL < g <= KNIFE_REL for g in gaps):
            knife += 1
            continue
        best = best_candidate(scores)
        expect[m] = (cands[best], scores[best])
    assert knife <= n // 8, knife
    bulk = mb.MazePool(n, (shape, shape))
    dout = torch.zeros(n, dtype=torch.float64, device="cuda")
    bulk.generate(algorithms=algo, toroidal=toroidal, seed=seed, candidates=6, difficulty_out=dout)
    queue = mb.MazePool(n, (shape, shape))
    queue.generate(algorithms=algo, toroidal=toroidal, seed=seed)    # configure the slots, generation count 1 ...
    queue.meta[:, mb.cabi.META_SPARE] = 0                             # ... back to 0: the keys of `bulk`
    ids, count = torch.arange(n, dtype=torch.int32, device="cuda"), torch.tensor([n], dtype=torch.int32, device="cuda")
    queue.generate(ids=ids, count_dev=count, configure=False, seed=seed, candidates=6)
    d = dout.cpu().numpy()
    for pool in (bulk, queue):
        meta = pool.meta_host()
        for m, (maze, score) in expect.items():
            _assert_slot(mb, pool, meta, m, algo, shape, toroidal, seed, m, maze=maze)
    for m, (maze, score) in expect.items():
        assert d[m] == pytest.approx(score, rel=KNIFE_REL), m


# ---- (c) metrics on the smallest mazes ---------------------------------------------------------

@pytest.mark.parametrize("shape", [5, 7, (7, 9), (9, 7)], ids=str)
def test_metrics_of_every_small_maze(shape):
    """maze_difficulty on every (start, tree) outcome of the smallest lattices: McClendon difficulty and
    complexity to 1e-9 relative, Kim-Crawfis L / DE / D, solution length and dead ends exactly."""
    import maze_b200 as mb
    nr, nc = _lattice(shape, False)
    ref = _lattice_scores(nr, nc)
    oids = sorted(ref)
    grids, starts, goals = [], [], []
    for oid in oids:
        start, grid = outcome_grid(oid, nr, nc)
        grids.append(grid)
        starts.append(start)
        goals.append(ref[oid][0])
    pool = mb.MazePool.from_grids(grids, starts, goals, False)
    out = pool.difficulty().cpu().numpy()
    want = np.array([[ref[o][1], ref[o][2]] for o in oids])
    np.testing.assert_allclose(out[:, :2], want, rtol=1e-9, atol=0)
    kim = np.array([[ref[o][3][k] for k in ("L", "DE", "D", "sol_len", "dead_end_count")] for o in oids], dtype=np.float64)
    np.testing.assert_array_equal(out[:, 2:7], kim)
