"""maze_difficulty through the C ABI: McClendon difficulty / complexity and Kim-Crawfis L / DE / D
against values the unmodified reference produced (tests/golden/metrics.npz, incl. the literal
15x15 known answers) and against the oracle on device-generated mazes of every generator."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from conftest import load_golden  # noqa: E402
from oracle.generation import ALGORITHMS  # noqa: E402
from oracle.metrics import kim_crawfis, mcclendon  # noqa: E402

REL = 1e-9   # float sums run in a different order than networkx iteration (SURVEY.md section 7)


def _pool_from_rows(z, rows):
    import maze_b200 as mb
    grids = [z[f"m{m['id']}_grid"] for m in rows]
    return mb, mb.MazePool.from_grids(grids, [m["start"] for m in rows], [m["goal"] for m in rows],
                                      [bool(m["no_border"]) for m in rows])


def test_literal_maze_known_answers():
    z, meta = load_golden("metrics")
    mb, pool = _pool_from_rows(z, meta[:1])
    out = pool.difficulty().cpu().numpy()[0]
    # reference outputs on the literal maze of testing_Mccledon.py:4-20 (BASELINE.md section 2)
    assert out[0] == pytest.approx(9.950639302928026, rel=1e-12)
    assert out[1] == pytest.approx(5.681612603202764, rel=1e-12)
    assert out[2] == 0.6288659793814433 and out[3] == 0.03278688524590164 and out[4] == 0.03278688524590164
    assert out[5] == 61


def test_golden_mazes_match_reference():
    z, meta = load_golden("metrics")
    mb, pool = _pool_from_rows(z, meta)
    out = pool.difficulty().cpu().numpy()
    for k, m in enumerate(meta):
        tag = (m["algo"], m["shape"], m["id"])
        assert out[k, 0] == pytest.approx(m["difficulty"], rel=REL), tag
        if m["no_border"]:
            continue   # the reference records only the difficulty for border-less mazes
        assert out[k, 1] == pytest.approx(m["complexity"], rel=REL), tag
        assert out[k, 2] == m["L"] and out[k, 3] == m["DE"] and out[k, 4] == m["D"], tag
        assert out[k, 5] == m["sol_len"], tag


def test_ids_select_slots():
    z, meta = load_golden("metrics")
    mb, pool = _pool_from_rows(z, meta)
    full = pool.difficulty().cpu().numpy()
    ids = [7, 3, 3, 20]
    part = pool.difficulty(ids).cpu().numpy()
    np.testing.assert_array_equal(part, full[ids])


@pytest.mark.parametrize("algo", ALGORITHMS)
@pytest.mark.parametrize("shape,toroidal", [(21, False), (41, False), (81, False), (129, False), (41, True), (79, True)])
def test_generated_mazes_match_oracle(algo, shape, toroidal):
    import maze_b200 as mb
    n = 24 if shape <= 41 else 8
    pool = mb.MazePool(n, (shape, shape))
    pool.generate(algorithms=algo, toroidal=toroidal, seed=1000 + shape)
    out = pool.difficulty().cpu().numpy()
    meta = pool.meta_host()
    for m in range(n):
        grid = pool.grid_host(m)
        start = (int(meta[m, 2]) & 0xffff, int(meta[m, 2]) >> 16)
        goal = (int(meta[m, 3]) & 0xffff, int(meta[m, 3]) >> 16)
        if toroidal:
            grid = np.pad(grid, 1)
            start, goal = (start[0] + 1, start[1] + 1), (goal[0] + 1, goal[1] + 1)
        d, c = mcclendon(grid, start, goal)
        k = kim_crawfis(grid, start, goal)
        assert out[m, 0] == pytest.approx(d, rel=REL), (algo, shape, m)
        assert out[m, 1] == pytest.approx(c, rel=REL), (algo, shape, m)
        assert out[m, 2] == k["L"] and out[m, 3] == k["DE"] and out[m, 4] == k["D"], (algo, shape, m)
        assert out[m, 5] == k["sol_len"] and out[m, 6] == k["dead_end_count"]


def test_unreachable_goal_gives_nan():
    import maze_b200 as mb
    g = np.zeros((7, 7), dtype=np.uint8)
    g[1, 1:4] = 1
    g[5, 5] = 2
    pool = mb.MazePool.from_grids([g], [(1, 1)], [(5, 5)], False)
    out = pool.difficulty().cpu().numpy()[0]
    assert np.isnan(out[:5]).all()


@pytest.mark.parametrize("algo,toroidal", [("r-prim", False), ("dfs", False), ("prim&kill", True)])
def test_best_of_k_selection(algo, toroidal):
    """BaseMazeEnv.generate_maze (base_maze_env.py:78-97): keep the least difficult of 1 + 5 draws,
    strict <.  Candidate c of a slot is the same maze for every k > c, so the kept difficulty is a
    running minimum over k and the kept maze only changes when the minimum does."""
    import maze_b200 as mb
    n, shape = 48, (21, 21)
    prev_d, prev_grids = None, None
    for k in range(1, 7):
        pool = mb.MazePool(n, shape)
        dout = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
        pool.generate(algorithms=algo, toroidal=toroidal, seed=77, candidates=k, difficulty_out=dout)
        d = dout.cpu().numpy()
        rescored = pool.difficulty().cpu().numpy()[:, 0]
        # the reported difficulty is the kept maze's (shared-memory float atomics: last-ulp run-to-run noise)
        np.testing.assert_allclose(d, rescored, rtol=1e-12)
        grids = [pool.grid_host(m).copy() for m in range(n)]
        if prev_d is not None:
            assert (d <= prev_d * (1 + 1e-12)).all()
            for m in range(n):
                if abs(d[m] - prev_d[m]) <= 1e-12 * prev_d[m]:
                    np.testing.assert_array_equal(grids[m], prev_grids[m])
        prev_d, prev_grids = d, grids
    # six draws must have found easier mazes for most slots
    pool1 = mb.MazePool(n, shape)
    pool1.generate(algorithms=algo, toroidal=toroidal, seed=77)
    d1 = pool1.difficulty().cpu().numpy()[:, 0]
    assert (prev_d <= d1 * (1 + 1e-12)).all() and (prev_d < d1 * (1 - 1e-9)).mean() > 0.5


@pytest.mark.parametrize("algo,toroidal", [("r-prim", False), ("dfs", False), ("prim&kill", False), ("r-prim", True)])
def test_best_of_six_keeps_the_reference_winner(algo, toroidal, monkeypatch):
    """generate_maze (base_maze_env.py:78-97, toroidal_maze_env.py:40-54): of the six draws the FIRST minimum of the
    McClendon difficulty is kept (scores equal to 1e-12 relative are one minimum: oracle.gen_exact.best_candidate).  Every candidate is materialised on its own (the MAZE_GEN_CANDIDATE_BASE test hook
    shifts the RNG key, candidates = 1), re-scored with the ORACLE (oracle.metrics.mcclendon, itself pinned to the
    reference's values), and the oracle's winner must be the maze the best-of-six launch kept -- through both code paths:
    the bulk pipeline (planes kernel + scoring kernel) and the single-kernel path of the regeneration queue."""
    import maze_b200 as mb
    from oracle.gen_exact import best_candidate
    from oracle.metrics import mcclendon
    n, S = 40, 21
    cands = []
    for c in range(6):
        monkeypatch.setenv("MAZE_GEN_CANDIDATE_BASE", str(c))
        pool = mb.MazePool(n, (S, S))
        pool.generate(algorithms=algo, toroidal=toroidal, seed=99)
        meta = pool.meta_host()
        cands.append([(pool.grid_host(m).copy(), int(meta[m, 2]), int(meta[m, 3])) for m in range(n)])
    monkeypatch.delenv("MAZE_GEN_CANDIDATE_BASE")

    def oracle_score(grid, start, goal):
        s, g = (start & 0xffff, start >> 16), (goal & 0xffff, goal >> 16)
        if toroidal:   # scored on the bordered maze before stripping (lib/maze_generation.py:48-56)
            grid, s, g = np.pad(grid, 1), (s[0] + 1, s[1] + 1), (g[0] + 1, g[1] + 1)
        return mcclendon(grid, s, g)[0]

    winners = []
    for m in range(n):
        scores = [oracle_score(*cands[c][m]) for c in range(6)]
        winners.append((best_candidate(scores), scores))   # the first of the lowest scores (ties to 1e-12) wins
    assert len({w for w, _ in winners}) >= 4          # the winner is not always the same candidate

    bulk = mb.MazePool(n, (S, S))
    dout = torch.zeros(n, dtype=torch.float64, device="cuda")
    bulk.generate(algorithms=algo, toroidal=toroidal, seed=99, candidates=6, difficulty_out=dout)
    queue = mb.MazePool(n, (S, S))
    queue.generate(algorithms=algo, toroidal=toroidal, seed=99)                       # configure the slots, generation count 1 ...
    queue.meta[:, mb.cabi.META_SPARE] = 0                                             # ... back to 0: same RNG keys as `bulk`
    ids, count = torch.arange(n, dtype=torch.int32, device="cuda"), torch.tensor([n], dtype=torch.int32, device="cuda")
    queue.generate(ids=ids, count_dev=count, configure=False, seed=99, candidates=6)  # device-side count: the single-kernel path
    for m in range(n):
        best, scores = winners[m]
        for pool in (bulk, queue):
            np.testing.assert_array_equal(pool.grid_host(m), cands[best][m][0], err_msg=f"slot {m}: kept maze is not candidate {best} {scores}")
        assert dout[m].item() == pytest.approx(scores[best], rel=1e-9)


def _ext_vector(d):
    return np.array([d["density"], d["T"], d["J"], d["CR"], d["AC"], d["FDE"], d["BDE"], d["L_DE"],
                     *d["T_DE"], *d["D_sharp"], *d["L_sharp"]], dtype=np.float64)


def test_extended_metrics_match_reference_bit_exactly():
    """maze_difficulty_ext against tests/golden/metrics_ext.npz (the unmodified MetricsCalculator's
    density / T / J / CR / DE_sub / L_DE / T_DE / D_sharp / L_sharp): identical float64 bit patterns,
    and the base record is the one maze_difficulty writes."""
    import json
    import os
    z, meta = load_golden("metrics")
    ext_rows = json.loads(str(np.load(os.path.join(os.path.dirname(__file__), "golden", "metrics_ext.npz"))["meta"]))
    rows = [next(m for m in meta if m["id"] == r["id"]) for r in ext_rows]
    mb, pool = _pool_from_rows(z, rows)
    base, ext = pool.difficulty(extended=True)
    base, ext = base.cpu().numpy(), ext.cpu().numpy()
    plain = pool.difficulty().cpu().numpy()
    assert np.array_equal(base[:, 2:7], plain[:, 2:7])
    np.testing.assert_allclose(base[:, :2], plain[:, :2], rtol=1e-12)
    for k, r in enumerate(ext_rows):
        want = _ext_vector(r)
        assert np.array_equal(ext[k, :17].view(np.uint64), want.view(np.uint64)), (rows[k]["algo"], rows[k]["shape"], ext[k, :17], want)
        assert not ext[k, 17:].any()


@pytest.mark.parametrize("shape,toroidal", [(81, False), (129, False), (41, True)])
def test_extended_metrics_match_oracle_on_generated_mazes(shape, toroidal):
    import maze_b200 as mb
    from oracle.metrics import kim_crawfis_extended
    n = 9
    pool = mb.MazePool(n, (shape, shape))
    pool.generate(algorithms=list(ALGORITHMS) * 3, toroidal=toroidal, seed=77 + shape)
    _, ext = pool.difficulty(extended=True)
    ext = ext.cpu().numpy()
    meta = pool.meta_host()
    for m in range(n):
        grid = pool.grid_host(m)
        start = (int(meta[m, 2]) & 0xffff, int(meta[m, 2]) >> 16)
        goal = (int(meta[m, 3]) & 0xffff, int(meta[m, 3]) >> 16)
        if toroidal:   # scored on the zero-padded (bordered) grid
            grid, start, goal = np.pad(grid, 1), (start[0] + 1, start[1] + 1), (goal[0] + 1, goal[1] + 1)
        want = _ext_vector(kim_crawfis_extended(grid, start, goal))
        assert np.array_equal(ext[m, :17].view(np.uint64), want.view(np.uint64)), (m, ext[m, :17], want)


def test_metrics_calculator_mirror_exposes_the_unused_methods():
    """lib.maze_difficulty_evaluation.MetricsCalculator with the reference's method names."""
    import json
    import os
    from lib.maze_difficulty_evaluation.metrics_calculator import MetricsCalculator
    z, meta = load_golden("metrics")
    r = json.loads(str(np.load(os.path.join(os.path.dirname(__file__), "golden", "metrics_ext.npz"))["meta"]))[5]
    m = next(x for x in meta if x["id"] == r["id"])
    maze = z[f"m{m['id']}_grid"].astype(int).tolist()
    mc = MetricsCalculator(maze, m["sol_len"])
    sol = [tuple(m["start"])]   # only the first block of the solution path is consulted
    assert mc.calculate_density() == r["density"]
    assert mc.calculate_T(sol) == r["T"] and mc.calculate_J(sol) == r["J"] and mc.calculate_CR(sol) == r["CR"]
    assert mc.calculate_DE_sub(sol) == (r["AC"], r["FDE"], r["BDE"])
    assert mc.calculate_L_DE(sol) == r["L_DE"]
    for k, t in enumerate(("AC", "FDE", "BDE")):
        assert mc.calculate_T_DE(sol, t) == r["T_DE"][k]
        assert mc.calculate_D_sharp(sol, t) == r["D_sharp"][k]
        assert mc.calculate_L_sharp(sol, t) == r["L_sharp"][k]


@pytest.mark.parametrize("toroidal", [False, True])
def test_bulk_best_of_k_pipeline_equals_the_single_kernel_path(toroidal, monkeypatch):
    """Bulk best-of-k draws its candidates with the warp generator into scratch and scores them in the CTA
    kernel; the regeneration-queue path does both in one kernel.  Same candidates, same scores, same kept maze."""
    import maze_b200 as mb
    n, shape = 300, (41, 41)
    algos = ["r-prim", "dfs", "prim&kill"] * 100

    def run():
        pool = mb.MazePool(n, shape)
        d = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
        pool.generate(algorithms=algos, toroidal=toroidal, seed=21, candidates=6, difficulty_out=d)
        return pool, d
    two, d2 = run()
    monkeypatch.setenv("MAZE_GEN_SINGLE_KERNEL", "1")
    one, d1 = run()
    monkeypatch.delenv("MAZE_GEN_SINGLE_KERNEL")
    assert torch.equal(two.grids, one.grids) and torch.equal(two.table, one.table) and torch.equal(two.meta, one.meta)
    np.testing.assert_allclose(d2.cpu().numpy(), d1.cpu().numpy(), rtol=1e-12)
    # a second generation of the same slots (generation count 1) differs from the first and again agrees
    two.generate(algorithms=algos, toroidal=toroidal, seed=21, candidates=6)
    monkeypatch.setenv("MAZE_GEN_SINGLE_KERNEL", "1")
    one.generate(algorithms=algos, toroidal=toroidal, seed=21, candidates=6)
    assert torch.equal(two.grids, one.grids) and torch.equal(two.meta, one.meta)
